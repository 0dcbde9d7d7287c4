"""Graph-captured inference (not a pytest file): eager `BoostedDETR.call(training=False)` against `GraphedInference`.

Workloads (tf32 mode, C = 82, A = 3):
  reference_default   the reference's default model: 4 blocks, 96 queries, 560 x 560 -> 18 x 18 = 324 tokens, batch 8
  config2             6 blocks, batch 16, 20 x 20
  config5_stride32    6 blocks, batch 4, 25 x 42 = 1 050 tokens (config 5 at the reference's stride)
  config5             6 blocks, batch 4, 110 x 182 = 20 020 tokens

Arms: `eager`; `graph` (threshold None: one graph around the multi-stream forward); `segmented` (threshold 2.0, never
reached: every block runs through the IF chain) beside `eager_exit_never`, the eager call with the same threshold (one
D2H copy and synchronisation per block boundary).  At config-2 size also the early-exit arms, eager and segmented graph:
an exit after block 1 and after block 3 (threshold 0, min_blocks 2 / 4).  BDETR_PDL=0 in the environment measures the
same with programmatic dependent launch off, in the eager calls and in the captured graphs.

Per arm: device time (CUDA events on the launching stream around one call, L2 flushed by a 256 MiB write outside the
brackets, as bench.py's device arm), e2e time (pinned host features in, the three predictions out to pinned host memory,
one synchronisation per call, perf_counter), and for eager the host's issue time of one call (perf_counter without a
synchronisation) and the library launches per call.  The arms alternate round by round; each number is the median of the
round medians, with the smallest and largest round median beside it.  Every graph arm is checked bit for bit against
the eager call with the same settings.

usage: python bench_tools/bench_infer_graph.py [--out FILE.json] [--rounds N] [--steps K] [--only NAME]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from boosted_detr_b200 import _lib  # noqa: E402

WORKLOADS = {
    "reference_default": dict(N=4, Q=96, rows=18, cols=18, B=8),
    "config2": dict(N=6, Q=100, rows=20, cols=20, B=16),
    "config5_stride32": dict(N=6, Q=100, rows=25, cols=42, B=4),
    "config5": dict(N=6, Q=100, rows=110, cols=182, B=4),
}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi name, power.limit, clocks.sm, clocks.max.sm": q.stdout.strip()}


def make_model(w):
    from boosted_detr_b200.boosted_model import BoostedDETR
    from boosted_detr_b200.parameters import ModelParameters
    p = ModelParameters("COCO").default_params()
    p.pop("pad_value"); p.pop("oov_value")
    p.update(num_object_preds=w["Q"], num_encoder_blocks=w["N"], num_decoder_blocks=w["N"],
             image_size=(w["rows"] * 32, w["cols"] * 32))
    model = BoostedDETR(**p, seed=0).build()
    assert model.num_categories == 82 and model.num_attributes == 3
    return model


class Arm:
    def __init__(self, name, model, call, settings):
        self.name, self.model, self.call, self.settings = name, model, call, settings
        self.dev, self.e2e, self.issue = [], [], []

    def apply(self):
        self.model.early_exit_threshold, self.model.early_exit_min_blocks = self.settings


def run_workload(name, w, rounds, steps, flush):
    model = make_model(w)
    lib = _lib.load()
    rng = np.random.default_rng(1)
    x = np.tanh(rng.standard_normal((w["B"], w["rows"], w["cols"], 256))).astype(np.float32)
    feats_h = torch.from_numpy(x).pin_memory()
    feats = feats_h.cuda()
    from boosted_detr_b200.graph import GraphedInference
    settings = {"never": (2.0, 1)}
    if name == "config2":
        settings.update({"exit_after_block_1": (0.0, 2), "exit_after_block_3": (0.0, 4)})
    res = {"shape": w, "tokens": w["rows"] * w["cols"]}

    def eager_call(inputs):
        return model.call(inputs, training=False)

    arms = [Arm("eager", model, eager_call, (None, 1))]
    model.early_exit_threshold = None
    g = GraphedInference(model, {"features": feats})
    res["graph_capture_ms"], res["graph_instantiate_ms"] = g.capture_seconds * 1e3, g.instantiate_seconds * 1e3
    arms.append(Arm("graph", model, g, (None, 1)))
    model.early_exit_threshold, model.early_exit_min_blocks = 2.0, 1
    s = GraphedInference(model, {"features": feats})
    res["segmented_capture_ms"], res["segmented_instantiate_ms"] = s.capture_seconds * 1e3, s.instantiate_seconds * 1e3
    for tag, st in settings.items():
        arms.append(Arm(f"eager_exit_{tag}", model, eager_call, st))
        arms.append(Arm(f"segmented_{tag}", model, s, st))

    # bit identity against the eager call with the same settings, and launch counts
    checks = {}
    for a in arms:
        a.apply()
        lib.bdetr_reset_launch_count()
        out = [t.clone() for t in a.call({"features": feats})]
        torch.cuda.synchronize()
        c = {"library_launches_per_call": int(lib.bdetr_launch_count())}
        if a.call is eager_call:
            c["exit_block"] = model.last_exit_block
        else:
            ref = [t.clone() for t in eager_call({"features": feats})]
            torch.cuda.synchronize()
            c.update(bit_identical_to_eager=all(torch.equal(p, q) for p, q in zip(out, ref)), exit_block=a.call.last_exit_block,
                     eager_exit_block=model.last_exit_block, graph_launches_per_call=1)
        checks[a.name] = c
    res["checks"] = checks

    hp = [torch.empty(t.shape).pin_memory() for t in arms[0].call({"features": feats})]
    for r in range(rounds):
        for a in arms:
            a.apply()
            for _ in range(2):
                a.call({"features": feats})
            torch.cuda.synchronize()
            dev, e2e, issue = [], [], []
            for _ in range(steps):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); a.call({"features": feats}); e1.record()
                e1.synchronize()
                dev.append(e0.elapsed_time(e1))
            for _ in range(steps):
                t0 = time.perf_counter()
                p = a.call({"features": feats_h})
                for h, t in zip(hp, p):
                    h.copy_(t, non_blocking=True)
                torch.cuda.current_stream().synchronize()
                e2e.append((time.perf_counter() - t0) * 1e3)
            if a.call is eager_call:
                for _ in range(steps):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    a.call({"features": feats})
                    issue.append((time.perf_counter() - t0) * 1e3)
                torch.cuda.synchronize()
            a.dev.append(float(np.median(dev)))
            a.e2e.append(float(np.median(e2e)))
            if issue:
                a.issue.append(float(np.median(issue)))
    stat = lambda v: {"median_ms": float(np.median(v)), "min_round_ms": float(min(v)), "max_round_ms": float(max(v))}
    res["arms"] = {}
    for a in arms:
        d = {"device": stat(a.dev), "e2e": stat(a.e2e)}
        if a.issue:
            d["host_issue"] = stat(a.issue)
        res["arms"][a.name] = d
    model.early_exit_threshold = None
    g.close(); s.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--only", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_infer_graph needs a CUDA device")
    lib = _lib.load()
    lib.bdetr_set_mode(_lib.MODE_TF32)
    flush = torch.empty(256 * 1024 * 1024 // 4, device="cuda")
    out = {"gpu": gpu_info(), "mode": "tf32", "pdl": int(lib.bdetr_get_pdl()), "rounds": args.rounds, "steps": args.steps,
           "l2": "flushed (256 MiB write) outside the event brackets of every device-time call", "workloads": {}}
    for name, w in WORKLOADS.items():
        if args.only and name != args.only:
            continue
        out["workloads"][name] = run_workload(name, w, args.rounds, args.steps, flush)
        print(json.dumps({name: out["workloads"][name]["arms"]}), flush=True)
    out["gpu_after"] = gpu_info()
    text = json.dumps(out, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        open(args.out, "w").write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
