"""Per-image early exit (not a pytest file): the per-batch exit against the per-image exit, eager and graph-captured.

Workloads (C = 82, A = 3):
  config5_tf32 / config5_fp16   6 blocks, batch 4, 110 x 182 = 20 020 tokens, tf32 / fp16 mode
  config2                       6 blocks, batch 16, 20 x 20, tf32
  reference_default             4 blocks, batch 8, 96 queries, 18 x 18, tf32
The images are scaled to different contrasts so that their confidences run apart; the threshold (min_blocks 1) is the
per-batch confidence, measured first, that spreads the exit blocks the most (most distinct exit blocks, then the work
fraction closest to 0.6).  The realised exit blocks, active counts and the work fraction sum(active) / (N * B) are
recorded with the bytes each compaction launch moves (read + write).

Arms: per_batch_eager, per_image_eager, per_batch_graph (IF chain of segments), per_image_graph (SWITCH chain),
graph_no_exit (threshold None, one graph), and the same four exit arms with a threshold no image reaches (`*_never`).
Device time: CUDA events on the launching stream around one call, L2 flushed by a 256 MiB write outside the brackets;
the arms alternate round by round, each number is the median of the round medians with the smallest and largest round
median beside it.  Every arm is checked bit for bit against its eager counterpart.  GPU name, power limit and SM clock
are read in the same run.

usage: python bench_tools/bench_exit_per_image.py [--out FILE.json] [--rounds N] [--steps K] [--only NAME]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from boosted_detr_b200 import _lib  # noqa: E402

WORKLOADS = {
    "config5_tf32": dict(N=6, Q=100, rows=110, cols=182, B=4, mode="tf32"),
    "config5_fp16": dict(N=6, Q=100, rows=110, cols=182, B=4, mode="fp16"),
    "config2": dict(N=6, Q=100, rows=20, cols=20, B=16, mode="tf32"),
    "reference_default": dict(N=4, Q=96, rows=18, cols=18, B=8, mode="tf32"),
}
MODES = {"tf32": _lib.MODE_TF32, "fp16": _lib.MODE_FP16}


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
    return BoostedDETR(**p, seed=0).build()


def exits(c, thr, N):
    """Per-image exit blocks and active counts (riders included) for min_blocks 1, as the plan kernel decides them."""
    B = c.shape[0]
    e = np.full(B, N - 1)
    for b in range(B):
        hit = [i for i in range(N - 1) if c[b, i] >= np.float32(thr)]
        if hit:
            e[b] = hit[0]
    return e


def counts_of(e, N, k_min):
    out = [len(e)]
    for i in range(N - 1):
        n = int((e > i).sum())
        out.append(max(n, k_min) if n else 0)
    return out


class Arm:
    def __init__(self, name, model, call, thr, per_image):
        self.name, self.model, self.call, self.thr, self.per_image = name, model, call, thr, per_image
        self.dev = []

    def apply(self):
        self.model.early_exit_threshold, self.model.early_exit_min_blocks = self.thr, 1
        self.model.early_exit_per_image = self.per_image


def run_workload(w, rounds, steps, flush):
    from boosted_detr_b200.graph import GraphedInference
    lib = _lib.load()
    lib.bdetr_set_mode(MODES[w["mode"]])
    model = make_model(w)
    N, B, Q, L = w["N"], w["B"], w["Q"], w["rows"] * w["cols"]
    rng = np.random.default_rng(1)
    x = np.tanh(rng.standard_normal((B, w["rows"], w["cols"], 256))).astype(np.float32)
    x *= np.linspace(0.25, 3.0, B, dtype=np.float32)[:, None, None, None]
    feats = {"features": torch.from_numpy(x).cuda()}
    # per-image confidences at every boundary, from the per-batch exit
    c = []
    for k in range(N - 1):
        model.early_exit_threshold, model.early_exit_min_blocks = 0.0, k + 1
        model.call(feats, training=False)
        c.append(model.last_image_confidence.numpy().copy())
    c = np.stack(c, 1)
    fused = model._use_fused(feats["features"])
    k_min = max(-(-128 // L), -(-128 // Q)) if fused else 1
    best = None
    for t in sorted(set(c.reshape(-1).tolist())):
        e = exits(c, t, N)
        frac = sum(counts_of(e, N, k_min)) / (N * B)
        key = (len(set(e.tolist())), -abs(frac - 0.6))
        if best is None or key > best[0]:
            best = (key, t)
    thr = float(best[1])
    res = {"shape": w, "tokens": L, "k_min": k_min, "fused": fused, "threshold": thr, "confidences": c.tolist()}

    def eager(inputs):
        return model.call(inputs, training=False)

    arms, graphs = [], {}
    model.early_exit_threshold, model.early_exit_per_image = None, False
    torch.cuda.synchronize()
    for tag, t, per_image in (("graph_no_exit", None, False), ("per_batch_graph", thr, False), ("per_image_graph", thr, True)):
        model.early_exit_threshold, model.early_exit_min_blocks, model.early_exit_per_image = t, 1, per_image
        torch.cuda.empty_cache()
        r0 = torch.cuda.memory_reserved()
        g = GraphedInference(model, feats)
        torch.cuda.synchronize()
        graphs[tag] = g
        res[tag] = {"capture_s": g.capture_seconds, "instantiate_s": g.instantiate_seconds,
                    "reserved_bytes_added": int(torch.cuda.memory_reserved() - r0)}
        if per_image:
            res[tag]["bodies"] = g.bodies
    arms.append(Arm("graph_no_exit", model, graphs["graph_no_exit"], None, False))
    for suffix, t in (("", thr), ("_never", 2.0)):
        arms.append(Arm("per_batch_eager" + suffix, model, eager, t, False))
        arms.append(Arm("per_image_eager" + suffix, model, eager, t, True))
        arms.append(Arm("per_batch_graph" + suffix, model, graphs["per_batch_graph"], t, False))
        arms.append(Arm("per_image_graph" + suffix, model, graphs["per_image_graph"], t, True))

    checks = {}
    for a in arms:
        a.apply()
        out = [t.clone() for t in a.call(feats)]
        ref = [t.clone() for t in eager(feats)]
        torch.cuda.synchronize()
        ck = {"bit_identical_to_eager": all(torch.equal(p, q) for p, q in zip(out, ref)), "last_exit_block": model.last_exit_block}
        if a.per_image:
            e, counts = model.last_exit_blocks.tolist(), model.last_active_counts.tolist()
            row = L * 256 + Q * (model.num_categories + model.num_attributes + 4)
            ck.update(exit_blocks=e, active_counts=counts, work_fraction=sum(counts) / (N * B),
                      compaction_bytes_per_launch=[8 * (counts[i + 1] * row + sum(1 for v in e if v == i) * (row - L * 256))
                                                   for i in range(N - 1)],
                      final_write_bytes=8 * sum(1 for v in e if v == N - 1) * (row - L * 256))
            if a.call is not eager:
                ck["state_identical_to_eager"] = (a.call.last_exit_blocks.tolist() == e and a.call.last_active_counts.tolist() == counts)
        checks[a.name] = ck
    res["checks"] = checks

    for _ in range(rounds):
        for a in arms:
            a.apply()
            for _ in range(2):
                a.call(feats)
            torch.cuda.synchronize()
            dev = []
            for _ in range(steps):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); a.call(feats); e1.record()
                e1.synchronize()
                dev.append(e0.elapsed_time(e1))
            a.dev.append(float(np.median(dev)))
    stat = lambda v: {"median_ms": float(np.median(v)), "min_round_ms": float(min(v)), "max_round_ms": float(max(v))}
    res["arms"] = {a.name: {"device": stat(a.dev)} for a in arms}
    model.early_exit_threshold, model.early_exit_per_image = None, False
    for g in graphs.values():
        g.close()
    lib.bdetr_set_mode(_lib.MODE_FP32)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--only", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_exit_per_image needs a CUDA device")
    lib = _lib.load()
    flush = torch.empty(256 * 1024 * 1024 // 4, device="cuda")
    out = {"gpu": gpu_info(), "pdl": int(lib.bdetr_get_pdl()), "rounds": args.rounds, "steps": args.steps,
           "l2": "flushed (256 MiB write) outside the event brackets of every device-time call", "workloads": {}}
    for name, w in WORKLOADS.items():
        if args.only and name != args.only:
            continue
        out["workloads"][name] = run_workload(w, args.rounds, args.steps, flush)
        print(json.dumps({name: {k: out["workloads"][name][k] for k in ("threshold", "arms")}}), flush=True)
    out["gpu_after"] = gpu_info()
    text = json.dumps(out, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        open(args.out, "w").write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
