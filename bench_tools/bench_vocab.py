"""Category vocabulary size (not a pytest file): what a C = 367 (Objects365) or C = 1205 (LVIS) vocabulary costs next to
COCO's C = 82.

  * bdetr_heads_fwd / bdetr_heads_bwd (through the wrappers the model uses) at M = 1600 rows, Dh = 256, A = 3,
    C in {82, 320, 367, 1205, 2048}; C <= 320 runs the one-kernel path, C > 320 the column slabs + row activation.
    The second Dense is 2 M Dh C FLOP.
  * target digest (bdetr_cost_targets_prepare) and cost matrix (bdetr_cost_matrix_prepared) at the config-2 shape
    (B 16, T 20, Q 100) and the config-4 shape (B 256, T 100, Q 300), A = 3, C in {82, 367, 1205}.
  * the CUDA-graphed training step at config-2 size (6 block pairs, batch 16, 20 x 20 features, 100 queries) at
    C = 82, 367 and 1205, and, from a torch.profiler run of eager steps, the GPU time per step by kernel family.

Tensor-core (tf32) mode.  CUDA events around each call or replay, L2 flushed (256 MiB write) outside the brackets, median
over the timed calls after warm-up; the vocabulary sizes alternate round by round so that clock drift hits all of them.

usage: python bench_tools/bench_vocab.py [--out FILE.json] [--rounds N]"""
import argparse
import json
import os
import re
import subprocess
import sys
from collections import defaultdict

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from boosted_detr_b200 import _lib  # noqa: E402
from util import synth_preds, synth_targets  # noqa: E402

HEADS_C = (82, 320, 367, 1205, 2048)
MATCH_C = (82, 367, 1205)
MATCH_SHAPES = {"config2": (16, 20, 100), "config4": (256, 100, 300)}
STEP_C = (82, 367, 1205)
M, D, A = 1600, 256, 3


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def time_calls(fn, flush, n):
    ts = []
    for _ in range(n):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return ts


def heads_fns(C):
    from boosted_detr_b200.layers import Layer
    from boosted_detr_b200.prediction_heads import (BoxPredictionHead, MultiClassPredictionHead, SingleClassPredictionHead,
                                                    heads_backward_fused, heads_forward_fused)
    Layer._rng = np.random.default_rng(1)
    Q = 100
    x = torch.randn(M // Q, Q, D, device="cuda")
    heads = (SingleClassPredictionHead(C, D, Q, name="cat"), MultiClassPredictionHead(A, D, Q, name="attr"),
             BoxPredictionHead(D, Q, name="box"))
    _, ctx = heads_forward_fused(heads, x, True, None, 1.0)
    d_cum = [torch.randn_like(t) for t in ctx["cum"]]
    d_x = torch.empty_like(x)
    return (lambda: heads_forward_fused(heads, x, True, None, 1.0),
            lambda: heads_backward_fused(heads, ctx, d_cum, d_x=d_x))


def matcher_fns(B, T, Q, C):
    from boosted_detr_b200.losses_and_metrics import PreparedTargets, pairwise_cost
    rng = np.random.default_rng(C + B)
    tr = [torch.from_numpy(a).cuda() for a in synth_targets(rng, B, T, C, A, attr_p=0.05)[:3]]
    pr = [torch.from_numpy(a).cuda() for a in synth_preds(rng, B, Q, C, A)]
    prep = PreparedTargets(tr)
    return (lambda: PreparedTargets(tr), lambda: pairwise_cost(tr, pr, 1000.0, 1.0, 1.0, prepared=prep))


def config2_model(C):
    from boosted_detr_b200.boosted_model import BoostedDETR
    from boosted_detr_b200.parameters import baseline_params
    p = baseline_params(2)
    p["vocab_dict"] = {"category": [f"cat_{i}" for i in range(C - 2)], "attribute": ["<none>"]}
    model = BoostedDETR(**p, attribute_weight=1.0, seed=0).build()
    assert model.num_categories == C
    rng = np.random.default_rng(2)
    B, T = 16, 20
    cat, attr, box, n = synth_targets(rng, B, T, C, model.num_attributes, attr_p=0.05)
    feats = np.tanh(rng.standard_normal((B, 20, 20, 256))).astype(np.float32)
    model.dropout_seed = 2024
    return model, {"features": feats, "category": cat, "attribute": attr, "bbox": box, "num_objects": n}


def graphed_step(C):
    from boosted_detr_b200.graph import GraphedTrainStep
    model, inputs = config2_model(C)
    gs = GraphedTrainStep(model, inputs)
    assert model._use_fused(torch.empty(inputs["features"].shape)), "config-2 size must take the fused path"
    return gs.replay


FAMILIES = [("heads second Dense + activation", r"heads_out_kernel|head_act_fwd"),
            ("heads backward (activation, BatchNorm, d_h)", r"heads_act_bwd|heads_bn_bwd|heads_dh"),
            ("heads hidden layers and BatchNorm statistics", r"heads_bn_stats|heads_bn_finalize"),
            ("matcher digest + cost matrix", r"cost_targets|cost_matrix"),
            ("assignment", r"lsap"),
            ("matched loss", r"matched_loss|pairwise_iou"),
            ("optimizer", r"adam|optim|sgd"),
            ("copies and fills", r"Memcpy|Memset|memcpy|memset|fill|copy")]


def kernel_breakdown(C, steps=3):
    """GPU time per eager training step by kernel family (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    model, inputs = config2_model(C)
    for _ in range(2):
        model.train_step(inputs)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            model.train_step(inputs)
        torch.cuda.synchronize()
    fam = defaultdict(float)
    per_kernel = defaultdict(float)
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = e.cuda_time_total
        if us <= 0:
            continue
        name = next((f for f, pat in FAMILIES if re.search(pat, e.key)), "other (GEMM, attention, LayerNorm, ...)")
        fam[name] += us / steps / 1000.0
        per_kernel[e.key] += us / steps / 1000.0
    return dict(fam), dict(per_kernel)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    lib = _lib.load()
    lib.bdetr_set_mode(_lib.MODE_TF32)
    flush = torch.empty(64 * 1024 * 1024, device="cuda")          # 256 MiB > 126 MB of L2
    res = {"gpu": gpu_info(), "mode": "tf32", "timing": "median of CUDA-event brackets, L2 flushed between calls",
           "heads": {}, "matcher": {}, "train_step_config2": {}, "step_breakdown_ms": {}}

    def run(group, keys, make, calls, flops=None):
        fns = {k: make(k) for k in keys}
        for fn in fns.values():
            for _ in range(3):
                fn()
        torch.cuda.synchronize()
        ts = {k: [] for k in keys}
        for _ in range(args.rounds):
            for k in keys:
                ts[k] += time_calls(fns[k], flush, calls)
        for k in keys:
            ms = float(np.median(ts[k]))
            e = {"ms": ms, "spread_ms": [float(np.min(ts[k])), float(np.max(ts[k]))]}
            if flops:
                e["second_dense_gflop"] = flops(k) / 1e9
                e["second_dense_tflops_at_call_time"] = flops(k) / (ms * 1e-3) / 1e12
            res[group][k] = e
            print(group, k, f"{ms:.4f} ms", flush=True)
        del fns
        torch.cuda.empty_cache()

    hf = {C: heads_fns(C) for C in HEADS_C}
    run("heads", [f"fwd_C{C}" for C in HEADS_C], lambda k: hf[int(k[5:])][0], 20, lambda k: 2.0 * M * D * int(k[5:]))
    run("heads", [f"bwd_C{C}" for C in HEADS_C], lambda k: hf[int(k[5:])][1], 20)
    del hf
    for shape, (B, T, Q) in MATCH_SHAPES.items():
        mf = {C: matcher_fns(B, T, Q, C) for C in MATCH_C}
        run("matcher", [f"{shape}_digest_C{C}" for C in MATCH_C], lambda k: mf[int(k.rsplit("C", 1)[1])][0], 20)
        run("matcher", [f"{shape}_cost_C{C}" for C in MATCH_C], lambda k: mf[int(k.rsplit("C", 1)[1])][1], 20)
        del mf
    run("train_step_config2", [f"C{C}" for C in STEP_C], lambda k: graphed_step(int(k[1:])), 10)
    base = res["train_step_config2"]["C82"]["ms"]
    for C in STEP_C:
        res["train_step_config2"][f"C{C}"]["over_C82"] = res["train_step_config2"][f"C{C}"]["ms"] / base
    for C in (82, 1205):
        fam, per_kernel = kernel_breakdown(C)
        res["step_breakdown_ms"][f"C{C}"] = {"families": fam,
                                              "top_kernels": dict(sorted(per_kernel.items(), key=lambda kv: -kv[1])[:25])}
    a, b = res["step_breakdown_ms"]["C82"]["families"], res["step_breakdown_ms"]["C1205"]["families"]
    res["step_breakdown_ms"]["C1205_minus_C82"] = {f: b.get(f, 0.0) - a.get(f, 0.0) for f in sorted(set(a) | set(b))}
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
