"""Head dim 64 against head dim 32 at the same model width D = 256 (not a pytest file): H = 4 vs H = 8.

  * attention core forward (bdetr_attention_core_fwd) at the config-2 / config-4 / config-5 shapes, and the attention
    backward (bdetr_attention_block_bwd: LayerNorm, output projection and projection GEMMs included) where it is trained;
  * the CUDA-graphed training step at config-2 size (6 block pairs, batch 16, 20 x 20 features, 100 queries) with
    num_encoder_heads = num_decoder_heads = 4 against 8.

Tensor-core (tf32) mode.  CUDA events around each call or replay, L2 flushed (256 MiB write) outside the brackets, median
over the timed calls after warm-up; the two head layouts alternate round by round so that clock drift hits both.
Attention rates are 4 * Lq * Lk * D FLOP per image (QK^T and PV) over the forward time.

usage: python bench_tools/bench_head_dim.py [--out FILE.json] [--rounds N]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from boosted_detr_b200 import _lib  # noqa: E402
from boosted_detr_b200.device import ptr, stream_ptr  # noqa: E402

FWD_SHAPES = [(16, 400, 400), (16, 100, 400), (4, 1050, 1050), (4, 20020, 20020)]
BWD_SHAPES = [(16, 400, 400), (16, 100, 400), (4, 1050, 1050)]
HEADS = (8, 4)
D = 256


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


def core_fn(B, H, Lq, Lk):
    d = D // H
    q, k, v = (torch.randn(B, L, D, device="cuda") for L in (Lq, Lk, Lk))
    o, lse = torch.empty(B, H, Lq, d, device="cuda"), torch.empty(B, H, Lq, device="cuda")
    return lambda: _lib.call("bdetr_attention_core_fwd", B, H, Lq, Lk, d, ptr(q), ptr(k), ptr(v), ptr(o), ptr(lse), stream_ptr())


def block_bwd_fn(B, H, Lq, Lk):
    from boosted_detr_b200.layers import Layer
    from boosted_detr_b200.transformers import AttentionBlock
    Layer._rng = np.random.default_rng(1)
    blk = AttentionBlock(H, name="blk")
    q = torch.randn(B, Lq, D, device="cuda")
    kv = q if Lq == Lk else torch.randn(B, Lk, D, device="cuda")
    _, ctx = blk.forward([q, kv, kv], training=True)
    go = torch.randn(B, Lq, D, device="cuda")
    return lambda: blk.backward(ctx, go)


def graphed_step(H):
    from boosted_detr_b200.boosted_model import BoostedDETR
    from boosted_detr_b200.graph import GraphedTrainStep
    from boosted_detr_b200.parameters import baseline_params
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
    from util import synth_targets
    p = baseline_params(2)
    p.update(num_encoder_heads=H, num_decoder_heads=H)
    model = BoostedDETR(**p, attribute_weight=1.0, seed=0).build()
    rng = np.random.default_rng(2)
    B, T = 16, 20
    cat, attr, box, n = synth_targets(rng, B, T, model.num_categories, model.num_attributes, attr_p=0.05)
    feats = np.tanh(rng.standard_normal((B, 20, 20, 256))).astype(np.float32)
    inputs = {"features": feats, "category": cat, "attribute": attr, "bbox": box, "num_objects": n}
    model.dropout_seed = 2024
    gs = GraphedTrainStep(model, inputs)
    assert model._use_fused(torch.empty(feats.shape)), "config-2 size must take the fused path"
    return gs.replay


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    lib = _lib.load()
    lib.bdetr_set_mode(_lib.MODE_TF32)
    flush = torch.empty(64 * 1024 * 1024, device="cuda")          # 256 MiB > 126 MB of L2
    res = {"gpu": gpu_info(), "mode": "tf32", "D": D, "timing": "median of CUDA-event brackets, L2 flushed between calls",
           "attention_fwd": {}, "attention_block_bwd": {}, "train_step_config2": {}}

    def run(group, key_fn, make, calls, flops=None):
        fns = {H: make(H) for H in HEADS}
        for fn in fns.values():
            for _ in range(3):
                fn()
        torch.cuda.synchronize()
        ts = {H: [] for H in HEADS}
        for _ in range(args.rounds):
            for H in HEADS:
                ts[H] += time_calls(fns[H], flush, calls)
        for H in HEADS:
            ms = float(np.median(ts[H]))
            e = {"H": H, "d": D // H, "ms": ms, "spread_ms": [float(np.min(ts[H])), float(np.max(ts[H]))]}
            if flops:
                e["tflops"] = flops / (ms * 1e-3) / 1e12
            res[group][key_fn(H)] = e
            print(group, key_fn(H), f"{ms:.4f} ms", f"{e.get('tflops', 0):.1f} TFLOP/s" if flops else "", flush=True)
        del fns
        torch.cuda.empty_cache()

    for (B, Lq, Lk) in FWD_SHAPES:
        run("attention_fwd", lambda H: f"B{B}_Lq{Lq}_Lk{Lk}_H{H}", lambda H: core_fn(B, H, Lq, Lk),
            20 if Lq < 5000 else 3, 4.0 * B * Lq * Lk * D)
    for (B, Lq, Lk) in BWD_SHAPES:
        run("attention_block_bwd", lambda H: f"B{B}_Lq{Lq}_Lk{Lk}_H{H}", lambda H: block_bwd_fn(B, H, Lq, Lk), 20)
    run("train_step_config2", lambda H: f"H{H}", graphed_step, 20)
    s8, s4 = res["train_step_config2"]["H8"]["ms"], res["train_step_config2"]["H4"]["ms"]
    res["train_step_config2"]["h4_over_h8"] = s4 / s8
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
