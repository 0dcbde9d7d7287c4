#!/usr/bin/env python
"""Benchmark of the Boosted_DETR hot path (BASELINE.json metric: images/sec fwd+bwd+matcher; matcher us/image; roofline %).

  python bench.py --gpus N --steps K --warmup W [--config 2|3|4|5]   our arm (one process per GPU under torchrun)
  python bench.py --impl reference --gpus N ... [--config ...]       the restated reference CPU path (oracle/) on host cores
  python bench.py ... --dump-outputs DIR                             also writes the outputs of the last timed step (see
                                                                     dump_outputs) for an output-for-output comparison

BASELINE.json configs (SURVEY.md §8):
  2 (default, the headline line)  training step, 6 enc/dec pairs, d 256, 8 heads, 100 queries, 20x20 features, 16 images
                                  per GPU (weak scaling), T = 20, C = 82, A = 3
  3  the same model with the attribute head at Fashionpedia sizes (C = 48, A = 296), GLOBAL batch 64 split over the N
     GPUs (strong scaling), NCCL gradient all-reduce
  4  matcher only: 300 queries x up to 100 targets, 256 images per GPU: cost matrix + per-image assignment + matched loss
  5  high-resolution inference: 110 x 182 features = 20 020 encoder tokens (and the stride-32 faithful 25 x 42 = 1 050),
     6 pairs, 4 images per GPU
A step of a training config = forward of all boosted blocks, Hungarian matching loss at every block, backward, gradient
all-reduce when N > 1, and the reference's optimizer update.  Prints ONE JSON line on rank 0; without --config the line
is config 2's and carries compact results of configs 3, 4, 5 under "other_configs" (same run, same box), the matcher
figure of the metric under "matcher_us_per_image", and one roofline block per kernel family.
"""
from __future__ import annotations

import argparse
import glob
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "images/sec fwd+bwd+matcher"
CONFIGS = {
    2: dict(kind="train", N=6, B=16, rows=20, cols=20, Q=100, T=20, D=256, H=8, C=82, A=3, scaling="weak"),
    3: dict(kind="train", N=6, global_B=64, rows=20, cols=20, Q=100, T=20, D=256, H=8, C=48, A=296, scaling="strong"),
    4: dict(kind="matcher", B=256, Q=300, T=100, C=82, A=3, scaling="weak"),
    5: dict(kind="infer", N=6, B=4, rows=110, cols=182, Q=100, T=20, D=256, H=8, C=82, A=3, scaling="weak"),
}
CFG = CONFIGS[2]                                # kept for tools that import bench


def per_gpu_batch(cfg, world):
    if "global_B" in cfg:
        assert cfg["global_B"] % world == 0
        return cfg["global_B"] // world
    return cfg["B"]


def describe(cfg_id, cfg, B, world):
    if cfg["kind"] == "train":
        return (f"BASELINE config {cfg_id}: Boosted DETR, {cfg['N']} enc/dec pairs, d_model {cfg['D']}, {cfg['H']} heads, "
                f"{cfg['Q']} queries, {cfg['rows']}x{cfg['cols']} features (640x640/32), batch {B}/GPU"
                + (f" (global {cfg['global_B']}, strong scaling)" if "global_B" in cfg else "")
                + f", T={cfg['T']}, C={cfg['C']}, A={cfg['A']}, training step = fwd + Hungarian loss at every block + bwd "
                "(+ grad all-reduce when N>1) + SGD-Nesterov update (per-variable clipnorm .1, CosineDecayRestarts), dropout .1 on")
    if cfg["kind"] == "matcher":
        return (f"BASELINE config 4: matcher only, {cfg['Q']} queries x up to {cfg['T']} targets, {B} images/GPU, C={cfg['C']}, "
                f"A={cfg['A']}: target digest + cost matrix + per-image assignment (scipy-exact) + matched loss")
    return (f"BASELINE config 5: high-resolution inference, {cfg['rows']}x{cfg['cols']} features = {cfg['rows'] * cfg['cols']} encoder "
            f"tokens, {cfg['N']} enc/dec pairs, {cfg['Q']} queries, {B} images/GPU, forward only")


def synth_batch(rank, B, C, A, cfg=CFG):
    from util import synth_targets
    rng = np.random.default_rng(1234 + rank)
    cat, attr, box, n = synth_targets(rng, B, cfg["T"], C, A)
    x = np.tanh(rng.standard_normal((B, cfg["rows"], cfg["cols"], cfg["D"]), dtype=np.float32))
    x = ((x - x.mean((0, 1, 2))) / x.std((0, 1, 2))).astype(np.float32)      # mimics BN o tanh o BN (backbone.py:90-95)
    return {"features": x, "category": cat, "attribute": attr, "bbox": box, "num_objects": n}


def make_model(cfg=CFG, seed=0, training=True, cfg_id=2):
    from boosted_detr_b200.boosted_model import BoostedDETR
    from boosted_detr_b200.parameters import baseline_params
    p = baseline_params(3 if cfg["A"] > 3 else 2)
    p.update(num_decoder_blocks=cfg["N"], num_encoder_blocks=cfg["N"], num_object_preds=cfg["Q"],
             image_size=(cfg["rows"] * 32, cfg["cols"] * 32))
    model = BoostedDETR(**p, attribute_weight=1.0, seed=seed, feature_shape=(cfg["rows"], cfg["cols"])).build(batch_size=1)
    assert (model.num_categories, model.num_attributes) == (cfg["C"], cfg["A"])
    # throughput runs: queries N(0, 0.02^2) instead of the zero init (SURVEY.md §8d)
    rng = np.random.default_rng(seed)
    q0 = model.DecoderPrep._weights["init_decoder_features"]
    model.set_weights_dict({"DecoderPrep/init_decoder_features": rng.normal(0, 0.02, tuple(q0.shape)).astype(np.float32)})
    if training:
        model.dropout_seed = 2024                                           # training-mode dropout (rate .1) is on
        # the reference's optimizer (Boosted_DETR_COCO.ipynb cell 26): the timed step ends with its update
        from boosted_detr_b200.optimizers import SGD, CosineDecayRestarts
        model.compile(optimizer=SGD(learning_rate=CosineDecayRestarts(1e-3, 4000, m_mul=.95, alpha=.1), momentum=.9, nesterov=True, clipnorm=0.1))
    return model


def algorithmic_flops_per_step(cfg, B, C, A, training=True):
    """SURVEY.md §8d (2 flops/MAC, batch-invariant work hoisted)."""
    L, D, Q, N = cfg["rows"] * cfg["cols"], cfg["D"], cfg["Q"], cfg["N"]
    f_enc = 12 * L * D * D + 4 * L * L * D
    f_dec = 4 * L * D * D + 4 * Q * L * D + 8 * Q * D * D
    f_heads = 6 * Q * D * D + 2 * Q * D * (C + A + 4)
    f_self = 8 * Q * D * D + 4 * Q * Q * D
    return (3 if training else 1) * (B * N * (f_enc + f_dec + f_heads) + (N - 1) * f_self)


def cost_algorithmic_bytes(B, T, Q, C, A):
    """SURVEY.md §8d: every input read once, the cost matrix written once (fp32)."""
    return 4.0 * B * (Q * C + Q * A + 4 * Q + T * C + T * A + 4 * T + T * Q)


DUMP_MAX_ELEMENTS = 1 << 22         # per array; a larger one is reduced to a fixed, seeded sample of its elements
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(outputs, out_dir):
    """`--dump-outputs`: writes each output as `out_dir/<name>.npy` (float32, or float64 for integer arrays) so that two
    builds run with the same arguments can be compared output for output.  An array of more than DUMP_MAX_ELEMENTS is
    flattened and reduced to the elements at sorted indices drawn with seed 0, which depend only on its size."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {}
    for name, a in outputs.items():
        a = np.asarray(a)
        a = a.astype(np.float32 if a.dtype.kind == "f" and a.dtype.itemsize <= 4 else np.float64)
        if a.size > DUMP_MAX_ELEMENTS:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMENTS, replace=False))]
        arrays[name] = a
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_MAX_BYTES}-byte limit")
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([f.strip() for f in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(s) > 2 + i and s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.samples)}


def time_kernel(fn, reps=50, iters=7, flush=None):
    """Average device time of one launch: `reps` back-to-back launches captured in a CUDA graph (no host launch
    gaps; a single launch bracketed by events is floored at ~10 us by the event/launch overhead), median of
    `iters` replays, CUDA events on the launching stream, L2 flushed before each replay."""
    import torch
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    ts = []
    for _ in range(iters):
        if flush is not None:
            flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); g.replay(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) / reps)
    return float(np.median(ts)) * 1e-3        # seconds


def ncu_traffic(kernel_substr):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the named kernel, read from the newest committed
    `profiles/*ncu_full*.csv` that lists it (tools/summarise_ncu.py output of an `ncu --set full` capture: header row,
    units row, one row per launch).  Returns (bytes or None, file name or None)."""
    import csv
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    best = (None, None)
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "*ncu_full*.csv"))):
        try:
            rows = list(csv.reader(open(path)))
            h, units = rows[0], rows[1]
            ki, ri, wi = h.index("Kernel Name"), h.index("dram__bytes_read.sum"), h.index("dram__bytes_write.sum")
        except Exception:
            continue
        for r in rows[2:]:
            if len(r) <= max(ki, ri, wi) or kernel_substr not in r[ki]:
                continue
            try:
                val = float(r[ri]) * scale.get(units[ri], 1.0) + float(r[wi]) * scale.get(units[wi], 1.0)
            except ValueError:
                continue
            best = (val, os.path.basename(path))
            break
    return best


def peaks_json():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def roofline_blocks(cfg, B, flush, peaks):
    """One roofline block per kernel family, each kernel timed ALONE, live, with CUDA events: the Dense GEMM of the
    training step (dominant family of config 2), the attention core at config 2's L = 400 and at config 5's
    L = 20 020 (tensor pipe), the cost-matrix kernels at config 4 for both vocabularies (HBM)."""
    import torch
    from boosted_detr_b200 import _lib
    from boosted_detr_b200.device import ptr, stream_ptr
    from util import synth_preds, synth_targets
    L, D, H = cfg["rows"] * cfg["cols"], cfg["D"], cfg["H"]
    mode = _lib.load().bdetr_get_mode()
    tpeak = peaks.get("bf16_tflops", 1590.0)
    hpeak = peaks.get("hbm_gbs", 6650.0)
    src = "MEASURED_PEAKS.json (burst figures, kernel timed alone)" if peaks else "fallback 1590 TFLOP/s / 6650 GB/s (B200_PROFILING.md)"
    M = B * L
    import ctypes
    x = torch.randn(M, D, device="cuda"); wt = [torch.randn(D, D, device="cuda") for _ in range(3)]
    bias = [torch.randn(D, device="cuda") for _ in range(3)]
    y = [torch.empty(M, D, device="cuda") for _ in range(3)]
    if mode:
        # the dominant GEMM of the fused path: the grouped q/k/v projection of one encoder block, [M,256] x 3 x [256,256]
        # (bdetr_pos_projection is the same grouped tcgen05 launch: one shared input, three weight / bias / output groups)
        Ws, bs, ys = _lib.PTR3(*[t.data_ptr() for t in wt]), _lib.PTR3(*[t.data_ptr() for t in bias]), _lib.PTR3(*[t.data_ptr() for t in y])
        fn = lambda: _lib.call("bdetr_pos_projection", M, D, ptr(x), 3, ctypes.byref(Ws), ctypes.byref(bs), ctypes.byref(ys), stream_ptr())
        flops, name = 2.0 * M * 3 * D * D, f"gemm_umma_kernel<128,...> grouped q/k/v projection [{M},{D}] x 3 x [{D},{D}]"
        ncu_name = "gemm_umma_kernel<128, 3, 0, 1>"
    else:
        fn = lambda: _lib.call("bdetr_gemm", M, D, D, ptr(x), 0, ptr(wt[0]), 0, ptr(bias[0]), 0, 0, ptr(y[0]), stream_ptr())
        flops, name, ncu_name = 2.0 * M * D * D, f"gemm_simt_kernel (Dense forward [{M},{D}]x[{D},{D}])", "gemm_simt_kernel"
    t_gemm = time_kernel(fn, flush=flush)
    ach = flops / t_gemm / 1e12
    traffic, traffic_src = ncu_traffic(ncu_name) if mode else (None, None)
    main = {"bound": "tensor", "kernel": name,
            "achieved": ach, "peak": tpeak, "unit": "TFLOP/s", "frac": ach / tpeak, "traffic": traffic, "traffic_source": traffic_src,
            "algorithmic_bytes": 4.0 * (M * D + 3 * D * D + 3 * M * D) if mode else 4.0 * (2 * M * D + D * D),
            "peak_source": src, "us_per_launch": t_gemm * 1e6, "mode": "tf32" if mode else "fp32",
            "note": "peak is the measured bf16 cuBLAS figure; the TF32 tensor peak is half of it"}
    others = {}

    def attn(Ba, La, reps):
        q, k, v = (torch.randn(Ba, La, D, device="cuda") for _ in range(3))
        o, lse = torch.empty(Ba, H, La, D // H, device="cuda"), torch.empty(Ba, H, La, device="cuda")
        t = time_kernel(lambda: _lib.call("bdetr_attention_core_fwd", Ba, H, La, La, D // H, ptr(q), ptr(k), ptr(v), ptr(o), ptr(lse), stream_ptr()),
                        reps=reps, iters=5, flush=flush)
        a = 4.0 * Ba * La * La * D / t / 1e12
        return {"bound": "tensor", "achieved": a, "peak": tpeak, "unit": "TFLOP/s", "frac": a / tpeak, "us_per_launch": t * 1e6,
                "shape": [Ba, H, La, La]}
    others["attention_core_fwd_L400"] = attn(B, L, 50)
    if mode:
        others["attention_core_fwd_L20020_config5"] = attn(2, 20020, 2)
        tr_, src_ = ncu_traffic("attention_fwd_umma_ms_kernel")
        others["attention_core_fwd_L20020_config5"].update(traffic=tr_, traffic_source=src_)
        # the fp16-operand kernel of BDETR_MODE_FP16 (cast of q / k / v included in the timed launch pair)
        q, k, v = (torch.randn(2, 20020, D, device="cuda") for _ in range(3))
        o, lse = torch.empty(2, H, 20020, D // H, device="cuda"), torch.empty(2, H, 20020, device="cuda")
        ws = torch.empty(_lib.load().bdetr_attention_f16_workspace_bytes(2, H, 20020, 20020, D // H) // 2, dtype=torch.float16, device="cuda")
        t16 = time_kernel(lambda: _lib.call("bdetr_attention_core_fwd_f16", 2, H, 20020, 20020, D // H, ptr(q), ptr(k), ptr(v), ptr(ws), ptr(o),
                                            ptr(lse), stream_ptr()), reps=2, iters=5, flush=flush)
        a16 = 4.0 * 2 * 20020 * 20020 * D / t16 / 1e12
        tr_, src_ = ncu_traffic("attention_fwd_umma_ms_f16")
        others["attention_core_fwd_L20020_config5_fp16"] = {"bound": "tensor", "achieved": a16, "peak": tpeak, "unit": "TFLOP/s", "frac": a16 / tpeak,
                                                            "us_per_launch": t16 * 1e6, "shape": [2, H, 20020, 20020], "traffic": tr_,
                                                            "traffic_source": src_, "note": "cast_f16x3_kernel + attention_fwd_umma_ms_f16_kernel"}
        del q, k, v, o, lse, ws
    for name, (C, A) in (("cost_matrix_config4_C82_A3", (82, 3)), ("cost_matrix_config4_C48_A296", (48, 296))):
        rng = np.random.default_rng(0)
        Bm, T, Q = 256, 100, 300
        tr = synth_targets(rng, Bm, T, C, A); pr = synth_preds(rng, Bm, Q, C, A)
        d = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (*tr, *pr)]
        cost = torch.empty(Bm, T, Q, device="cuda")
        prep = torch.empty(_lib.load().bdetr_cost_targets_bytes(Bm, T, C, A), dtype=torch.uint8, device="cuda")
        f_all = lambda: (_lib.call("bdetr_cost_targets_prepare", Bm, T, C, A, ptr(d[0]), ptr(d[1]), ptr(d[2]), ptr(prep), stream_ptr()),
                         _lib.call("bdetr_cost_matrix_prepared", Bm, T, Q, C, A, ptr(prep), ptr(d[4]), ptr(d[5]), ptr(d[6]), 1000.0, 1.0, 1.0, ptr(cost), stream_ptr()))
        f_pairs = lambda: _lib.call("bdetr_cost_matrix_prepared", Bm, T, Q, C, A, ptr(prep), ptr(d[4]), ptr(d[5]), ptr(d[6]), 1000.0, 1.0, 1.0, ptr(cost), stream_ptr())
        t_all = time_kernel(f_all, reps=20, flush=flush)
        t_pairs = time_kernel(f_pairs, reps=20, flush=flush)
        nbytes = cost_algorithmic_bytes(Bm, T, Q, C, A)
        tr_, src_ = ncu_traffic("cost_matrix_kernel")
        others[name] = {"bound": "hbm", "achieved": nbytes / t_all / 1e9, "peak": hpeak, "unit": "GB/s", "frac": nbytes / t_all / 1e9 / hpeak,
                        "us_per_launch": t_all * 1e6, "pair_kernel_us": t_pairs * 1e6, "algorithmic_bytes": nbytes,
                        "traffic": tr_ if A == 3 else None, "traffic_source": src_ if A == 3 else None,
                        "note": "target digest + pair kernel back to back; algorithmic bytes = inputs once + cost once"}
    main["other_kernels"] = others
    return main


# ---------------------------------------------------------------------------------------------------------------------
# CPU legs (the restated reference path, oracle/): only bench.py's cpu_baseline / --impl reference may run these
# ---------------------------------------------------------------------------------------------------------------------
def host_weights(cfg, C, A, seed=0):
    from util import make_weights
    rng = np.random.default_rng(seed)
    w = make_weights(rng, cfg["N"], cfg["rows"], cfg["cols"], cfg["D"], cfg["Q"], C, A, perturb=False)
    return w


def cpu_reference_train_steps(cfg, B, C, A, steps, warmup, threads):
    """The restated reference CPU path (oracle/reference_path.py, torch CPU fp32) on the host cores: full training step
    including the SGD update."""
    import torch
    from oracle import reference_path as R
    torch.set_num_threads(threads)
    w = host_weights(cfg, C, A)
    batch = synth_batch(0, B, C, A, cfg)
    tg = (batch["category"], batch["attribute"], batch["bbox"], batch["num_objects"])
    times, acc = [], {}
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        _, grads, stats = R.train_step_reference(w, batch["features"], tg, cfg["N"], cfg["H"], torch.float32, dropout_seed=2024,
                                                 weights=R.model_weights(1.0))
        if not acc:
            acc = {k: np.zeros_like(v, dtype=np.float32) for k, v in grads.items()}
        lr = R.cosine_decay_restarts(it, 1e-3, 4000, 2.0, .95, .1)
        new_w, acc = R.sgd_step_reference({k: w[k] for k in grads}, grads, acc, lr, .9, True, .1, dtype=np.float32)
        w.update(new_w)
        w.update({k: np.asarray(v, np.float32) for k, v in stats.items()})
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    return float(np.mean(times))


def cpu_reference_matcher(cfg, sample_B, steps, warmup, threads):
    """The reference's literal matcher path on the host: broadcast cost arrays (oracle weighted_cost, torch CPU fp32) ->
    python loop over images -> scipy.optimize.linear_sum_assignment -> matched loss.  Returns seconds per image."""
    import torch
    from oracle import reference_path as R
    from util import synth_preds, synth_targets
    torch.set_num_threads(threads)
    rng = np.random.default_rng(1234)
    tr = synth_targets(rng, sample_B, cfg["T"], cfg["C"], cfg["A"])
    pr = synth_preds(rng, sample_B, cfg["Q"], cfg["C"], cfg["A"])
    y_true = [torch.tensor(tr[0]), torch.tensor(tr[1]), torch.tensor(tr[2]), tr[3]]
    y_pred = [torch.tensor(p) for p in pr]
    ts = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        R.matching_loss(y_true, y_pred, R.model_weights(1.0))
        if it >= warmup:
            ts.append(time.perf_counter() - t0)
    return float(np.mean(ts)) / sample_B


def cpu_reference_infer(cfg, sample_B, steps, warmup, threads):
    """Restated reference inference (oracle boosted_detr_call, torch CPU fp32); attention evaluated in query-row slices
    so that the [B,H,L,L] scores of a 20 020-token image fit in host memory (same arithmetic).  Seconds per image."""
    import torch
    from oracle import reference_path as R
    torch.set_num_threads(threads)
    R.ATTENTION_QUERY_CHUNK = 2048
    w = R.params_to_torch(host_weights(cfg, cfg["C"], cfg["A"]), torch.float32)
    feats = torch.tensor(synth_batch(0, sample_B, cfg["C"], cfg["A"], cfg)["features"])
    ts = []
    with torch.no_grad():
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            R.boosted_detr_call(w, feats, None, cfg["N"], cfg["H"], training=False)
            if it >= warmup:
                ts.append(time.perf_counter() - t0)
    R.ATTENTION_QUERY_CHUNK = 0
    return float(np.mean(ts)) / sample_B


def reference_arm(cfg_id, cfg, args, cores):
    """`--impl reference`: the reference's own CPU implementation of the path (its restatement in oracle/: TensorFlow is
    not installable here) on all host cores, same config / metric / unit, each step a bounded sample."""
    B = per_gpu_batch(cfg, 1 if cfg["scaling"] == "strong" else 1)
    steps, warm = max(1, min(args.steps, 3)), min(args.warmup, 1)
    if cfg["kind"] == "train":
        B = cfg.get("global_B", cfg.get("B"))
        sample_B = min(B, 16)
        sec = cpu_reference_train_steps(cfg, sample_B, cfg["C"], cfg["A"], steps, warm, cores)
        val, sample = sample_B / sec, f"{steps} full training steps of {sample_B} images (oracle/reference_path.py, torch CPU fp32, {cores} threads; TF unavailable)"
        ms = sec * 1e3
    elif cfg["kind"] == "matcher":
        sample_B = 32
        spi = cpu_reference_matcher(cfg, sample_B, steps, warm, cores)
        val, sample, ms = 1.0 / spi, f"{steps} passes over {sample_B} of the {cfg['B']} images: broadcast cost arrays + scipy loop + matched loss (oracle, torch CPU fp32, {cores} threads)", spi * cfg["B"] * 1e3
    else:
        spi = cpu_reference_infer(cfg, 1, min(steps, 2), warm, cores)
        val, sample, ms = 1.0 / spi, f"{min(steps, 2)} forward passes of 1 of the {cfg['B']} images at {cfg['rows'] * cfg['cols']} tokens (oracle, torch CPU fp32, {cores} threads, attention in 2048-query slices)", spi * cfg["B"] * 1e3
    return {"impl": "reference", "metric": METRIC, "value": val, "unit": "images/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": ms, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "fp32",
            "data": "synthetic", "config": {"workload": describe(cfg_id, cfg, cfg.get("global_B", cfg.get("B")), 1)}, "gpu_launches": 0,
            "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


# ---------------------------------------------------------------------------------------------------------------------
# GPU legs
# ---------------------------------------------------------------------------------------------------------------------
class Ctx:
    """rank / world / timing helpers shared by the GPU legs."""

    def __init__(self, rank, world, local, args, flush):
        self.rank, self.world, self.local, self.args, self.flush = rank, world, local, args, flush

    def barrier(self):
        import torch
        import torch.distributed as dist
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, seconds):
        import torch
        import torch.distributed as dist
        t = torch.tensor([seconds], device="cuda", dtype=torch.float64)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed_device(self, step, steps, reset=None):
        """EXACTLY `steps` steps, each bracketed by CUDA events on the launching stream with `reset()` (when given) and an
        L2 flush (256 MiB write) outside the brackets; barrier + synchronize on both sides; max over ranks of the summed time."""
        import torch
        times = []
        self.barrier()
        for _ in range(steps):
            if reset is not None:
                reset()
            self.flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); step(); b.record()
            b.synchronize()
            times.append(a.elapsed_time(b))
        self.barrier()
        return self.max_over_ranks(sum(times) / 1e3) / steps

    def timed_e2e(self, fn, steps):
        import torch
        for _ in range(3):
            out = fn()
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            out = fn()
        torch.cuda.synchronize()
        return self.max_over_ranks(time.perf_counter() - t0) / steps, out


def run_train(cx, cfg_id, cfg, outputs=None):
    """`outputs` (optional dict): receives what the last timed step computed, as host arrays."""
    import torch
    from boosted_detr_b200 import _lib
    from boosted_detr_b200.graph import GraphedTrainStep
    from boosted_detr_b200.parallel import DataParallel
    args, world, rank = cx.args, cx.world, cx.rank
    lib = _lib.load()
    B, C, A = per_gpu_batch(cfg, world), cfg["C"], cfg["A"]
    model = make_model(cfg, cfg_id=cfg_id)
    DataParallel(model, overlap=not args.no_overlap)
    # The state a step updates in place: the weights, the BatchNorm moving statistics and the optimizer's momentum (zero
    # before the first update).  The split-K weight gradients accumulate with float reduce-adds, so consecutive steps
    # drift apart from run to run; restoring the initial state before every device-timed step makes each of them --
    # and the last one, whose outputs --dump-outputs writes -- compute the same thing from the same inputs in every run.
    in_place = [model._flat[0]] + [o._weights[k] for _, o, k in model.named_weights() if k in o._non_trainable]
    initial = [t.clone() for t in in_place]

    def reset():
        for t, t0 in zip(in_place, initial):
            t.copy_(t0)
        if model.optimizer._accum is not None:
            model.optimizer._accum.zero_()
    batch = synth_batch(rank, B, C, A, cfg)
    if args.no_graph:
        dev_batch = {k: torch.from_numpy(v).cuda() for k, v in batch.items()}
        step = lambda: model.train_step(dev_batch, return_host=False)
    else:
        gs = GraphedTrainStep(model, batch)
        step = gs.replay
    for _ in range(max(args.warmup, 3)):
        step()
    # ---- end-to-end: public API with HOST buffers (pinned H2D in, metric means + matcher status D2H out) every step.
    # The next batch's H2D copy is queued right behind the running step's launch (GraphedTrainStep prefetch).
    host_batch = {k: torch.from_numpy(np.ascontiguousarray(v, np.int32 if k == "num_objects" else np.float32)).pin_memory()
                  for k, v in batch.items()}
    host_batch2 = {k: v.clone().pin_memory() for k, v in host_batch.items()}
    prefetch = os.environ.get("BDETR_E2E_PREFETCH", "1") == "1" and not args.no_graph
    if args.no_graph:
        e2e_fn = lambda: model.train_step(batch)
    elif prefetch:
        pair = [host_batch, host_batch2]
        state = {"i": 0}

        def e2e_fn():
            cur, nxt = pair[state["i"] & 1], pair[(state["i"] + 1) & 1]
            state["i"] += 1
            return gs(cur, prefetch=nxt)
    else:
        e2e_fn = lambda: gs(host_batch)
    e2e_sec, logs = cx.timed_e2e(e2e_fn, args.steps)
    # ---- device arm (the headline): inputs resident in HBM, each step from the initial state (reset outside the brackets)
    sec = cx.timed_device(step, args.steps, reset)
    if outputs is not None:
        # what a caller of the step holds after it: the metric tensors and the updated variables (by variable name, so
        # that the layout of the flat buffer does not enter the comparison)
        outputs.update({k: v.float().cpu().numpy() for k, v in model.metric_tensors.items()})
        outputs["metric_means"] = model.metric_means.cpu().numpy()
        w = model.get_weights_dict()
        outputs["weights"] = np.concatenate([w[n].reshape(-1) for n in sorted(w)])
    h2d = sum(v.nbytes for v in batch.values())
    d2h = 4 * 6 + 4 * cfg["N"] * B                         # six metric means + per-block, per-image matcher status flags
    launches = None
    if rank == 0 or world == 1:
        pass
    res = {"value": B * world / sec, "ms_per_step": sec * 1e3, "per_gpu_batch": B, "global_batch": B * world,
           "e2e": {"value": B * world / e2e_sec, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                   "ms_per_step": e2e_sec * 1e3, "input_prefetch": prefetch},
           "loss": logs.get("loss") if isinstance(logs, dict) else None,
           "step_algorithmic_tflops": algorithmic_flops_per_step(cfg, B, C, A) / sec / 1e12,
           "parameters": model.num_parameters()}
    return res, model, batch


def count_launches(model, batch):
    """Kernels of ONE step, counted by running it eagerly (rank 0 only, collectives detached)."""
    import torch
    from boosted_detr_b200 import _lib
    lib = _lib.load()
    dev_batch = {k: torch.from_numpy(v).cuda() for k, v in batch.items()}
    model.grad_allreduce = model.grad_bucket_hook = None
    lib.bdetr_reset_launch_count()
    model.train_step(dev_batch, return_host=False)
    torch.cuda.synchronize()
    return int(lib.bdetr_launch_count())


def run_matcher(cx, cfg, outputs=None):
    """Config 4.  Device arm: inputs resident in HBM.  e2e arm: MatchingLoss public call on pinned HOST arrays (H2D of
    targets + predictions, D2H of the [5,B] losses, the [B,T] assignment and the status flags).  `outputs` as in
    run_train."""
    import torch
    from boosted_detr_b200 import _lib
    from boosted_detr_b200.device import ptr, stream_ptr
    from boosted_detr_b200.losses_and_metrics import raise_for_status
    from util import synth_preds, synth_targets
    lib = _lib.load()
    B, T, Q, C, A = cfg["B"], cfg["T"], cfg["Q"], cfg["C"], cfg["A"]
    rng = np.random.default_rng(1234 + cx.rank)
    tr = synth_targets(rng, B, T, C, A); pr = synth_preds(rng, B, Q, C, A)
    host = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in (*tr, *pr)]
    d = [h.cuda() for h in host]
    cost = torch.empty(B, T, Q, device="cuda")
    prep = torch.empty(lib.bdetr_cost_targets_bytes(B, T, C, A), dtype=torch.uint8, device="cuda")
    c4r = torch.empty(B, T, dtype=torch.int32, device="cuda"); r4c = torch.empty(B, Q, dtype=torch.int32, device="cuda")
    st = torch.empty(B, dtype=torch.int32, device="cuda")
    losses = torch.empty(5, B, device="cuda"); iou = torch.empty(Q, device="cuda")
    h_out = (torch.empty(5, B).pin_memory(), torch.empty(B, T, dtype=torch.int32).pin_memory(), torch.empty(B, dtype=torch.int32).pin_memory())

    def step():
        s = stream_ptr()
        _lib.call("bdetr_cost_targets_prepare", B, T, C, A, ptr(d[0]), ptr(d[1]), ptr(d[2]), ptr(prep), s)
        _lib.call("bdetr_cost_matrix_prepared", B, T, Q, C, A, ptr(prep), ptr(d[4]), ptr(d[5]), ptr(d[6]), 1000.0, 1.0, 1.0, ptr(cost), s)
        _lib.call("bdetr_lsap_assign", B, T, Q, ptr(cost), ptr(d[3]), ptr(c4r), ptr(r4c), None, None, ptr(st), s)
        _lib.call("bdetr_matched_loss_fwd", B, T, Q, C, A, ptr(d[0]), ptr(d[1]), ptr(d[2]), ptr(d[3]), ptr(d[4]), ptr(d[5]), ptr(d[6]),
                  ptr(c4r), ptr(r4c), 1000.0, 1.0, 1.0, 100.0, ptr(losses), ptr(iou), s)

    for _ in range(3):
        step()
    lib.bdetr_reset_launch_count()
    step()
    torch.cuda.synchronize()
    launches = int(lib.bdetr_launch_count())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step()
    sec = cx.timed_device(g.replay, cx.args.steps)

    def e2e():
        for h, dv in zip(host, d):
            dv.copy_(h, non_blocking=True)
        g.replay()
        h_out[0].copy_(losses, non_blocking=True); h_out[1].copy_(c4r, non_blocking=True); h_out[2].copy_(st, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        raise_for_status(h_out[2])
        return h_out[0]
    e2e_sec, _ = cx.timed_e2e(e2e, cx.args.steps)
    if outputs is not None:
        outputs.update(losses=h_out[0].numpy().copy(), assignment=h_out[1].numpy().astype(np.float64), iou=iou.cpu().numpy())
    # the pieces, each alone (graph of 20 back-to-back launches, L2 flushed)
    s = stream_ptr
    parts = {
        "targets_prepare_us": time_kernel(lambda: _lib.call("bdetr_cost_targets_prepare", B, T, C, A, ptr(d[0]), ptr(d[1]), ptr(d[2]), ptr(prep), s()), reps=20, iters=5, flush=cx.flush) * 1e6,
        "cost_pairs_us": time_kernel(lambda: _lib.call("bdetr_cost_matrix_prepared", B, T, Q, C, A, ptr(prep), ptr(d[4]), ptr(d[5]), ptr(d[6]), 1000.0, 1.0, 1.0, ptr(cost), s()), reps=20, iters=5, flush=cx.flush) * 1e6,
        "lsap_us": time_kernel(lambda: _lib.call("bdetr_lsap_assign", B, T, Q, ptr(cost), ptr(d[3]), ptr(c4r), ptr(r4c), None, None, ptr(st), s()), reps=10, iters=5, flush=cx.flush) * 1e6,
        "matched_loss_us": time_kernel(lambda: _lib.call("bdetr_matched_loss_fwd", B, T, Q, C, A, ptr(d[0]), ptr(d[1]), ptr(d[2]), ptr(d[3]), ptr(d[4]), ptr(d[5]), ptr(d[6]),
                                                         ptr(c4r), ptr(r4c), 1000.0, 1.0, 1.0, 100.0, ptr(losses), ptr(iou), s()), reps=20, iters=5, flush=cx.flush) * 1e6}
    h2d = sum(h.numel() * h.element_size() for h in host)
    d2h = sum(h.numel() * h.element_size() for h in h_out)
    world = cx.world
    return {"value": B * world / sec, "ms_per_step": sec * 1e3, "per_gpu_batch": B, "global_batch": B * world,
            "matcher_us_per_image": sec / B * 1e6, "parts": parts, "launches_per_step": launches,
            "e2e": {"value": B * world / e2e_sec, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_sec * 1e3, "us_per_image": e2e_sec / B * 1e6}}


def run_infer(cx, cfg, also_faithful=True, outputs=None):
    """Config 5: inference only.  Device arm: features resident in HBM; e2e arm: `model(inputs)` on pinned host features
    (H2D every step) + D2H of the three prediction tensors.  `outputs` as in run_train (the full-size variant)."""
    import torch
    from boosted_detr_b200 import _lib
    lib = _lib.load()
    out = {}
    variants = [("", cfg)]
    if also_faithful:
        variants.append(("stride32_1050_tokens", dict(cfg, rows=25, cols=42)))
    for tag, c in variants:
        B = c["B"]
        model = make_model(c, training=False)
        feats_h = torch.from_numpy(synth_batch(cx.rank, B, c["C"], c["A"], c)["features"]).pin_memory()
        feats = feats_h.cuda()
        fn = lambda: model.call({"features": feats}, training=False)
        for _ in range(2):
            fn()
        lib.bdetr_reset_launch_count()
        preds = fn()
        torch.cuda.synchronize()
        launches = int(lib.bdetr_launch_count())
        assert all(bool(torch.isfinite(t).all()) for t in preds)
        steps = cx.args.steps
        sec = cx.timed_device(fn, steps)
        hp = [torch.empty(t.shape).pin_memory() for t in preds]

        def e2e():
            p = model.call({"features": feats_h}, training=False)
            for h, t in zip(hp, p):
                h.copy_(t, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return hp
        e2e_sec, last = cx.timed_e2e(e2e, steps)
        if outputs is not None and not tag:
            outputs.update({k: h.numpy().copy() for k, h in zip(("category", "attribute", "bbox"), last)})
        flops = algorithmic_flops_per_step(c, B, c["C"], c["A"], training=False)
        r = {"value": B * cx.world / sec, "ms_per_step": sec * 1e3, "per_gpu_batch": B, "global_batch": B * cx.world, "steps": steps,
             "tokens": c["rows"] * c["cols"], "algorithmic_tflops": flops / sec / 1e12, "launches_per_step": launches,
             "e2e": {"value": B * cx.world / e2e_sec, "unit": "images/s", "h2d_bytes_per_step": feats_h.numel() * 4,
                     "d2h_bytes_per_step": sum(h.numel() * 4 for h in hp), "ms_per_step": e2e_sec * 1e3}}
        if not tag and lib.bdetr_get_mode() == _lib.MODE_TF32:
            # the same forward with fp16 attention operands (BDETR_MODE_FP16 = the reference's mixed_float16 policy)
            lib.bdetr_set_mode(_lib.MODE_FP16)
            try:
                for _ in range(2):
                    fn()
                p16 = fn()
                torch.cuda.synchronize()
                sec16 = cx.timed_device(fn, steps)
                e2e16, _ = cx.timed_e2e(e2e, steps)
                dev = max(float((a - b).abs().max() / b.abs().max().clamp_min(1e-30)) for a, b in zip(p16, preds))
                r["fp16_operands"] = {"value": B * cx.world / sec16, "ms_per_step": sec16 * 1e3, "algorithmic_tflops": flops / sec16 / 1e12,
                                      "e2e": {"value": B * cx.world / e2e16, "unit": "images/s", "ms_per_step": e2e16 * 1e3},
                                      "max_normalised_prediction_difference_vs_tf32": dev}
            finally:
                lib.bdetr_set_mode(_lib.MODE_TF32)
        if tag:
            out[tag] = r
        else:
            out.update(r)
        del model, feats, feats_h
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5])
    ap.add_argument("--no-extras", action="store_true", help="config 2 only: skip the compact configs 3 / 4 / 5 blocks")
    ap.add_argument("--mode", default=os.environ.get("BDETR_MODE", "tf32"), choices=["fp32", "tf32", "fp16"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-overlap", action="store_true", help="one gradient all-reduce after the backward instead of per-block buckets under it")
    ap.add_argument("--no-conc", action="store_true", help="disable multi-stream concurrency inside the step (A/B timing)")
    ap.add_argument("--no-pdl", action="store_true", help="disable programmatic dependent launch (A/B timing)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--max-seconds", type=float, default=540.0, help="hard wall-clock limit: a wedged run prints what it has and exits")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path computed in its last step as DIR/<name>.npy "
                    "(rank 0; --impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cfg_id, cfg = args.config, CONFIGS[args.config]
    cores = os.cpu_count() or 1
    state = {"line": None}
    t_start = time.time()

    def _watchdog():
        time.sleep(args.max_seconds)
        sys.stderr.write(f"bench.py: exceeded --max-seconds {args.max_seconds:.0f}\n")
        if rank == 0 and state["line"] is not None:          # the headline was measured: print it rather than lose it
            state["line"]["aborted"] = "wall-clock limit reached during the secondary blocks"
            print(json.dumps(state["line"]), flush=True)
            os._exit(0)
        os._exit(3)
    threading.Thread(target=_watchdog, daemon=True).start()

    if args.impl == "reference":
        if rank != 0:
            return
        print(json.dumps(reference_arm(cfg_id, cfg, args, cores)))
        return

    import torch
    from boosted_detr_b200 import _lib
    from boosted_detr_b200.parallel import init_from_env
    rank, world, local = init_from_env()
    torch.cuda.set_device(local)
    lib = _lib.load()
    lib.bdetr_set_mode({"tf32": _lib.MODE_TF32, "fp16": _lib.MODE_FP16, "fp32": _lib.MODE_FP32}[args.mode])
    lib.bdetr_set_pdl(0 if args.no_pdl else 1)
    lib.bdetr_set_concurrency(0 if args.no_conc else 1)
    flush = torch.empty(256 * 1024 * 1024 // 4, device="cuda")
    cx = Ctx(rank, world, local, args, flush)
    B = per_gpu_batch(cfg, world)
    config = {"workload": describe(cfg_id, cfg, B, world), "per_gpu_batch": B, "global_batch": B * world, "parallelism": f"dp{world}",
              "l2": "flushed between timed steps (256 MiB write outside the event brackets); per-step CUDA events"}
    sampler = ClockSampler(local)
    if rank == 0:                                                # one nvidia-smi poller per job, not one per GPU
        sampler.start()

    model = batch = None
    outputs = {} if args.dump_outputs and rank == 0 else None
    if cfg["kind"] == "train":
        main_res, model, batch = run_train(cx, cfg_id, cfg, outputs)
    elif cfg["kind"] == "matcher":
        main_res = run_matcher(cx, cfg, outputs)
    else:
        main_res = run_infer(cx, cfg, outputs=outputs)
    if outputs is not None:
        dump_outputs(outputs, args.dump_outputs)
    sampler.stop_flag = True
    line = None
    if rank == 0:
        sampler.join(timeout=2)
        line = {"metric": METRIC, "value": main_res["value"], "unit": "images/s", "n_gpus": world, "steps": main_res.get("steps", args.steps),
                "warmup": max(args.warmup, 3), "ms_per_step": main_res["ms_per_step"], "higher_is_better": True, "scaling": cfg["scaling"],
                "vs_baseline": None, "dtype": args.mode, "data": "synthetic (random-init weights)",
                "config": config, "clocks": sampler.summary(), "e2e": main_res["e2e"],
                "cuda_graph": not args.no_graph, "pdl": not args.no_pdl, "concurrent_streams": not args.no_conc,
                "allreduce": ("none" if world == 1 or cfg["kind"] != "train" else "one call after backward" if args.no_overlap else
                              "per-block buckets overlapped with backward, inside the CUDA graph")}
        for k in ("loss", "step_algorithmic_tflops", "matcher_us_per_image", "parts", "tokens", "algorithmic_tflops", "stride32_1050_tokens", "parameters", "fp16_operands"):
            if k in main_res:
                line[k] = main_res[k]
        state["line"] = line

    # ---- compact blocks for the other BASELINE configs (same run, same box; every rank takes part) -----------------
    others = {}
    if cfg_id == 2 and not args.no_extras:
        if model is not None:
            model.grad_allreduce = model.grad_bucket_hook = None
        for oid in (4, 5, 3):
            ocfg = CONFIGS[oid]
            if time.time() - t_start > args.max_seconds * 0.55:
                others[str(oid)] = {"skipped": "time budget"}
                continue
            try:
                if ocfg["kind"] == "matcher":
                    r = run_matcher(cx, ocfg)
                elif ocfg["kind"] == "infer":
                    r = run_infer(cx, ocfg)
                else:
                    r, m3, _ = run_train(cx, oid, ocfg)
                    del m3
                r["workload"] = describe(oid, ocfg, per_gpu_batch(ocfg, world), world)
                r["scaling"] = ocfg["scaling"]
                others[str(oid)] = r
            except Exception as e:                                # a secondary block must not lose the headline
                others[str(oid)] = {"error": f"{type(e).__name__}: {e}"[:300]}
            torch.cuda.empty_cache()
        # the other precision class north_star names: the same training step in the fp32 (1e-5 parity, SIMT) mode
        if args.mode != "fp32" and time.time() - t_start < args.max_seconds * 0.7:
            saved_steps = args.steps
            try:
                lib.bdetr_set_mode(_lib.MODE_FP32)
                args.steps = min(args.steps, 10)
                r, m32, _ = run_train(cx, 2, CONFIGS[2])
                del m32
                others["2_fp32_mode"] = {"value": r["value"], "ms_per_step": r["ms_per_step"], "e2e": r["e2e"], "loss": r["loss"], "dtype": "fp32",
                                         "steps": args.steps, "workload": describe(2, CONFIGS[2], per_gpu_batch(CONFIGS[2], world), world)}
            except Exception as e:
                others["2_fp32_mode"] = {"error": f"{type(e).__name__}: {e}"[:300]}
            finally:
                args.steps = saved_steps
                lib.bdetr_set_mode({"tf32": _lib.MODE_TF32, "fp16": _lib.MODE_FP16, "fp32": _lib.MODE_FP32}[args.mode])
            torch.cuda.empty_cache()
    if rank != 0:
        return                                                   # (no collective below this line: the other ranks are gone)

    if others:
        line["other_configs"] = others
        if "4" in others and "matcher_us_per_image" in others["4"]:
            line["matcher_us_per_image"] = others["4"]["matcher_us_per_image"]
            line["matcher_parts_us"] = others["4"]["parts"]
    if cfg["kind"] == "train":
        lps = count_launches(model, batch)
        line["gpu_launches"] = lps * args.steps
        line["gpu_launches_per_step"] = lps
    else:
        line["gpu_launches"] = int(main_res.get("launches_per_step", 0)) * line["steps"]
        line["gpu_launches_per_step"] = main_res.get("launches_per_step")
    peaks = peaks_json()
    try:
        line["roofline"] = roofline_blocks(CONFIGS[2], CONFIGS[2]["B"], flush, peaks)
        if cfg["kind"] == "matcher":                             # this config's dominant kernel is the cost matrix
            rb = line["roofline"]["other_kernels"]["cost_matrix_config4_C82_A3"]
            line["roofline"] = dict(rb, kernel="cost_targets_kernel + cost_matrix_kernel", other_kernels=line["roofline"]["other_kernels"])
        elif cfg["kind"] == "infer":
            rb = line["roofline"]["other_kernels"].get("attention_core_fwd_L20020_config5")
            if rb:
                line["roofline"] = dict(rb, kernel="attention_fwd_umma_ms_kernel", other_kernels=line["roofline"]["other_kernels"])
    except Exception as e:
        line["roofline"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    if not args.no_cpu_baseline and world == 1:
        try:
            if cfg["kind"] == "train":
                sb = min(B, 16)
                sec = cpu_reference_train_steps(cfg, sb, cfg["C"], cfg["A"], 1, 1, cores)
                line["cpu_baseline"] = {"value": sb / sec, "unit": "images/s", "cores": cores, "kind": "port",
                                        "sample": f"1 full training step of {sb} images after 1 warm-up (oracle/reference_path.py, torch CPU fp32, {cores} threads)"}
            elif cfg["kind"] == "matcher":
                spi = cpu_reference_matcher(cfg, 32, 2, 1, cores)
                line["cpu_baseline"] = {"value": 1.0 / spi, "unit": "images/s", "cores": cores, "kind": "port", "us_per_image": spi * 1e6,
                                        "sample": f"2 passes over 32 of the {cfg['B']} images (oracle broadcast cost + scipy loop + matched loss, {cores} threads)"}
            else:
                spi = cpu_reference_infer(cfg, 1, 1, 0, cores)
                line["cpu_baseline"] = {"value": 1.0 / spi, "unit": "images/s", "cores": cores, "kind": "port",
                                        "sample": f"1 forward pass of 1 image at {cfg['rows'] * cfg['cols']} tokens (oracle, torch CPU fp32, {cores} threads)"}
            if cfg_id == 2 and "matcher_us_per_image" in line:
                spi = cpu_reference_matcher(CONFIGS[4], 32, 1, 1, cores)
                line["matcher_cpu_us_per_image"] = spi * 1e6
        except Exception as e:
            line["cpu_baseline"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    print(json.dumps(line))
    sys.stdout.flush()


if __name__ == "__main__":
    main()
