"""The attention backward core (bdetr_attention_core_bwd) on its own: the tcgen05 dQ and dK/dV kernels (tf32 mode) and the
SIMT kernels (fp32 mode) against the true fp64 gradient of softmax(Q K^T / sqrt(d)) V, at the model's shapes, at every
tile edge (64-key / 64-query tiles, 128-row CTAs), at long sequences and with peaky scores.

The block-level tests see these gradients only after the projection and LayerNorm backward, at bars of 5e-3 to 1e-2.
Here each of dQ, dK, dV and delta has its own bar, and each bar is checked to sit below the error that dropping a single
row's term causes: the last query's term from dK / dV, the last key's term from dQ.  Every output is written into a
NaN-filled buffer followed by canary rows: all outputs must be finite (every row written) and the canaries untouched
(nothing written past the end).  Each case runs twice and must give the same bits (the kernels use no atomics)."""
import numpy as np
import pytest
import torch

from test_dense_gpu import nerr
from test_tc_gpu import tf32

pytestmark = pytest.mark.gpu

# Worst errors over these cases on a B200 (1000 W power limit): fp32 mode dq 3.6e-6, dk 6.8e-6, dv 4.5e-6; tf32 mode (P and
# dS truncated to tf32 before the MMAs that consume them, fp32 sums) dq 7.4e-4, dk 6.8e-4, dv 6.4e-4; delta, the same
# fp32 arithmetic in both modes, 3.6e-7.  The smallest one-row-dropped error is 3.0e-2.
BARS = {"fp32": {"dq": 1e-5, "dk": 1e-5, "dv": 1e-5, "delta": 1e-6},
        "tf32": {"dq": 1.5e-3, "dk": 1.5e-3, "dv": 1.5e-3, "delta": 1e-6}}

HEADS = [(8, 32), (4, 64), (8, 64)]                       # (H, d): model width 256 at d = 32 and 64, and 512 at d = 64
SHAPES = [                                                # (B, Lq, Lk, query scale)
    (16, 400, 400, 1.0), (16, 100, 400, 1.0), (1, 100, 100, 1.0),        # encoder, decoder cross, hoisted decoder self
    (2, 1, 1, 1.0), (3, 130, 257, 1.0),
    (2, 1, 129, 1.0), (2, 63, 65, 1.0), (2, 64, 64, 1.0), (2, 65, 63, 1.0),
    (2, 127, 128, 1.0), (2, 128, 127, 1.0), (2, 129, 1, 1.0), (2, 1, 64, 1.0),
    (1, 2100, 2100, 1.0), (2, 700, 2100, 1.0),
    (2, 700, 2100, 12.0),                                 # peaky: scores with a standard deviation of 12
]
CANARY_ROWS = 128                                         # one CTA's worth of rows past the end of every output
SENTINEL = 0x7FA5A5A5                                     # a NaN payload no kernel writes


@pytest.fixture()
def mode():
    from boosted_detr_b200 import _lib
    lib = _lib.load()

    def set_mode(m):
        lib.bdetr_set_mode({"fp32": _lib.MODE_FP32, "tf32": _lib.MODE_TF32}[m])
    yield set_mode
    lib.bdetr_set_mode(_lib.MODE_FP32)


def _inputs(B, H, Lq, Lk, d, qs):
    rng = np.random.default_rng(B * 100003 + H * 1009 + Lq * 31 + Lk * 7 + d)
    D = H * d
    q = tf32(rng.standard_normal((B, Lq, D)) * qs)
    k, v = tf32(rng.standard_normal((B, Lk, D))), tf32(rng.standard_normal((B, Lk, D)))
    do = tf32(rng.standard_normal((B, H, Lq, d)))
    return q, k, v, do


_ref_cache = {}


def _reference(B, H, Lq, Lk, d, qs):
    """fp64 dQ / dK / dV in the [B, L, H*d] layout, the floor of each one's normalisation, and per gradient the largest
    single term a kernel drops when it skips the last key (dQ) or the last query (dK, dV) of a (b, h) pair, normalised
    like the error."""
    key = (B, H, Lq, Lk, d, qs)
    if key in _ref_cache:
        return _ref_cache[key]
    _ref_cache.clear()
    q, k, v, do = _inputs(B, H, Lq, Lk, d, qs)
    sc = 1.0 / np.sqrt(d)
    dq, dk, dv = np.empty((B, Lq, H * d)), np.empty((B, Lk, H * d)), np.empty((B, Lk, H * d))
    drop = {"dq": 0.0, "dk": 0.0, "dv": 0.0}
    cancel = {"dq": 0.0, "dk": 0.0}
    for b in range(B):
        for h in range(H):
            cols = slice(h * d, (h + 1) * d)
            Q, K, V = (x[b, :, cols].astype(np.float64) for x in (q, k, v))
            dO = do[b, h].astype(np.float64)
            s = Q @ K.T * sc
            p = np.exp(s - s.max(-1, keepdims=True))
            p /= p.sum(-1, keepdims=True)
            dp = dO @ V.T
            ds = p * (dp - (dO * (p @ V)).sum(-1, keepdims=True))
            dq[b, :, cols] = ds @ K * sc
            dk[b, :, cols] = ds.T @ Q * sc
            dv[b, :, cols] = p.T @ dO
            drop["dq"] = max(drop["dq"], np.abs(np.outer(ds[:, -1], K[-1])).max() * sc)
            drop["dk"] = max(drop["dk"], np.abs(np.outer(ds[-1], Q[-1])).max() * sc)
            drop["dv"] = max(drop["dv"], np.abs(np.outer(p[-1], dO[-1])).max())
            cancel["dq"] = max(cancel["dq"], np.abs(p * dp).max() * np.abs(K).max() * sc)
            cancel["dk"] = max(cancel["dk"], np.abs(p * dp).max() * np.abs(Q).max() * sc)
    ref = {"dq": dq, "dk": dk, "dv": dv}
    # at Lk = 1 the softmax is constant: dQ and dK are zero and are measured against the size of the terms that cancel
    floor = {g: cancel[g] if Lk == 1 and g in cancel else 1e-30 for g in ref}
    sens = {g: drop[g] / max(np.abs(ref[g]).max(), floor[g]) for g in ref}
    _ref_cache[key] = (ref, floor, sens)
    return _ref_cache[key]


def _guarded(n_rows, row_len):
    """A [n_rows * row_len] float view at the start of a sentinel-filled buffer with CANARY_ROWS more rows behind it."""
    buf = torch.full(((n_rows + CANARY_ROWS) * row_len,), SENTINEL, dtype=torch.int32, device="cuda")
    return buf, buf.view(torch.float32)[:n_rows * row_len]


def _backward(B, H, Lq, Lk, d, q, k, v, do):
    """o and lse from the GPU's own forward, then the backward core twice into fresh guarded buffers."""
    from boosted_detr_b200 import _lib
    from boosted_detr_b200.device import ptr, stream_ptr
    D = H * d
    tq, tk, tv, tdo = (torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (q, k, v, do))
    o = torch.full((B, H, Lq, d), float("nan"), device="cuda")
    lse = torch.full((B, H, Lq), float("nan"), device="cuda")
    _lib.call("bdetr_attention_core_fwd", B, H, Lq, Lk, d, ptr(tq), ptr(tk), ptr(tv), ptr(o), ptr(lse), stream_ptr())
    runs = []
    for _ in range(2):
        bufs = {"delta": _guarded(B * H * Lq, 1), "dq": _guarded(B * Lq, D), "dk": _guarded(B * Lk, D), "dv": _guarded(B * Lk, D)}
        _lib.call("bdetr_attention_core_bwd", B, H, Lq, Lk, d, ptr(tq), ptr(tk), ptr(tv), ptr(o), ptr(lse), ptr(tdo),
                  *(ptr(bufs[g][1]) for g in ("delta", "dq", "dk", "dv")), stream_ptr())
        torch.cuda.synchronize()
        runs.append({g: b.cpu().numpy() for g, (b, _) in bufs.items()})
    for g, raw in runs[0].items():
        n = raw.size - CANARY_ROWS * (1 if g == "delta" else D)
        assert (raw[n:] == SENTINEL).all(), f"{g}: written past its last row"
        assert np.isfinite(raw[:n].view(np.float32)).all(), f"{g}: rows not written"
        assert np.array_equal(raw, runs[1][g]), f"{g}: two runs differ"
    out = {g: raw[:raw.size - CANARY_ROWS * (1 if g == "delta" else D)].view(np.float32) for g, raw in runs[0].items()}
    return (out["delta"].reshape(B, H, Lq), out["dq"].reshape(B, Lq, D), out["dk"].reshape(B, Lk, D),
            out["dv"].reshape(B, Lk, D), o.cpu().numpy())


@pytest.mark.parametrize("m", ["fp32", "tf32"])
@pytest.mark.parametrize("B,Lq,Lk,qs", SHAPES)
@pytest.mark.parametrize("H,d", HEADS)
def test_attention_core_bwd_vs_fp64(mode, m, H, d, B, Lq, Lk, qs):
    """dQ, dK, dV within the mode's bar of the fp64 gradient (at Lk = 1 the softmax is constant, so dQ and dK are exactly
    zero and are measured against the size of the terms that cancel); delta within 1e-6 of the fp64 row sum of
    dO * o over the GPU's own o.  On every case with N(0, 1) scores, each bar must also sit below the error of dropping one
    row's term, so that a kernel that skips the last row of a tile cannot pass."""
    mode(m)
    q, k, v, do = _inputs(B, H, Lq, Lk, d, qs)
    delta, dq, dk, dv, o = _backward(B, H, Lq, Lk, d, q, k, v, do)
    ref, floor, sens = _reference(B, H, Lq, Lk, d, qs)
    err = {g: nerr(got, ref[g], floor[g]) for g, got in (("dq", dq), ("dk", dk), ("dv", dv))}
    err["delta"] = nerr(delta, (do.astype(np.float64) * o.astype(np.float64)).sum(-1))
    print(f"{m} attention bwd B{B} H{H} d{d} Lq{Lq} Lk{Lk} qs{qs:g}: "
          + " ".join(f"{g} {e:.2e}" for g, e in err.items()) + " | one row dropped: "
          + " ".join(f"{g} {s:.2e}" for g, s in sens.items()))
    bars = BARS[m]
    for g, e in err.items():
        assert e < bars[g], g
    if qs == 1.0:
        for g, s in sens.items():
            if Lk == 1 and g != "dv":                      # zero gradient: no row to miss
                continue
            assert bars[g] < s, f"{g}: the bar {bars[g]:.1e} does not catch a dropped row ({s:.1e})"
