"""Inference parity at BASELINE config 5 (4 images of 110 x 182 features = 20 020 encoder tokens, 6 boosted blocks, Q = 100,
COCO vocabulary) in BDETR_MODE_TF32 and BDETR_MODE_FP16, against fp64.

Layer level: the fused entry points the inference forward runs (training = 0), driven through the wrappers the model uses,
with every GEMM operand rounded to tf32 on the host as in test_fused_tc_gpu.py.  Every buffer the wrappers allocate is
filled with NaN first, so a row or tile that no kernel writes fails.  The attention stage is checked on its own, from the
saved q / k / v projections: an fp64 softmax over ALL keys of the GPU's own (in fp16 mode: fp16-rounded) projections, on
sampled query rows of every image and head -- the first 130, the last 140 (the ragged last query tile and the last
multi-stream CTA, which has one live stream) and a stride.  The query projection is scaled by 4 in the peaky cases so that
each row's softmax is carried by a few keys (printed as the mean effective key count 1 / sum p^2) and the reference maximum
is raised after the first key tile; with Glorot weights the softmax over 20 020 keys is nearly flat and its error hides.

Model level: BoostedDETR.call(training=False) at config 5 and at its stride-32 variant (25 x 42 = 1 050 tokens) against
the oracle evaluated in fp64 by torch on the GPU (cuBLAS DGEMM and torch softmax; no project kernel), with determinism,
pinned-host-input and launch-count checks.  Bars and the measured errors are listed in DESIGN.md §2."""
import math

import numpy as np
import pytest
import torch

from test_dense_gpu import _model_and_data
from test_fused_tc_gpu import D, H, _dev, _host, _prepare, _randn, nerr, tf32

pytestmark = pytest.mark.gpu

L5, ROWS5, COLS5, B5, N5 = 20020, 110, 182, 4, 6
d = D // H
QSCALE = 4.0                     # power of two: the scaled tf32 query kernel stays exactly tf32

# normalised max error bars.  Each is a few times the largest error measured over this file's cases on a B200 (1000 W
# power limit), in brackets, and never looser than the layer bars of test_fused_tc_gpu.py for the same entry point.
BARS = {
    "proj": 1e-3,            # q / k / v projections vs fp64, stored tf32-rounded (half an ulp: 4.9e-4)  [4.3e-4]
    "o": 1e-3,               # attention output vs the fp64 softmax of the GPU's own projections         [4.6e-4]
    "lse": 1e-4,             # log-sum-exp, same reference                                               [3.2e-5]
    "out": 1.5e-3,           # block output (out-projection + residual + LayerNorm) from the GPU's o     [4.2e-4]
    "ffn": 1.5e-3,           # fused FFN block output, all 80 080 rows                                   [3.9e-4]
    "pos_projection": 5e-6,  #                                                                            [9.4e-7]
    "heads": 5e-6,           # running predictions of the fused heads, inference BatchNorm               [2.2e-6]
    # the three prediction tensors of the 6-block forward [1.06e-3: config 5, tf32 mode, category].  DESIGN §2's
    # tensor-core bar is 1e-3, but tf32 arithmetic alone fills it at this depth: the same forward evaluated by torch with
    # tf32 cuBLAS GEMMs (fp32 elsewhere) is 9.7e-4 from fp64 on the category predictions of this data, in fp32 1.9e-6.
    "model": 1.5e-3,
}


@pytest.fixture()
def lib():
    from boosted_detr_b200 import _lib
    lib = _lib.load()
    yield lib
    lib.bdetr_set_mode(_lib.MODE_FP32)


@pytest.fixture()
def nan_alloc(monkeypatch):
    """Every buffer the layer wrappers allocate starts as NaN."""
    from boosted_detr_b200 import prediction_heads, transformers

    def nan_empty(*shape, dtype=torch.float32):
        return torch.full(shape, float("nan"), dtype=dtype, device="cuda")
    empty_like = torch.empty_like
    monkeypatch.setattr(transformers, "empty", nan_empty)
    monkeypatch.setattr(prediction_heads, "empty", nan_empty)
    monkeypatch.setattr(torch, "empty_like", lambda t, **kw: empty_like(t, **kw).fill_(float("nan")))


def _set_mode(lib, name):
    from boosted_detr_b200 import _lib
    mode = {"tf32": _lib.MODE_TF32, "fp16": _lib.MODE_FP16}[name]
    lib.bdetr_set_mode(mode)
    assert lib.bdetr_get_mode() == mode


def _g64(a):
    return torch.as_tensor(np.asarray(a), dtype=torch.float64, device="cuda")


def _p64(w):
    return {k: _g64(v) for k, v in w.items()}


def _sample_rows(L):
    return np.unique(np.concatenate([np.arange(0, min(130, L)), np.arange(max(L - 140, 0), L), np.arange(0, L, 97)]))


def _is_tf32(t):
    """Finite and stored tf32-rounded (low 13 mantissa bits zero): the next GEMM reads it as a tf32 operand."""
    return bool(torch.isfinite(t).all()) and bool(((t.view(torch.int32) & 0x1FFF) == 0).all())


def _report(tag, errs, bars):
    for k, e in errs.items():
        print(f"config5-err {tag} {k} {e:.3e} (bar {bars[k]:.1e})")
    bad = {k: e for k, e in errs.items() if not e < bars[k]}
    assert not bad, f"{tag}: over the bar: {bad}"


def _scale_query(blk, w, s):
    """Multiply QueryProjection/kernel by s on the device and in the oracle's copy."""
    for n, o, k in blk.named_weights():
        if k.endswith("QueryProjection/kernel"):
            o._weights[k].mul_(s)
    key = "p/AttentionLayer/QueryProjection/kernel"
    w[key] = (w[key] * s).astype(np.float32)


def _attention_ref(qp, kp, vp, rows, f16):
    """fp64 softmax attention of one image over all keys: qp [Lq,D], kp / vp [Lk,D] (device fp32, the GPU's own
    projections); returns o [H,R,d], lse [H,R] (log2 units, as the kernels store it) and the effective key count [H,R]."""
    cast = (lambda t: t.half().double()) if f16 else (lambda t: t.double())
    R, Lk = len(rows), kp.shape[0]
    q = cast(qp[torch.as_tensor(rows, device="cuda")]).view(R, H, d).transpose(0, 1)
    k = cast(kp).view(Lk, H, d).transpose(0, 1)
    v = cast(vp).view(Lk, H, d).transpose(0, 1)
    s = (q @ k.transpose(1, 2)) / math.sqrt(d)
    mx = s.amax(-1, keepdim=True)
    p = torch.exp_(s.sub_(mx))
    l = p.sum(-1, keepdim=True)
    p.div_(l)
    o = p @ v
    neff = 1.0 / p.square_().sum(-1)
    return o, (torch.log(l[..., 0]) + mx[..., 0]) / math.log(2.0), neff


def _check_attention(tag, sv, w, x, mem, pos, rows, f16, resid_pos, key_pos):
    """Stage by stage: projections vs fp64, tf32 storage, the attention core vs an fp64 softmax of the GPU's own
    projections on `rows`, and the block output (out-projection + residual + LayerNorm) from the GPU's own o."""
    from oracle import reference_path as R
    B, Lq, Lk = x.shape[0], x.shape[1], mem.shape[1]
    p = _p64(w)
    gx, gm, gpos = _g64(x), _g64(mem), _g64(pos)
    qin = gx + gpos if resid_pos else gx
    kin = gm + gpos if key_pos else gm
    errs = {}
    for nm, src, proj in (("qp", qin, "QueryProjection"), ("kp", kin, "KeyProjection"), ("vp", gm, "ValueProjection")):
        assert _is_tf32(sv[nm]), f"{tag}: {nm} is not stored tf32-rounded (or not written)"
        errs[nm] = nerr(_host(sv[nm]), R.dense(src, p, f"p/AttentionLayer/{proj}").cpu().numpy())
    _report(tag + " proj", errs, {k: BARS["proj"] for k in errs})

    assert _is_tf32(sv["o"]), f"{tag}: o is not stored tf32-rounded (or not written)"
    assert bool(torch.isfinite(sv["lse"]).all()), f"{tag}: lse not written"
    o_ref, l_ref, neff = zip(*(_attention_ref(sv["qp"][b], sv["kp"][b], sv["vp"][b], rows, f16) for b in range(B)))
    ri = torch.as_tensor(rows, device="cuda")
    o_got = torch.stack([sv["o"][b][:, ri] for b in range(B)])
    l_got = torch.stack([sv["lse"][b][:, ri] for b in range(B)])
    print(f"{tag}: {len(rows)} rows x {H} heads x {B} images, mean effective keys {float(torch.stack(neff).mean()):.1f} of {Lk}")
    _report(tag + " attention", {"o": nerr(_host(o_got), _host(torch.stack(o_ref))),
                                 "lse": nerr(_host(l_got), _host(torch.stack(l_ref)))}, BARS)

    # sv.o [B,H,Lq,d] is re-read as [B,Lq,D] with no permute (reference transformers.py:100)
    a = R.dense(sv["o"].double().reshape(B, Lq, D), p, "p/AttentionLayer/OutputProjection")
    return R.layer_norm(qin + a, p, "p/LayerNorm")


def _attention_block(rng, qscale):
    from boosted_detr_b200.layers import Layer
    from boosted_detr_b200.transformers import AttentionBlock
    Layer._rng = np.random.default_rng(int(rng.integers(1 << 30)))
    blk = AttentionBlock(H, name="blk")
    x = _dev(np.zeros((1, 128, D)))
    blk.maybe_build([x, x, x])
    w = _prepare(blk, rng, "p/")
    if qscale != 1.0:
        _scale_query(blk, w, qscale)
    return blk, w


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["tf32", "fp16"])
@pytest.mark.parametrize("B,L,qscale", [(4, L5, QSCALE), (4, L5, 1.0), (4, 1050, QSCALE), (4, 1536, QSCALE), (5, 1536, QSCALE)])
def test_encoder_attention_inference(lib, nan_alloc, mode, B, L, qscale):
    """EncoderBlock's attention in inference (encoder fold: tab_q, tab_k, resid_pos).  B = 4 at L = 20 020 runs the
    multi-stream kernel (1 696 CTAs; in fp16 mode the cast + fp16 kernel through the fused entry point), L = 1 050 the
    one-tile kernel, and L = 1 536 sits on the multi-stream eligibility edge: 128 CTAs at B = 4 (one-tile), 160 at B = 5."""
    from boosted_detr_b200.transformers import make_fold, pos_projection
    _set_mode(lib, mode)
    rng = np.random.default_rng(B * 100000 + L + int(qscale))
    blk, w = _attention_block(rng, qscale)
    x, pos = _randn(rng, B, L, D), _randn(rng, L, D, scale=0.5)
    dx, dpos = _dev(x), _dev(pos)
    tabs = pos_projection(dpos, [(blk.AttentionLayer, "QueryProjection"), (blk.AttentionLayer, "KeyProjection")])
    fold = make_fold(pos=dpos, tab_q=tabs[0], tab_k=tabs[1], resid_pos=True, pos_tc=dpos)
    out, ctx = blk.forward_fused(dx, dx, fold, False)
    torch.cuda.synchronize()
    sv = ctx["saved"]
    assert sv["z"] is None
    n16 = int(lib.bdetr_attention_f16_workspace_bytes(B, H, L, L, d))
    assert ("ws16" in sv) == (mode == "fp16" and n16 > 0), (mode, n16)
    f16 = "ws16" in sv
    tag = f"enc {mode} B{B} L{L} x{qscale:g}" + (" fp16-kernel" if f16 else "")
    ref = _check_attention(tag, sv, w, x, x, pos, _sample_rows(L), f16, True, True)
    _report(tag + " block", {"out": nerr(_host(out), _host(ref))}, BARS)


@pytest.mark.parametrize("qscale", [QSCALE, 1.0])
def test_decoder_cross_attention_inference(lib, nan_alloc, qscale):
    """Decoder cross-attention (decoder fold: tab_k) of 4 x 100 queries against 4 x 20 020 keys: the one-tile kernel
    through 157 key tiles, the last with 52 keys.  Lq = 100 is not served by the fp16 kernel, so fp16 mode must give the
    tf32 bits."""
    from boosted_detr_b200.transformers import make_fold, pos_projection
    B, Q = B5, 100
    rng = np.random.default_rng(100 + int(qscale))
    blk, w = _attention_block(rng, qscale)
    dec, enc, pos = _randn(rng, B, Q, D), _randn(rng, B, L5, D), _randn(rng, L5, D, scale=0.5)
    ddec, denc, dpos = _dev(dec), _dev(enc), _dev(pos)
    got = {}
    for mode in ("tf32", "fp16"):
        _set_mode(lib, mode)
        tab_k = pos_projection(dpos, [(blk.AttentionLayer, "KeyProjection")])[0]
        fold = make_fold(pos=dpos, tab_k=tab_k, pos_tc=dpos)
        out, ctx = blk.forward_fused(ddec, denc, fold, False)
        torch.cuda.synchronize()
        got[mode] = (out, ctx["saved"])
    assert "ws16" not in got["fp16"][1]
    for nm in ("qp", "kp", "vp", "o", "lse", "mean", "rstd"):
        assert torch.equal(got["fp16"][1][nm], got["tf32"][1][nm]), f"fp16 mode changed {nm}"
    assert torch.equal(got["fp16"][0], got["tf32"][0]), "fp16 mode changed the block output"
    out, sv = got["tf32"]
    tag = f"dec B{B} Q{Q} Lk{L5} x{qscale:g}"
    ref = _check_attention(tag, sv, w, dec, enc, pos, np.arange(Q), False, False, True)
    _report(tag + " block", {"out": nerr(_host(out), _host(ref))}, BARS)


# ---------------------------------------------------------------------------------------------------------------------
def test_ffn_inference_config5(lib, nan_alloc):
    """FeedForwardBlock on the fused path at M = 4 x 20 020 = 80 080 rows (625 row tiles of 128 and a ragged one of 80),
    inference: every row against fp64."""
    from oracle import reference_path as R
    from boosted_detr_b200.layers import Layer
    from boosted_detr_b200.transformers import FeedForwardBlock
    _set_mode(lib, "tf32")
    M = B5 * L5
    rng = np.random.default_rng(80080)
    Layer._rng = np.random.default_rng(9)
    x = _randn(rng, M, D)
    dx = _dev(x)
    blk = FeedForwardBlock(name="ffn")
    blk.maybe_build([dx])
    w = _prepare(blk, rng, "p/")
    out, ctx = blk.forward([dx], training=False)
    torch.cuda.synchronize()
    assert ctx["fused"] and ctx["saved"]["z"] is None
    assert _is_tf32(ctx["saved"]["h"]), "hidden activations not stored tf32-rounded (or not written)"
    ref = R.feed_forward_block(_g64(x), _p64(w), "p", R.Dropout(None), 0, False)
    _report(f"ffn M{M}", {"ffn": nerr(_host(out), _host(ref))}, BARS)


def test_pos_projection_config5(lib):
    """tab[g] = pos W[g] + b[g] at L = 20 020 for the encoder's two projections and the model's three (encoder q, k and
    decoder k)."""
    from boosted_detr_b200.transformers import pos_projection
    _set_mode(lib, "tf32")
    rng = np.random.default_rng(20020)
    blks = [_attention_block(rng, 1.0) for _ in range(2)]
    pairs = [(blks[0], "QueryProjection"), (blks[0], "KeyProjection"), (blks[1], "KeyProjection")]
    pos = _randn(rng, L5, D)
    gpos = _g64(pos)
    errs = {}
    for n in (2, 3):
        tabs = pos_projection(_dev(pos), [(b.AttentionLayer, nm) for (b, _), nm in pairs[:n]])
        torch.cuda.synchronize()
        for g, ((_, w), nm) in enumerate(pairs[:n]):
            W, bias = (_g64(w[f"p/AttentionLayer/{nm}/{s}"]) for s in ("kernel", "bias"))
            errs[f"n{n} tab{g}"] = nerr(_host(tabs[g]), _host(gpos @ W + bias))
    _report("pos_projection", errs, {k: BARS["pos_projection"] for k in errs})


@pytest.mark.parametrize("variant", ["block0", "later"])
@pytest.mark.parametrize("C,A", [(82, 3), (48, 296)])
def test_heads_inference(lib, nan_alloc, C, A, variant):
    """The fused heads of one block in inference at M = 4 x 100: block 0's form (mult 2, no running sum in) and a later
    block's (mult 1 onto running predictions).  BatchNorm runs on the moving statistics, which stay bit-unchanged."""
    from oracle import reference_path as R
    from boosted_detr_b200.layers import Layer
    from boosted_detr_b200.prediction_heads import (BoxPredictionHead, MultiClassPredictionHead, SingleClassPredictionHead,
                                                    heads_forward_fused)
    _set_mode(lib, "tf32")
    B, Q = B5, 100
    rng = np.random.default_rng(C * 7 + A + len(variant))
    Layer._rng = np.random.default_rng(11)
    x = _randn(rng, B, Q, D)
    dx = _dev(x)
    heads = (SingleClassPredictionHead(C, D, Q, name="cat"), MultiClassPredictionHead(A, D, Q, name="attr"),
             BoxPredictionHead(D, Q, name="box"))
    w = {}
    for hd in heads:
        hd.maybe_build([dx])
        w.update(_prepare(hd, rng, hd.name + "/"))
    mult = 2.0 if variant == "block0" else 1.0
    cum_np = None if variant == "block0" else [tf32(rng.uniform(0, 1, (B, Q, n))) for n in (C, A, 4)]
    stats0 = {(hd.name, k): _host(hd._weights[k]).copy() for hd in heads for k in ("BatchNorm/moving_mean", "BatchNorm/moving_variance")}
    cum, _ = heads_forward_fused(heads, dx, False, None if cum_np is None else [_dev(c) for c in cum_np], mult)
    torch.cuda.synchronize()
    for hd in heads:
        for k in ("BatchNorm/moving_mean", "BatchNorm/moving_variance"):
            assert np.array_equal(_host(hd._weights[k]), stats0[(hd.name, k)]), f"{hd.name} {k} changed in inference"
    p, tx = _p64(w), _g64(x)
    errs = {}
    for i, (hd, fn, c) in enumerate(zip(heads, (R.category_head, R.attribute_head, R.box_head), cum)):
        ref = (0.0 if cum_np is None else _g64(cum_np[i])) + mult * fn(tx, p, hd.name, False)
        errs[hd.name] = nerr(_host(c), _host(ref))
    _report(f"heads C{C} A{A} {variant}", errs, {k: BARS["heads"] for k in errs})


# ---------------------------------------------------------------------------------------------------------------------
def _model_run(rows, cols):
    """BoostedDETR.call(training=False) in both tensor-core modes (twice on device features, once on pinned host features)
    and the oracle's predictions in fp64 on the GPU."""
    from oracle import reference_path as R
    from boosted_detr_b200 import _lib
    lib = _lib.load()
    model, w, inputs = _model_and_data(N=N5, B=B5, rows=rows, cols=cols)
    feats = inputs["features"]
    dev, pinned = torch.from_numpy(feats).cuda(), torch.from_numpy(feats).pin_memory()
    run = {}
    try:
        for mode in ("tf32", "fp16"):
            _set_mode(lib, mode)
            model.call({"features": dev}, training=False)
            torch.cuda.synchronize()
            lib.bdetr_reset_launch_count()
            first = [t.clone() for t in model.call({"features": dev}, training=False)]
            torch.cuda.synchronize()
            launches = int(lib.bdetr_launch_count())
            exit_block = model.last_exit_block
            again = [t.clone() for t in model.call({"features": dev}, training=False)]
            host = [t.clone() for t in model.call({"features": pinned}, training=False)]
            torch.cuda.synchronize()
            run[mode] = {"preds": first, "again": again, "pinned": host, "launches": launches, "exit": exit_block}
    finally:
        lib.bdetr_set_mode(_lib.MODE_FP32)
    saved = R.ATTENTION_QUERY_CHUNK
    R.ATTENTION_QUERY_CHUNK = 256
    try:
        with torch.no_grad():
            out = R.boosted_detr_call(_p64(w), _g64(feats), None, N5, H, training=False)
        run["oracle"] = [t.cpu() for t in out["preds"]]
    finally:
        R.ATTENTION_QUERY_CHUNK = saved
    del model
    torch.cuda.empty_cache()
    return run


@pytest.fixture(scope="module")
def model_runs():
    cache = {}

    def get(cfg):
        if cfg not in cache:
            cache[cfg] = _model_run(*{"config5": (ROWS5, COLS5), "stride32": (25, 42)}[cfg])
        return cache[cfg]
    return get


@pytest.mark.parametrize("mode", ["tf32", "fp16"])
@pytest.mark.parametrize("cfg", ["config5", "stride32"])
def test_model_inference_vs_fp64(model_runs, cfg, mode):
    """The three prediction tensors against fp64 (bar explained at BARS), and no early exit at the default threshold
    (None)."""
    run = model_runs(cfg)
    r = run[mode]
    assert r["exit"] == N5 - 1, r["exit"]
    errs = {nm: nerr(_host(g), run["oracle"][i].numpy()) for i, (nm, g) in enumerate(zip(("cat", "attr", "box"), r["preds"]))}
    _report(f"model {cfg} {mode}", errs, {k: BARS["model"] for k in errs})


@pytest.mark.parametrize("mode", ["tf32", "fp16"])
@pytest.mark.parametrize("cfg", ["config5", "stride32"])
def test_model_inference_deterministic(model_runs, cfg, mode):
    """Two consecutive calls give identical bits (the inference forward has no float atomics), and a call on pinned host
    features (bench.py's e2e arm) gives the bits of a call on device features."""
    r = model_runs(cfg)[mode]
    for i in range(3):
        assert torch.equal(r["again"][i], r["preds"][i]), f"prediction {i}: two consecutive calls differ"
        assert torch.equal(r["pinned"][i], r["preds"][i]), f"prediction {i}: pinned host features give other bits"


@pytest.mark.parametrize("cfg", ["config5", "stride32"])
def test_model_inference_fp16_dispatch(lib, model_runs, cfg):
    """At 20 020 tokens fp16 mode adds one cast launch per encoder block (the fp16 kernel ran at B = 4); at 1 050 tokens
    the fp16 kernel does not serve the shape and fp16 mode must give the tf32 launches and bits."""
    run = model_runs(cfg)
    L = ROWS5 * COLS5 if cfg == "config5" else 25 * 42
    served = lib.bdetr_attention_f16_workspace_bytes(B5, H, L, L, d) > 0
    assert served == (cfg == "config5")
    if served:
        assert run["fp16"]["launches"] == run["tf32"]["launches"] + N5, (run["fp16"]["launches"], run["tf32"]["launches"])
    else:
        assert run["fp16"]["launches"] == run["tf32"]["launches"]
        for i in range(3):
            assert torch.equal(run["fp16"]["preds"][i], run["tf32"]["preds"][i]), f"prediction {i}: fp16 mode changed the bits"
