"""Layer-level parity of the fused tensor-core entry points the model runs in BDETR_MODE_TF32 (ops_fused.cu,
heads_fused.cu) against the fp64 oracle: bdetr_pos_projection, bdetr_attention_fused_* (encoder fold, decoder fold, no
fold), bdetr_ffn_fused_*, bdetr_decoder_self_* and bdetr_heads_*, driven through the wrappers the model uses.

Every GEMM operand (inputs, positional table, Dense kernels) is rounded to nearest tf32 on the host and written into the
layer, and the oracle is fed exactly those values.  What remains is the kernels' own rounding of the intermediates they
produce (q / k / v projections, attention output, hidden activations, data gradients) and fp32 accumulation, so the bars
below are tight enough to see one wrong row tile or column quarter -- which the whole-model tests, held to 5e-2 by the
ill-conditioned .999 clip, cannot.

Accumulation contracts: every parameter-gradient buffer, d_pos, d_q0 and the accumulated data gradients are pre-filled
with random values G0 of the size of the expected increment, and got - G0 is compared; a frozen layer must leave them
bit-identical.  Errors are normalised max errors (nerr) per tensor; the measured maxima are listed in DESIGN.md §2."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from test_dense_gpu import nerr
from test_tc_gpu import tf32

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
D, H = 256, 8
SEED, SITE = 2024, 13
ARM_ENV = "BDETR_TEST_AB_ARM"        # set in the child interpreter of test_ab_arm_keeps_layer_parity

# normalised max error bars per entry point: outputs, data gradients, parameter gradients, positional gradient, BatchNorm
# batch statistics (the moving-statistic increments).  Each is a few times the largest error measured over this file's
# cases on a B200 (1000 W power limit), in brackets, and never looser than the layer-twin tf32 bars (2e-3 / 5e-3 / 1e-2).
BARS = {
    "pos_projection": {"out": 5e-6},                                                      # [8.9e-7]
    "attention": {"out": 1.5e-3, "data": 2.5e-3, "param": 3e-3, "pos": 3e-3},             # [4.3e-4, 7.0e-4, 7.7e-4, 9.0e-4]
    "ffn": {"out": 1.5e-3, "data": 1e-3, "param": 1.5e-3},                                # [4.3e-4, 1.9e-4, 4.1e-4]
    "decoder_self": {"out": 1.5e-3, "data": 3e-4, "param": 3e-3},                         # [4.6e-4, 6.9e-5, 8.3e-4]
    "heads": {"out": 5e-6, "data": 1e-3, "param": 4e-3, "stats": 5e-5},                   # [1.0e-6, 2.4e-4, 1.1e-3, 1.0e-5]
}


@pytest.fixture()
def tc_mode():
    from boosted_detr_b200 import _lib
    lib = _lib.load()
    lib.bdetr_set_mode(_lib.MODE_TF32)
    yield
    lib.bdetr_set_mode(_lib.MODE_FP32)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def _host(t):
    return t.detach().cpu().numpy()


def _t64(a, grad=False):
    return torch.tensor(np.asarray(a), dtype=torch.float64, requires_grad=grad)


def _randn(rng, *shape, scale=1.0):
    return tf32(rng.standard_normal(shape) * scale)


def _seed_word(on):
    return torch.tensor([SEED], dtype=torch.int32, device="cuda") if on else None


def _fill(t, rng, ref):
    """Pre-fill the device buffer `t` with random values of the size of `ref` (the expected increment); returns them."""
    scale = max(float(np.abs(np.asarray(ref)).max()), 1e-6)
    a = (rng.standard_normal(tuple(t.shape)) * scale).astype(np.float32)
    t.copy_(torch.from_numpy(a))
    return a


def _name(prefix, n):
    return prefix + n.split("/", 1)[1]


def _prepare(layer, rng, prefix):
    """Randomise the biases, LayerNorm / BatchNorm parameters and moving statistics of a built layer, round every value
    to tf32 and write it back in place; returns {prefix + name below the layer: array} for the oracle."""
    w = {}
    for n, o, k in layer.named_weights():
        a = _host(o._weights[k]).astype(np.float64)
        if k.endswith(("/bias", "/beta")):
            a = rng.normal(0, 0.1, a.shape)
        elif k.endswith("/gamma"):
            a = 1.0 + rng.normal(0, 0.1, a.shape)
        elif k.endswith("moving_mean"):
            a = rng.normal(0, 0.2, a.shape)
        elif k.endswith("moving_variance"):
            a = rng.uniform(0.5, 1.5, a.shape)
        a = tf32(a)
        o._weights[k].copy_(torch.from_numpy(a))
        w[_name(prefix, n)] = a
    return w


def _floor(name, p):
    # the key-bias gradient is mathematically zero (softmax is shift invariant): judge it on the query-bias scale
    if name.endswith("KeyProjection/bias"):
        return float(p[name.replace("KeyProjection", "QueryProjection")].grad.abs().max())
    return 1e-30


def _prefill_grads(layer, p, prefix, rng):
    g0 = {}
    for n, o, k in layer.named_weights():
        if k in o._grads:
            name = _name(prefix, n)
            g0[name] = _fill(o._grads[k], rng, max(float(p[name].grad.abs().max()), _floor(name, p)))
    return g0


def _report(tag, errs, bar):
    for k, e in errs.items():
        print(f"fused-err {tag} {k} {e:.3e} (bar {bar:.0e})")
    bad = {k: e for k, e in errs.items() if not e < bar}
    assert not bad, f"{tag}: over the {bar:.0e} bar: {bad}"


def _check_params(tag, layer, prefix, p, g0, frozen, bar):
    errs = {}
    for n, o, k in layer.named_weights():
        if k not in o._grads:
            continue
        name = _name(prefix, n)
        got = _host(o._grads[k])
        if frozen:
            assert np.array_equal(got, g0[name]), f"{tag}: the frozen layer's {name} gradient buffer was written"
        else:
            errs[name] = nerr(got.astype(np.float64) - g0[name], p[name].grad.numpy(), _floor(name, p))
    _report(tag + " param", errs, bar)


# ---------------------------------------------------------------------------------------------------------------------
def test_pos_projection(tc_mode):
    """tab[g] = pos_tc W[g] + b[g] (one grouped GEMM) for one and three projections, ragged and multi-tile row counts."""
    from boosted_detr_b200.layers import Layer
    from boosted_detr_b200.transformers import AttentionBlock, pos_projection
    rng = np.random.default_rng(7)
    Layer._rng = np.random.default_rng(7)
    blk = AttentionBlock(H, name="blk")
    x = _dev(np.zeros((1, 128, D)))
    blk.maybe_build([x, x, x])
    w = _prepare(blk, rng, "p/")
    names = ["QueryProjection", "KeyProjection", "ValueProjection"]
    errs = {}
    for L in (100, 400, 1050):
        pos = _randn(rng, L, D)
        for n in (1, 3):
            tabs = pos_projection(_dev(pos), [(blk.AttentionLayer, nm) for nm in names[:n]])
            torch.cuda.synchronize()
            for nm, t in zip(names, tabs):
                W, b = (w[f"p/AttentionLayer/{nm}/{s}"].astype(np.float64) for s in ("kernel", "bias"))
                errs[f"L{L} n{n} {nm}"] = nerr(_host(t), pos.astype(np.float64) @ W + b)
    _report("pos_projection out", errs, BARS["pos_projection"]["out"])


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["plain", "seed_acc", "no_dq", "frozen"])
@pytest.mark.parametrize("B,L", [(16, 400), (3, 130)])
def test_attention_encoder_fold(tc_mode, B, L, variant):
    """EncoderBlock's attention: q = k = x + pos, v = x, residual x + pos, folded as tab_q / tab_k / resid_pos / pos_tc.
    plain: dropout off; seed_acc: dropout keyed by the device seed word and d_query accumulated (acc_flags bit 0);
    no_dq: d_query NULL (parameter and positional gradients only); frozen: gw and d_pos NULL."""
    from oracle import reference_path as R
    from boosted_detr_b200.layers import Layer, dropout_site_key
    from boosted_detr_b200.transformers import AttentionBlock, make_fold, pos_projection
    rng = np.random.default_rng(B * 1000 + L)
    Layer._rng = np.random.default_rng(5)
    x, pos, go = _randn(rng, B, L, D), _randn(rng, L, D, scale=0.5), rng.standard_normal((B, L, D))
    dx, dpos = _dev(x), _dev(pos)
    blk = AttentionBlock(H, name="blk")
    blk.maybe_build([dx, dx, dx])
    w = _prepare(blk, rng, "p/")
    dropout, acc, need_dq, frozen = variant in ("seed_acc", "no_dq"), variant == "seed_acc", variant != "no_dq", variant == "frozen"
    blk.rate = 0.1 if dropout else 0.0
    tabs = pos_projection(dpos, [(blk.AttentionLayer, "QueryProjection"), (blk.AttentionLayer, "KeyProjection")])
    fold = make_fold(pos=dpos, tab_q=tabs[0], tab_k=tabs[1], resid_pos=True, pos_tc=dpos)
    out, ctx = blk.forward_fused(dx, dx, fold, True, dropout_site_key(SITE) if dropout else 0, _seed_word(dropout))

    p = R.params_to_torch(w, torch.float64, requires_grad=True)
    tx, tpos = _t64(x, True), _t64(pos, True)
    qk = tx + tpos
    ref = R.attention_block(qk, qk, tx, p, "p", H, R.Dropout(SEED if dropout else None), SITE, True)
    (ref * _t64(go)).sum().backward()

    blk.trainable = not frozen
    g0 = _prefill_grads(blk, p, "p/", rng)
    d_pos = torch.empty(L, D, device="cuda")
    pos0 = _fill(d_pos, rng, tpos.grad)
    d_query = torch.empty(B, L, D, device="cuda") if acc else None
    dq0 = _fill(d_query, rng, tx.grad) if acc else 0.0
    d_q, _ = blk.backward_fused(ctx, _dev(go), d_query=d_query, acc=(acc, False), d_pos=d_pos, need_dq=need_dq)
    torch.cuda.synchronize()

    tag = f"attention enc B{B} L{L} {variant}"
    bars = BARS["attention"]
    _report(tag + " out", {"out": nerr(_host(out), ref.detach().numpy())}, bars["out"])
    if need_dq:
        _report(tag + " data", {"d_query": nerr(_host(d_q) - dq0, tx.grad.numpy())}, bars["data"])
    else:
        assert d_q is None
    if frozen:
        assert np.array_equal(_host(d_pos), pos0), "frozen block: d_pos was written"
    else:
        _report(tag + " pos", {"d_pos": nerr(_host(d_pos) - pos0, tpos.grad.numpy())}, bars["pos"])
    _check_params(tag, blk, "p/", p, g0, frozen, bars["param"])


@pytest.mark.parametrize("variant", ["acc", "no_dm"])
@pytest.mark.parametrize("B", [16, 2])
def test_attention_decoder_fold(tc_mode, B, variant):
    """Decoder cross-attention: key = enc + pos (tab_k, pos_tc), value = enc, no positional residual.  acc: dropout by
    the seed word, d_query and d_memory accumulated (acc_flags bits 0 and 1); no_dm: d_memory NULL."""
    from oracle import reference_path as R
    from boosted_detr_b200.layers import Layer, dropout_site_key
    from boosted_detr_b200.transformers import AttentionBlock, make_fold, pos_projection
    Q, Lk = 100, 400
    rng = np.random.default_rng(B * 10 + len(variant))
    Layer._rng = np.random.default_rng(6)
    dec, enc, pos = _randn(rng, B, Q, D), _randn(rng, B, Lk, D), _randn(rng, Lk, D, scale=0.5)
    go = rng.standard_normal((B, Q, D))
    ddec, denc, dpos = _dev(dec), _dev(enc), _dev(pos)
    blk = AttentionBlock(H, name="blk")
    blk.maybe_build([ddec, denc, denc])
    w = _prepare(blk, rng, "p/")
    acc = dropout = variant == "acc"
    blk.rate = 0.1 if dropout else 0.0
    tab_k = pos_projection(dpos, [(blk.AttentionLayer, "KeyProjection")])[0]
    fold = make_fold(pos=dpos, tab_k=tab_k, pos_tc=dpos)
    out, ctx = blk.forward_fused(ddec, denc, fold, True, dropout_site_key(SITE) if dropout else 0, _seed_word(dropout))

    p = R.params_to_torch(w, torch.float64, requires_grad=True)
    tdec, tenc, tpos = _t64(dec, True), _t64(enc, True), _t64(pos, True)
    ref = R.attention_block(tdec, tenc + tpos, tenc, p, "p", H, R.Dropout(SEED if dropout else None), SITE, True)
    (ref * _t64(go)).sum().backward()

    g0 = _prefill_grads(blk, p, "p/", rng)
    d_pos = torch.empty(Lk, D, device="cuda")
    pos0 = _fill(d_pos, rng, tpos.grad)
    d_query = d_memory = None
    dq0 = dm0 = 0.0
    if acc:
        d_query, d_memory = torch.empty(B, Q, D, device="cuda"), torch.empty(B, Lk, D, device="cuda")
        dq0, dm0 = _fill(d_query, rng, tdec.grad), _fill(d_memory, rng, tenc.grad)
    d_q, d_m = blk.backward_fused(ctx, _dev(go), d_query=d_query, d_memory=d_memory, acc=(acc, acc), d_pos=d_pos,
                                  need_dm=acc)
    torch.cuda.synchronize()

    tag = f"attention dec B{B} {variant}"
    bars = BARS["attention"]
    _report(tag + " out", {"out": nerr(_host(out), ref.detach().numpy())}, bars["out"])
    errs = {"d_query": nerr(_host(d_q) - dq0, tdec.grad.numpy())}
    if acc:
        errs["d_memory"] = nerr(_host(d_m) - dm0, tenc.grad.numpy())
    else:
        assert d_m is None
    _report(tag + " data", errs, bars["data"])
    _report(tag + " pos", {"d_pos": nerr(_host(d_pos) - pos0, tpos.grad.numpy())}, bars["pos"])
    _check_params(tag, blk, "p/", p, g0, False, bars["param"])


def test_attention_no_fold_cross(tc_mode):
    """fold = NULL: plain cross-attention with a ragged query and key length, dropout by the seed word."""
    from oracle import reference_path as R
    from boosted_detr_b200.layers import Layer, dropout_site_key
    from boosted_detr_b200.transformers import AttentionBlock
    B, Lq, Lk = 3, 130, 257
    rng = np.random.default_rng(8)
    Layer._rng = np.random.default_rng(8)
    q, m, go = _randn(rng, B, Lq, D), _randn(rng, B, Lk, D), rng.standard_normal((B, Lq, D))
    dq, dm = _dev(q), _dev(m)
    blk = AttentionBlock(H, name="blk")
    blk.maybe_build([dq, dm, dm])
    w = _prepare(blk, rng, "p/")
    out, ctx = blk.forward_fused(dq, dm, None, True, dropout_site_key(SITE), _seed_word(True))
    p = R.params_to_torch(w, torch.float64, requires_grad=True)
    tq, tm = _t64(q, True), _t64(m, True)
    ref = R.attention_block(tq, tm, tm, p, "p", H, R.Dropout(SEED), SITE, True)
    (ref * _t64(go)).sum().backward()
    g0 = _prefill_grads(blk, p, "p/", rng)
    d_q, d_m = blk.backward_fused(ctx, _dev(go))
    torch.cuda.synchronize()
    tag = f"attention cross B{B} Lq{Lq} Lk{Lk}"
    bars = BARS["attention"]
    _report(tag + " out", {"out": nerr(_host(out), ref.detach().numpy())}, bars["out"])
    _report(tag + " data", {"d_query": nerr(_host(d_q), tq.grad.numpy()), "d_memory": nerr(_host(d_m), tm.grad.numpy())},
            bars["data"])
    _check_params(tag, blk, "p/", p, g0, False, bars["param"])


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["off", "host_key", "seed_acc", "frozen"])
@pytest.mark.parametrize("M", [128, 200, 1000, 6400])
def test_ffn_fused(tc_mode, M, variant):
    """FeedForwardBlock on the fused path (DenseRelu GEMM, DenseLinear + Dropout + residual + cluster LayerNorm, grouped
    split-K weight gradients).  off: dropout off, and the inference forward (z NULL) equals the training forward at
    rate 0 bit for bit; host_key: dropout keyed on the host; seed_acc: keyed by the seed word, d_x accumulated;
    frozen: gw NULL."""
    from oracle import reference_path as R
    from boosted_detr_b200.layers import Layer, dropout_site_key
    from boosted_detr_b200.transformers import FeedForwardBlock
    rng = np.random.default_rng(M + len(variant))
    Layer._rng = np.random.default_rng(9)
    x, go = _randn(rng, M, D), rng.standard_normal((M, D))
    dx = _dev(x)
    blk = FeedForwardBlock(name="ffn")
    blk.maybe_build([dx])
    w = _prepare(blk, rng, "p/")
    dropout, acc, frozen = variant in ("host_key", "seed_acc"), variant == "seed_acc", variant == "frozen"
    blk.rate = 0.1 if dropout else 0.0
    key = {"host_key": R.dropout_key(SEED, SITE), "seed_acc": dropout_site_key(SITE)}.get(variant, 0)
    out, ctx = blk.forward([dx], training=True, dropout_key=key, seed_dev=_seed_word(variant == "seed_acc"))
    assert ctx["fused"]
    if variant == "off":
        out_inf, ctx_inf = blk.forward([dx], training=False)
        assert ctx_inf["fused"] and ctx_inf["saved"]["z"] is None
        assert torch.equal(out_inf, out), "inference forward differs from the training forward at rate 0"

    p = R.params_to_torch(w, torch.float64, requires_grad=True)
    tx = _t64(x, True)
    ref = R.feed_forward_block(tx, p, "p", R.Dropout(SEED if dropout else None), SITE, True)
    (ref * _t64(go)).sum().backward()

    blk.trainable = not frozen
    g0 = _prefill_grads(blk, p, "p/", rng)
    d_x = torch.empty(M, D, device="cuda") if acc else None
    dx0 = _fill(d_x, rng, tx.grad) if acc else 0.0
    d_x = blk.backward(ctx, _dev(go), d_x=d_x, acc=acc)
    torch.cuda.synchronize()

    tag = f"ffn M{M} {variant}"
    bars = BARS["ffn"]
    _report(tag + " out", {"out": nerr(_host(out), ref.detach().numpy())}, bars["out"])
    _report(tag + " data", {"d_x": nerr(_host(d_x) - dx0, tx.grad.numpy())}, bars["data"])
    _check_params(tag, blk, "p/", p, g0, frozen, bars["param"])


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["seed", "frozen"])
@pytest.mark.parametrize("B,Q", [(1, 100), (3, 100), (16, 100), (2, 300)])
def test_decoder_self_hoisted(tc_mode, B, Q, variant):
    """Decoder self-attention hoisted out of the batch: [Q,D] projections / attention / output projection once, Dropout
    (its own mask per image over the broadcast rows) + residual + LayerNorm per image; d_q0 accumulates the batch sum.
    seed: dropout by the seed word; frozen: dropout off, gw NULL."""
    from oracle import reference_path as R
    from boosted_detr_b200.layers import Layer, dropout_site_key
    from boosted_detr_b200.transformers import AttentionBlock
    rng = np.random.default_rng(B * 1000 + Q + len(variant))
    Layer._rng = np.random.default_rng(10)
    q0, go = _randn(rng, Q, D, scale=0.5), rng.standard_normal((B, Q, D))
    dq0 = _dev(q0)
    blk = AttentionBlock(H, name="blk")
    blk.maybe_build([dq0.view(1, Q, D)] * 3)
    w = _prepare(blk, rng, "p/")
    dropout, frozen = variant == "seed", variant == "frozen"
    blk.rate = 0.1 if dropout else 0.0
    out, ctx = blk.forward_hoisted(dq0, dq0, B, True, dropout_site_key(SITE) if dropout else 0, _seed_word(dropout))

    p = R.params_to_torch(w, torch.float64, requires_grad=True)
    tq0 = _t64(q0, True)
    dec = tq0.unsqueeze(0).expand(B, Q, D)
    ref = R.attention_block(dec, dec, dec, p, "p", H, R.Dropout(SEED if dropout else None), SITE, True)
    (ref * _t64(go)).sum().backward()

    blk.trainable = not frozen
    g0 = _prefill_grads(blk, p, "p/", rng)
    d_q0 = torch.empty(Q, D, device="cuda")
    q00 = _fill(d_q0, rng, tq0.grad)
    blk.backward_hoisted(ctx, _dev(go), d_q0)
    torch.cuda.synchronize()

    tag = f"decoder_self B{B} Q{Q} {variant}"
    bars = BARS["decoder_self"]
    _report(tag + " out", {"out": nerr(_host(out), ref.detach().numpy())}, bars["out"])
    _report(tag + " data", {"d_q0": nerr(_host(d_q0) - q00, tq0.grad.numpy())}, bars["data"])
    _check_params(tag, blk, "p/", p, g0, frozen, bars["param"])


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["mult2", "cum_frozen"])
@pytest.mark.parametrize("M", [200, 1600, 6400])
@pytest.mark.parametrize("C,A", [(82, 3), (48, 296)])
def test_heads_fused(tc_mode, C, A, M, variant):
    """The three prediction heads of one block in one call (COCO C = 82, A = 3 and Fashionpedia C = 48, A = 296).
    mult2: mult 2, cum_in NULL, all BatchNorms training, d_x accumulated; cum_frozen: mult 1 onto running predictions,
    the attribute head frozen (bn_training 1,0,1 and gw[1] NULL): its moving statistics and gradient buffers must stay
    bit-identical.  Two identical forwards must agree bit for bit (outputs and moving statistics)."""
    from oracle import reference_path as R
    from boosted_detr_b200.layers import Layer
    from boosted_detr_b200.prediction_heads import (BN_MOMENTUM, BoxPredictionHead, MultiClassPredictionHead,
                                                    SingleClassPredictionHead, heads_backward_fused, heads_forward_fused)
    Q = 100
    B = M // Q
    rng = np.random.default_rng(C * 7 + A + M + len(variant))
    Layer._rng = np.random.default_rng(11)
    x = _randn(rng, B, Q, D)
    dx = _dev(x)
    heads = (SingleClassPredictionHead(C, D, Q, name="cat"), MultiClassPredictionHead(A, D, Q, name="attr"),
             BoxPredictionHead(D, Q, name="box"))
    w = {}
    for hd in heads:
        hd.maybe_build([dx])
        w.update(_prepare(hd, rng, hd.name + "/"))
    frozen = variant == "cum_frozen"
    heads[1].trainable = not frozen
    mult = 2.0 if variant == "mult2" else 1.0
    cum_np = None if variant == "mult2" else [tf32(rng.uniform(0, 1, (B, Q, n))) for n in (C, A, 4)]
    cum_in = None if cum_np is None else [_dev(c) for c in cum_np]
    stat_keys = [(hd, f"BatchNorm/{s}") for hd in heads for s in ("moving_mean", "moving_variance")]
    stats0 = {(hd.name, k): _host(hd._weights[k]).copy() for hd, k in stat_keys}

    first, _ = heads_forward_fused(heads, dx, True, cum_in, mult)
    torch.cuda.synchronize()
    stats1 = {(hd.name, k): _host(hd._weights[k]).copy() for hd, k in stat_keys}
    for hd, k in stat_keys:                      # rerun from the same moving statistics
        hd._weights[k].copy_(torch.from_numpy(stats0[(hd.name, k)]))
    cum, ctx = heads_forward_fused(heads, dx, True, cum_in, mult)
    torch.cuda.synchronize()
    for a, b in zip(first, cum):
        assert torch.equal(a, b), "two identical forwards differ"
    for hd, k in stat_keys:
        assert np.array_equal(_host(hd._weights[k]), stats1[(hd.name, k)]), f"{hd.name} {k}: not deterministic"

    p = R.params_to_torch(w, torch.float64, requires_grad=True)
    tx = _t64(x, True)
    new_stats, refs = {}, []
    for k, (hd, fn) in enumerate(zip(heads, (R.category_head, R.attribute_head, R.box_head))):
        a = fn(tx, p, hd.name, hd.trainable, new_stats)
        refs.append((0.0 if cum_np is None else _t64(cum_np[k])) + mult * a)
    d_cum = [rng.standard_normal(tuple(r.shape)) for r in refs]
    sum((r * _t64(g)).sum() for r, g in zip(refs, d_cum)).backward()

    tag = f"heads C{C} A{A} M{M} {variant}"
    bars = BARS["heads"]
    _report(tag + " out", {hd.name: nerr(_host(c), r.detach().numpy()) for hd, c, r in zip(heads, cum, refs)}, bars["out"])
    errs = {}
    for hd, k in stat_keys:
        got, before = _host(hd._weights[k]), stats0[(hd.name, k)].astype(np.float64)
        if not hd.trainable:
            assert np.array_equal(got, before), f"frozen head {hd.name}: {k} was updated"
            continue
        # judge the increment (the batch statistic's share): the momentum term alone would hide a wrong statistic
        errs[f"{hd.name} {k}"] = nerr(got - BN_MOMENTUM * before, new_stats[f"{hd.name}/{k}"].numpy() - BN_MOMENTUM * before)
    _report(tag + " stats", errs, bars["stats"])

    g0 = {}
    for hd in heads:
        g0.update(_prefill_grads(hd, p, hd.name + "/", rng))
    acc = variant == "mult2"
    d_x = torch.empty(B, Q, D, device="cuda") if acc else None
    dx0 = _fill(d_x, rng, tx.grad) if acc else 0.0
    d_x = heads_backward_fused(heads, ctx, [_dev(g) for g in d_cum], d_x=d_x, acc=acc)
    torch.cuda.synchronize()
    _report(tag + " data", {"d_x": nerr(_host(d_x) - dx0, tx.grad.numpy())}, bars["data"])
    for hd in heads:
        _check_params(f"{tag} {hd.name}", hd, hd.name + "/", p, g0, not hd.trainable, bars["param"])


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("Lq,Lk", [(200, 130), (130, 200)])
def test_attention_fused_rejects_fold_rows_mismatch(tc_mode, Lq, Lk):
    """The fold's positional table has Lk rows; resid_pos and tab_q need Lq == Lk.  Both entry points reject a mismatch
    with BDETR_E_BAD_SHAPE before launching anything (the NaN-filled outputs stay untouched); the decoder fold (tab_k
    only) is accepted at the same shapes."""
    import ctypes
    from boosted_detr_b200 import _lib
    from boosted_detr_b200.device import ptr, stream_ptr
    from boosted_detr_b200.layers import Layer
    from boosted_detr_b200.transformers import LN_EPS, AttentionBlock, _struct, make_fold, pos_projection
    lib = _lib.load()
    B = 2
    rng = np.random.default_rng(12)
    Layer._rng = np.random.default_rng(12)
    dq, dm, dpos = _dev(_randn(rng, B, Lq, D)), _dev(_randn(rng, B, Lk, D)), _dev(_randn(rng, Lk, D))
    blk = AttentionBlock(H, name="blk")
    blk.maybe_build([dq, dm, dm])
    tq, tk = pos_projection(dpos, [(blk.AttentionLayer, "QueryProjection"), (blk.AttentionLayer, "KeyProjection")])
    w, gw = blk._structs()
    nan = lambda *s: torch.full(s, float("nan"), device="cuda")
    sv = {"qp": nan(B, Lq, D), "kp": nan(B, Lk, D), "vp": nan(B, Lk, D), "o": nan(B, H, Lq, D // H), "lse": nan(B, H, Lq),
          "z": nan(B, Lq, D), "mean": nan(B * Lq), "rstd": nan(B * Lq)}
    sc = {"d_qp": nan(B, Lq, D), "d_kp": nan(B, Lk, D), "d_vp": nan(B, Lk, D), "d_o": nan(B, H, Lq, D // H),
          "d_z": nan(B, Lq, D), "delta": nan(B, H, Lq)}
    svs, scs = _struct(_lib.AttnSaved, sv), _struct(_lib.AttnScratch, sc)
    out, d_out, d_query, d_memory, d_pos = nan(B, Lq, D), _dev(rng.standard_normal((B, Lq, D))), nan(B, Lq, D), nan(B, Lk, D), nan(Lk, D)
    d_resid, sums = nan(B, Lq, D), nan(4, max(Lq, Lk), D)
    bad = {"resid_pos": make_fold(pos=dpos, tab_k=tk, resid_pos=True, pos_tc=dpos),
           "tab_q + tab_k": make_fold(pos=dpos, tab_q=tq, tab_k=tk, pos_tc=dpos),
           "tab_q": make_fold(pos=dpos, tab_q=tq, pos_tc=dpos)}
    for what, fold in bad.items():
        rc = lib.bdetr_attention_fused_fwd(B, Lq, Lk, D, H, ptr(dq), ptr(dm), ctypes.byref(fold), ctypes.byref(w), 0.0, 0, None,
                                           LN_EPS, 1, ptr(out), ctypes.byref(svs), stream_ptr())
        assert rc == _lib.BDETR_E_BAD_SHAPE, (what, rc)
        rc = lib.bdetr_attention_fused_bwd(B, Lq, Lk, D, H, ptr(dq), ptr(dm), ctypes.byref(fold), ctypes.byref(w), 0.0, 0, None,
                                           ctypes.byref(svs), ptr(d_out), ptr(d_query), ptr(d_memory), 0, ptr(d_pos),
                                           ctypes.byref(gw), ctypes.byref(scs), ptr(d_resid), ptr(sums), stream_ptr())
        assert rc == _lib.BDETR_E_BAD_SHAPE, (what, rc)
        torch.cuda.synchronize()
        for nm, t in (("out", out), ("d_query", d_query), ("d_memory", d_memory), ("d_pos", d_pos), *sv.items()):
            assert torch.isnan(t).all(), f"{what}: {nm} was written by a rejected call"
    fold = make_fold(pos=dpos, tab_k=tk, pos_tc=dpos)
    rc = lib.bdetr_attention_fused_fwd(B, Lq, Lk, D, H, ptr(dq), ptr(dm), ctypes.byref(fold), ctypes.byref(w), 0.0, 0, None,
                                       LN_EPS, 1, ptr(out), ctypes.byref(svs), stream_ptr())
    torch.cuda.synchronize()
    assert rc == _lib.BDETR_OK and torch.isfinite(out).all()


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.skipif(os.environ.get(ARM_ENV) is not None, reason="already inside an A/B arm run")
@pytest.mark.parametrize("var,value", [("BDETR_LN_SPLIT", "1"), ("BDETR_LN_SPLIT", "2"), ("BDETR_UMMA_STAGES", "deep"),
                                       ("BDETR_WGRAD_CTAS", "148,296")])
def test_ab_arm_keeps_layer_parity(var, value):
    """The A/B arms DESIGN §5 keeps for repeating its measurements compute the same layers: the FFN and encoder-attention
    cases of this file rerun in a child interpreter with the switch set (the library reads it once per process)."""
    here = os.path.abspath(__file__)
    cmd = [sys.executable, *(["-s"] if sys.flags.no_user_site else []), "-m", "pytest", "-q", "-x", "-m", "gpu",
           "-p", "no:cacheprovider", f"{here}::test_ffn_fused", f"{here}::test_attention_encoder_fold"]
    env = {**os.environ, var: value, ARM_ENV: "1"}
    r = subprocess.run(cmd, cwd=ROOT, env=env, timeout=1500, capture_output=True, text=True)
    print(r.stdout[-4000:], r.stderr[-2000:])
    assert r.returncode == 0, f"{var}={value}: layer parity fails in this arm"
