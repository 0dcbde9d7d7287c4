"""Attention at head dim 64 (four heads at model width 256, eight at 512) on the fp32 SIMT path and the tf32 tcgen05 path:
the attention core against an fp64 softmax, AttentionBlock and the fused entry points against the fp64 oracle, whole
BoostedDETR steps with 4-head (and mixed 4 / 8-head) layers, and the head dims that are still refused.  The bars are the
ones the 8-head (d = 32) tests of the same entry points use."""
import numpy as np
import pytest
import torch

import test_dense_gpu as TD
import test_fused_tc_gpu as TF
from test_dense_gpu import _model_and_data, nerr
from test_tc_gpu import tf32

pytestmark = pytest.mark.gpu


@pytest.fixture()
def mode():
    from boosted_detr_b200 import _lib
    lib = _lib.load()

    def set_mode(m):
        lib.bdetr_set_mode({"fp32": _lib.MODE_FP32, "tf32": _lib.MODE_TF32, "fp16": _lib.MODE_FP16}[m])
    yield set_mode
    lib.bdetr_set_mode(_lib.MODE_FP32)


@pytest.fixture()
def tc_mode(mode):
    mode("tf32")


def _softmax_ref(q, k, v, H, d, rows=None):
    """fp64 attention of [B,L,H*d] inputs: o [B,H,len(rows),d] and lse [B,H,len(rows)] (log2 units) for the query rows `rows`."""
    B, Lq = q.shape[:2]
    rows = np.arange(Lq) if rows is None else rows
    o = np.empty((B, H, len(rows), d)); lse = np.empty((B, H, len(rows)))
    for b in range(B):
        for h in range(H):
            qh = q[b, rows, h * d:(h + 1) * d].astype(np.float64)
            kh = k[b, :, h * d:(h + 1) * d].astype(np.float64)
            vh = v[b, :, h * d:(h + 1) * d].astype(np.float64)
            s = qh @ kh.T / np.sqrt(d)
            mx = s.max(-1, keepdims=True)
            p = np.exp(s - mx)
            o[b, h] = (p / p.sum(-1, keepdims=True)) @ vh
            lse[b, h] = (np.log(p.sum(-1)) + mx[:, 0]) / np.log(2.0)
    return o, lse


def _core(B, H, Lq, Lk, d, q, k, v):
    from boosted_detr_b200 import _lib
    from boosted_detr_b200.device import ptr, stream_ptr
    dq, dk, dv = (torch.from_numpy(x).cuda() for x in (q, k, v))
    o = torch.full((B, H, Lq, d), float("nan"), device="cuda")
    lse = torch.full((B, H, Lq), float("nan"), device="cuda")
    _lib.call("bdetr_attention_core_fwd", B, H, Lq, Lk, d, ptr(dq), ptr(dk), ptr(dv), ptr(o), ptr(lse), stream_ptr())
    torch.cuda.synchronize()
    return o.cpu().numpy(), lse.cpu().numpy()


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,Lq,Lk", [(2, 400, 400), (16, 100, 400), (3, 130, 257), (1, 1050, 1050), (2, 4096, 4096)])
@pytest.mark.parametrize("m", ["fp32", "tf32"])
def test_attention_core_d64(mode, m, B, Lq, Lk):
    """bdetr_attention_core_fwd with H = 4, d = 64: fp32 mode within 1e-5 of an fp64 softmax, tf32 mode (inputs rounded to
    tf32 like the producers store them) within the bars of test_attention_core_multistream."""
    mode(m)
    H, d = 4, 64
    D = H * d
    rng = np.random.default_rng(Lq * 3 + Lk)
    q, k, v = (rng.standard_normal((B, L, D)).astype(np.float32) for L in (Lq, Lk, Lk))
    if m == "tf32":
        q, k, v = tf32(q), tf32(k), tf32(v)
    o, lse = _core(B, H, Lq, Lk, d, q, k, v)
    assert np.isfinite(o).all() and np.isfinite(lse).all()
    rows = None if Lq <= 1050 else np.unique(np.concatenate([np.arange(0, Lq, 61), np.arange(Lq - 130, Lq)]))
    ref_o, ref_l = _softmax_ref(q, k, v, H, d, rows)
    if rows is not None:
        o, lse = o[:, :, rows], lse[:, :, rows]
    e_o, e_l = nerr(o, ref_o), nerr(lse, ref_l)
    print(f"{m} attention core d=64 B{B} Lq{Lq} Lk{Lk}: o {e_o:.2e} lse {e_l:.2e}")
    if m == "fp32":
        assert e_o < 1e-5 and e_l < 1e-5
    else:
        assert e_o < 1e-3 and e_l < 1e-4


def test_attention_core_d64_at_config5_length(tc_mode):
    """L = 20 020 (config 5's 110 x 182 feature map) at d = 64, one image: served by the one-tile-per-CTA kernel (the
    multi-stream kernel is d = 32 only); a strided subsample of the query rows against an fp64 softmax over all keys."""
    B, H, d, L = 1, 4, 64, 20020
    rng = np.random.default_rng(20021)
    q = tf32(rng.standard_normal((B, L, H * d)) * 1.5)
    k, v = tf32(rng.standard_normal((B, L, H * d))), tf32(rng.standard_normal((B, L, H * d)))
    o, lse = _core(B, H, L, L, d, q, k, v)
    assert np.isfinite(o).all() and np.isfinite(lse).all()
    rows = np.unique(np.concatenate([np.arange(0, L, 257), np.arange(L - 140, L), np.arange(0, 130)]))
    ref_o, ref_l = _softmax_ref(q, k, v, H, d, rows)
    e_o, e_l = nerr(o[:, :, rows], ref_o), nerr(lse[:, :, rows], ref_l)
    print(f"attention core d=64 L={L}: {len(rows)} sampled rows x {H} heads: o {e_o:.2e} lse {e_l:.2e}")
    assert e_o < 1e-3 and e_l < 1e-4


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("Lq,Lk,selfattn", [(400, 400, True), (100, 400, False), (130, 257, False)])
@pytest.mark.parametrize("D,H", [(256, 4), (512, 8)])
@pytest.mark.parametrize("m", ["fp32", "tf32"])
def test_attention_block_d64(mode, m, D, H, Lq, Lk, selfattn):
    """AttentionBlock forward and backward (data and parameter gradients) through bdetr_attention_block_fwd / _bwd against
    R.attention_block.  fp32: the bars of test_attention_block_vs_oracle; tf32: those of test_attention_block_tf32."""
    from oracle import reference_path as R
    from boosted_detr_b200.layers import Layer
    from boosted_detr_b200.transformers import AttentionBlock
    mode(m)
    B = 2
    rng = np.random.default_rng(D + H + Lq + Lk)
    Layer._rng = np.random.default_rng(1)
    q = rng.standard_normal((B, Lq, D)).astype(np.float32)
    k = q if selfattn else rng.standard_normal((B, Lk, D)).astype(np.float32)
    v = rng.standard_normal((B, Lk, D)).astype(np.float32)
    go = rng.standard_normal((B, Lq, D)).astype(np.float32)
    blk = AttentionBlock(H, name="blk")
    dq = torch.from_numpy(q).cuda()
    dk = dq if selfattn else torch.from_numpy(k).cuda()
    dv = torch.from_numpy(v).cuda()
    blk.maybe_build([dq, dk, dv])
    for n, o, kk in blk.named_weights():
        if kk.endswith("bias") or kk.endswith("beta"):
            o._weights[kk].copy_(torch.from_numpy(rng.normal(0, 0.1, o._weights[kk].shape).astype(np.float32)))
        if kk.endswith("gamma"):
            o._weights[kk].copy_(torch.from_numpy((1 + rng.normal(0, 0.1, o._weights[kk].shape)).astype(np.float32)))
    out, ctx = blk.forward([dq, dk, dv], training=False)
    d_q, d_k, d_v = blk.backward(ctx, torch.from_numpy(go).cuda())
    torch.cuda.synchronize()
    w = {n[len("blk/"):]: o._weights[kk].cpu().numpy() for n, o, kk in blk.named_weights()}
    p = R.params_to_torch({"p/" + n: a for n, a in w.items()}, torch.float64, requires_grad=True)
    tq = torch.tensor(q, dtype=torch.float64, requires_grad=True)
    tk = tq if selfattn else torch.tensor(k, dtype=torch.float64, requires_grad=True)
    tv = torch.tensor(v, dtype=torch.float64, requires_grad=True)
    ref = R.attention_block(tq, tk, tv, p, "p", H, R.Dropout(None), 0, False)
    (ref * torch.tensor(go, dtype=torch.float64)).sum().backward()
    e_out = nerr(out.cpu().numpy(), ref.detach().numpy())
    data = {"d_query": nerr(d_q.cpu().numpy(), tq.grad.numpy()), "d_value": nerr(d_v.cpu().numpy(), tv.grad.numpy())}
    if not selfattn:
        data["d_key"] = nerr(d_k.cpu().numpy(), tk.grad.numpy())
    params = {}
    for n, o, kk in blk.named_weights():
        floor = 1e-30
        if "KeyProjection/bias" in n:      # mathematically zero: judged on the query-bias scale (fp32) or skipped (tf32)
            if m == "tf32":
                continue
            floor = float(p["p/AttentionLayer/QueryProjection/bias"].grad.abs().max())
        params[n] = nerr(o._grads[kk].cpu().numpy(), p["p/" + n[len("blk/"):]].grad.numpy(), floor)
    worst = max(params.items(), key=lambda kv: kv[1])
    print(f"{m} attention block D{D} H{H} Lq{Lq} Lk{Lk}: out {e_out:.2e} data {data} worst param {worst}")
    if m == "fp32":
        assert e_out < 1e-5
        assert max(list(data.values()) + list(params.values())) < 2e-5
        return
    sv = ctx["saved"]
    d = D // H
    ref_o, ref_l = _softmax_ref(*(sv[n].cpu().numpy() for n in ("qp", "kp", "vp")), H, d)
    e_o, e_l = nerr(sv["o"].cpu().numpy(), ref_o), nerr(sv["lse"].cpu().numpy(), ref_l)
    print(f"   core o {e_o:.2e} lse {e_l:.2e}")
    assert e_o < 1e-3 and e_l < 1e-4
    assert e_out < 2e-3
    assert data["d_query"] < 5e-3 and data["d_value"] < 1e-2 and data.get("d_key", 0.0) < 1e-2
    assert worst[1] < 1e-2


# ---------------------------------------------------------------------------------------------------------------------
# The fused entry points at H = 4: test_fused_tc_gpu's cases and DESIGN §2 bars with that file's head count set to 4.
@pytest.fixture()
def four_heads(tc_mode, monkeypatch):
    monkeypatch.setattr(TF, "H", 4)


@pytest.mark.parametrize("variant", ["plain", "seed_acc", "no_dq", "frozen"])
@pytest.mark.parametrize("B,L", [(16, 400), (3, 130)])
def test_attention_encoder_fold_h4(four_heads, B, L, variant):
    TF.test_attention_encoder_fold(None, B, L, variant)


@pytest.mark.parametrize("variant", ["acc", "no_dm"])
@pytest.mark.parametrize("B", [16, 2])
def test_attention_decoder_fold_h4(four_heads, B, variant):
    TF.test_attention_decoder_fold(None, B, variant)


def test_attention_no_fold_cross_h4(four_heads):
    TF.test_attention_no_fold_cross(None)


@pytest.mark.parametrize("variant", ["seed", "frozen"])
@pytest.mark.parametrize("B,Q", [(1, 100), (3, 100), (16, 100), (2, 300)])
def test_decoder_self_hoisted_h4(four_heads, B, Q, variant):
    TF.test_decoder_self_hoisted(None, B, Q, variant)


# ---------------------------------------------------------------------------------------------------------------------
# Whole model.  The step tests run on a model built with other head counts, and the oracle is told the same counts: its
# train_step_reference takes one head count, which serves the encoder blocks, and its decoder_block is wrapped so that the
# decoder blocks use the decoder's own count (the reference constructor's separate num_encoder_heads / num_decoder_heads).
@pytest.fixture()
def heads(monkeypatch):
    from boosted_detr_b200.parameters import ModelParameters
    from oracle import reference_path as R

    def set_heads(enc, dec):
        orig_params, orig_ref, orig_dec = ModelParameters.default_params, R.train_step_reference, R.decoder_block

        def params(self, value=None):
            p = orig_params(self, value)
            p.update(num_encoder_heads=enc, num_decoder_heads=dec)
            return p

        def ref(params_, features, targets, num_blocks, num_heads, *a, **kw):
            assert num_heads == 8           # what the 8-head tests pass
            return orig_ref(params_, features, targets, num_blocks, enc, *a, **kw)

        def decoder_block(enc_value, dec_in, enc_key, p, prefix, num_heads, *a, **kw):
            assert num_heads == enc
            return orig_dec(enc_value, dec_in, enc_key, p, prefix, dec, *a, **kw)
        monkeypatch.setattr(ModelParameters, "default_params", params)
        monkeypatch.setattr(R, "train_step_reference", ref)
        monkeypatch.setattr(R, "decoder_block", decoder_block)
    return set_heads


def test_model_train_step_h4_fp32(heads):
    """Config-1 size (2 block pairs, batch 2, 20 x 20 features, 100 queries), 4 encoder and 4 decoder heads, fp32 mode:
    forward, Hungarian loss and every gradient within the bars of test_model_train_step_vs_oracle."""
    heads(4, 4)
    TD.test_model_train_step_vs_oracle(2, 2, 20, 20, False, "COCO")


@pytest.mark.parametrize("enc,dec", [(4, 4), (4, 8)])
def test_model_train_step_h4_tf32(tc_mode, heads, enc, dec):
    """The same size in tf32 mode (the fused path), 4 / 4 heads and a mixed model with 4 encoder and 8 decoder heads,
    against the fp64 oracle given the GPU's assignments: loss vector and running predictions within 1e-3, the whole
    gradient within the 5e-2 relative L2 of test_config2_size_tf32_vs_fp64_oracle.  (Single bias gradients of the last
    block reach 0.05-0.12 in relative L2 on this data for 8-head decoders too: the loss gradient is ill-conditioned next to
    the .999 clip, so test_model_train_step_tf32's per-tensor 5e-2 bar holds only for some random models.)"""
    from oracle import reference_path as R
    from test_bench_path_gpu import _masks_from_ctx
    heads(enc, dec)
    N, B, T, Q = 2, 2, 20, 100
    model, w, inputs = _model_and_data(N=N, B=B, rows=20, cols=20, Q=Q, T=T, attribute_weight=0.0)
    assert model.EncoderTransformerBlocks[0].num_attention_heads == enc and model.DecoderBlocks[0].num_attention_heads == dec
    model.train_step(inputs)
    torch.cuda.synchronize()
    masks = _masks_from_ctx(model.last_ctx_train, B, T, Q)
    tg = (inputs["category"], inputs["attribute"], inputs["bbox"], inputs["num_objects"])
    out, grads, _ = R.train_step_reference(w, inputs["features"], tg, N, 8, torch.float64, weights=R.model_weights(0.0),
                                           forced_masks=masks)
    e_loss = nerr(model.metric_tensors["loss"].cpu().numpy(), out["loss"].detach().numpy())
    e_pred = {n: nerr(g_.cpu().numpy(), r_.detach().numpy()) for g_, r_, n in zip(model.last_preds, out["preds"], ["cat", "attr", "box"])}
    g = model.get_grads_dict()
    assert set(g) == set(grads)
    num = sum(float(((g[k].astype(np.float64) - grads[k]) ** 2).sum()) for k in grads)
    rel = (num / sum(float((grads[k] ** 2).sum()) for k in grads)) ** 0.5
    print(f"tf32 step enc {enc} / dec {dec} heads: loss {e_loss:.2e} preds {e_pred} whole-gradient rel L2 {rel:.2e}")
    assert e_loss < 1e-3 and max(e_pred.values()) < 1e-3
    assert rel < 5e-2


def test_graph_replay_equals_eager_h4_config2(tc_mode, heads):
    """Config-2 size (6 block pairs, batch 16, 20 x 20 features) with 4 heads everywhere, tf32 mode, dropout on: the
    captured step's replay equals the eager step bit for bit (metric vectors and running predictions)."""
    from boosted_detr_b200.graph import GraphedTrainStep
    heads(4, 4)
    model, _, inputs = _model_and_data(N=6, B=16, rows=20, cols=20)
    assert model.EncoderTransformerBlocks[0].num_attention_heads == 4 and model.DecoderBlocks[0].num_attention_heads == 4
    assert model._use_fused(torch.empty(inputs["features"].shape)), "a 4-head width-256 model takes the fused path"
    w0 = {k: v.copy() for k, v in model.get_weights_dict().items()}
    seed = 2024
    model.dropout_seed = seed
    model.train_step(inputs)
    torch.cuda.synchronize()
    eager = ({k: v.clone() for k, v in model.metric_tensors.items()}, [p.clone() for p in model.last_preds])
    model.set_weights_dict(w0)
    model.dropout_seed = seed + 17
    gs = GraphedTrainStep(model, inputs)
    model.set_weights_dict(w0)
    model.dropout_seed = seed
    gs.load(inputs)
    gs.replay()
    torch.cuda.synchronize()
    for k in ("loss", "Category_Loss", "Attribute_Loss", "Box_Loss", "Existence_Loss", "IOU"):
        assert torch.equal(gs.metrics[k], eager[0][k]), k
    for a, b in zip(model.last_preds, eager[1]):
        assert torch.equal(a, b)


def test_fp16_mode_h4_equals_tf32(mode, heads):
    """BDETR_MODE_FP16 at d = 64: the fp16 attention kernel serves d = 32 only, so inference runs the tf32 kernels and the
    predictions are bit-identical to tf32 mode (4 images x 48 x 40 = 1 920 encoder tokens, a length the fp16 kernel would
    take at d = 32)."""
    from boosted_detr_b200 import _lib
    heads(4, 4)
    assert _lib.load().bdetr_attention_f16_workspace_bytes(4, 4, 1920, 1920, 64) == 0
    model, _, inputs = _model_and_data(N=2, B=4, rows=48, cols=40)
    got = {}
    for m in ("tf32", "fp16"):
        mode(m)
        got[m] = [p.clone() for p in model.call({"features": inputs["features"]}, training=False)]
        torch.cuda.synchronize()
    for a, b in zip(got["tf32"], got["fp16"]):
        assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("m", ["fp32", "tf32"])
@pytest.mark.parametrize("H", [16, 2])
def test_other_head_dims_are_refused(mode, m, H):
    """d = 16 (16 heads at 256) and d = 128 (2 heads at 256) return BDETR_E_UNSUPPORTED, naming the supported head dims."""
    from boosted_detr_b200 import _lib
    from boosted_detr_b200.device import ptr, stream_ptr
    mode(m)
    lib = _lib.load()
    B, L, D = 1, 130, 256
    d = D // H
    x = torch.zeros(B, L, D, device="cuda")
    o, lse = torch.empty(B, H, L, d, device="cuda"), torch.empty(B, H, L, device="cuda")
    rc = lib.bdetr_attention_core_fwd(B, H, L, L, d, ptr(x), ptr(x), ptr(x), ptr(o), ptr(lse), stream_ptr())
    assert rc == _lib.BDETR_E_UNSUPPORTED
    msg = lib.bdetr_last_error().decode()
    assert "32" in msg and "64" in msg, msg


def test_forced_multistream_refused_at_d64(tc_mode):
    """bdetr_debug_force_attention_kernel(2 | 20..28) at d = 64: BDETR_E_UNSUPPORTED from the host, nothing launched,
    outputs untouched."""
    from boosted_detr_b200 import _lib
    from boosted_detr_b200.device import ptr, stream_ptr
    lib = _lib.load()
    B, H, L, d = 1, 4, 2100, 64
    x = torch.ones(B, L, H * d, device="cuda")
    o, lse = torch.full((B, H, L, d), float("nan"), device="cuda"), torch.full((B, H, L), float("nan"), device="cuda")
    try:
        for which in (2, 20, 24, 28):
            assert lib.bdetr_debug_force_attention_kernel(which) == 0
            torch.cuda.synchronize()
            n0 = lib.bdetr_launch_count()
            rc = lib.bdetr_attention_core_fwd(B, H, L, L, d, ptr(x), ptr(x), ptr(x), ptr(o), ptr(lse), stream_ptr())
            assert rc == _lib.BDETR_E_UNSUPPORTED, which
            assert lib.bdetr_launch_count() == n0, which
    finally:
        lib.bdetr_debug_force_attention_kernel(0)
    torch.cuda.synchronize()
    assert torch.isnan(o).all() and torch.isnan(lse).all()
    # and the automatic choice at this length and d = 64 is the one-tile kernel, which serves it
    o2, lse2 = _core(B, H, L, L, d, np.ones((B, L, H * d), np.float32), np.ones((B, L, H * d), np.float32),
                     np.ones((B, L, H * d), np.float32))
    assert np.allclose(o2, 1.0) and np.isfinite(lse2).all()
