"""Category vocabularies beyond COCO and Fashionpedia: Objects365 (C = 367), LVIS (C = 1205) and the 2048-class limit.

The fused heads run a category (or attribute) head wider than 320 outputs as column slabs of raw logits plus a row
activation; the matcher digests targets of more than 1024 classes, or too many to stage, straight from global memory,
and the cost matrix gathers the probabilities of the classes that occur instead of staging the whole 64 x C tile.
The existing test bodies are reused at the new shapes with their own bars; the model-level ones run on a synthetic
vocabulary of the wanted size."""
import numpy as np
import pytest
import torch

import test_bench_path_gpu as bench_path
import test_dense_gpu as dense
import test_detr_gpu as detr
import test_inference_tail_gpu as tail
from test_dense_gpu import nerr
import test_fused_tc_gpu as fused
import test_matcher_gpu as matcher
from test_fused_tc_gpu import _randn
from test_matcher_gpu import W, _check_assign, _dev, _oracle_cost, _ulp_diff
from util import synth_preds, synth_targets

pytestmark = pytest.mark.gpu

D = 256


@pytest.fixture()
def tc_mode():
    from boosted_detr_b200 import _lib
    lib = _lib.load()
    lib.bdetr_set_mode(_lib.MODE_TF32)
    yield
    lib.bdetr_set_mode(_lib.MODE_FP32)


@pytest.fixture()
def vocab(monkeypatch):
    """vocab(C, A): every ModelParameters vocabulary gets C - 2 categories and A - 2 attributes."""
    from boosted_detr_b200.parameters import ModelParameters

    def set_sizes(C, A=3):
        v = {"category": [f"cat_{i}" for i in range(C - 2)], "attribute": [f"attr_{i}" for i in range(A - 2)]}
        monkeypatch.setattr(ModelParameters, "default_vocab", lambda self: v)
    return set_sizes


@pytest.fixture()
def oracle_takes_gpu_relu_pattern(monkeypatch):
    """A hidden pre-activation within fp32 rounding of zero can land on the other side of the ReLU kink on the GPU than
    in fp64 (test_heads_fused's data at C = 2048, M = 200 has one at 1.9e-7), and the two backward passes then disagree
    on that element of d_h by its whole value.  Like the forced assignments of the whole-model tests, the fp64 oracle
    takes the GPU's ReLU pattern -- but only where its own pre-activation is within 1e-5 of the largest one; a pattern
    that differs anywhere else fails."""
    from boosted_detr_b200 import prediction_heads as PH
    seen = {}
    real_fwd, real_relu = PH.heads_forward_fused, torch.relu

    def fwd(heads, x, training, cum_in, mult):
        cum, ctx = real_fwd(heads, x, training, cum_in, mult)
        seen["h"], seen["k"] = ctx["saved"]["h"].cpu().numpy(), 0          # [3, M, Dh] after the ReLU
        return cum, ctx

    def relu(z):
        if z.dtype != torch.float64 or "h" not in seen:
            return real_relu(z)
        k = seen["k"]
        seen["k"] = (k + 1) % 3                                             # the oracle runs cat, attr, box in order
        keep = torch.from_numpy(seen["h"][k] > 0).reshape(z.shape)
        differ = keep != (z.detach() > 0)
        if differ.any():
            near = float(z.detach()[differ].abs().max())
            print(f"head {k}: {int(differ.sum())} ReLU decision(s) differ from the GPU's, largest |pre-activation| {near:.1e}")
            assert near <= 1e-5 * float(z.detach().abs().max()), "ReLU pattern differs away from the kink"
        return z * keep.to(z.dtype)

    monkeypatch.setattr(PH, "heads_forward_fused", fwd)
    monkeypatch.setattr(torch, "relu", relu)


# ---- 1. fused heads --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["mult2", "cum_frozen"])
@pytest.mark.parametrize("M", [200, 1600])
@pytest.mark.parametrize("C,A", [(367, 3), (1205, 3), (2048, 3), (82, 400)])
def test_heads_fused_wide(tc_mode, oracle_takes_gpu_relu_pattern, C, A, M, variant):
    fused.test_heads_fused(tc_mode, C, A, M, variant)


def test_heads_fused_wide_identical_rows_stay_identical(tc_mode):
    """Query rows that enter the heads identical leave them bit-identical, in every slab of the category head."""
    from boosted_detr_b200.layers import Layer
    from boosted_detr_b200.prediction_heads import (BoxPredictionHead, MultiClassPredictionHead, SingleClassPredictionHead,
                                                    heads_forward_fused)
    C, A, B, Q = 1205, 3, 4, 100
    rng = np.random.default_rng(3)
    Layer._rng = np.random.default_rng(11)
    x = _randn(rng, B, Q, D)
    x[:, 1::3] = x[:, :1]                       # every third query of an image repeats its first
    x[2] = x[0]                                 # and one image repeats another (a different row tile)
    dx = torch.from_numpy(x).cuda()
    heads = (SingleClassPredictionHead(C, D, Q, name="cat"), MultiClassPredictionHead(A, D, Q, name="attr"),
             BoxPredictionHead(D, Q, name="box"))
    cum, _ = heads_forward_fused(heads, dx, True, None, 1.0)
    for k, c in enumerate(cum):
        c = c.cpu().numpy()
        assert (c[:, 1::3] == c[:, :1]).all(), f"head {k}: repeated rows differ"
        assert (c[2] == c[0]).all(), f"head {k}: repeated image differs"
    assert np.allclose(cum[0].sum(-1).cpu().numpy(), 1.0, atol=1e-5)


# ---- 2. cost matrix, assignment, matched loss ------------------------------------------------------------------------
_WIDE = [(2, 20, 100, 367, 3, 0), (2, 20, 100, 1205, 3, 0), (2, 100, 300, 1205, 3, 0), (2, 20, 100, 2048, 3, 0),
         (2, 20, 100, 1205, 296, 0), (2, 20, 100, 1205, 3, 4)]


@pytest.mark.parametrize("B,T,Q,C,A,multi_hot,w_attr",
                         [pytest.param(*c, 1.0, id="-".join(map(str, c))) for c in _WIDE]
                         + [(2, 20, 100, 1205, 3, 0, 0.0), (2, 100, 300, 2048, 3, 0, 0.0)])
def test_cost_matrix_wide_vs_oracle(B, T, Q, C, A, multi_hot, w_attr):
    """Costs of the wide digest + gather cost kernels within 3 ulp of the fp32 oracle, built one image at a time; the
    assignment on the GPU cost bit-exact against scipy.  multi_hot: that many target rows per image carry five
    classes each, so the image has more class slots than target rows (the slots past the staged ones are read from
    global memory).  w_attr = 0: the gather kernel without the attribute term."""
    from boosted_detr_b200.losses_and_metrics import pairwise_cost
    rng = np.random.default_rng(C + T + A + multi_hot)
    tr = synth_targets(rng, B, T, C, A, attr_p=0.05)
    if multi_hot:
        for b in range(B):
            for t in range(min(multi_hot, int(tr[3][b]))):
                tr[0][b, t, rng.choice(np.arange(2, C), 5, replace=False)] = 1.0
    pr = synth_preds(rng, B, Q, C, A)
    w = (W[0], W[1], w_attr, W[3])
    got = pairwise_cost(_dev(*tr[:3]), _dev(*pr), w[0], w[1], w[2]).cpu().numpy()
    assert np.isfinite(got).all()
    worst = 0
    for b in range(B):
        one = lambda arrs: [a[b:b + 1] for a in arrs]
        trb = one(tr[:3]) + [tr[3][b:b + 1]]
        ref32 = _oracle_cost(trb, one(pr), w, torch.float32)[0]
        if multi_hot:       # a sum over several classes: the oracle sums in its own order
            ref64 = _oracle_cost(trb, one(pr), w, torch.float64)[0]
            assert np.abs(got[b] - ref64).max() / np.abs(ref64).max() < 1e-5
        else:
            worst = max(worst, int(_ulp_diff(got[b], ref32).max()))
    print(f"cost[{B},{T},{Q}] C={C} A={A} w_attr={w_attr}: max ulp vs fp32 oracle {worst}")
    assert worst <= 3
    _check_assign(got, tr[3])


def test_matched_loss_and_gradient_c1205():
    matcher.test_matched_loss_and_gradient_vs_oracle(2, 20, 100, 1205, 3, 1.0)


# ---- 3. / 4. whole model ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", [1205, 367])
def test_model_tf32_wide_vocab_vs_fp64_oracle(tc_mode, vocab, C):
    """BoostedDETR with 3 block pairs, batch 8, 20x20 features, Q = 100, T = 20, dropout on, fused path, against the
    fp64 oracle with the GPU's assignments (the bars of test_config2_size_tf32_vs_fp64_oracle)."""
    from oracle import reference_path as R
    vocab(C)
    N, B, T, Q = 3, 8, 20, 100
    model, w, inputs = dense._model_and_data(N=N, B=B, rows=20, cols=20, Q=Q, T=T)
    assert model.num_categories == C
    model.dropout_seed = 2024
    model.train_step(inputs)
    torch.cuda.synchronize()
    assert model._use_fused(inputs["features"])
    masks = bench_path._masks_from_ctx(model.last_ctx_train, B, T, Q)
    tg = (inputs["category"], inputs["attribute"], inputs["bbox"], inputs["num_objects"])
    out, grads, stats = R.train_step_reference(w, inputs["features"], tg, N, 8, torch.float64, dropout_seed=2024,
                                               weights=R.model_weights(1.0), forced_masks=masks)
    m = model.metric_tensors
    e_loss = nerr(m["loss"].cpu().numpy(), out["loss"].detach().numpy())
    print(f"C={C}: loss vector {e_loss:.2e}")
    assert e_loss < 1e-3
    for k in ["Category_Loss", "Attribute_Loss", "Box_Loss", "Existence_Loss"]:
        e = nerr(m[k].cpu().numpy(), out["metrics"][k].detach().numpy())
        print(f"  {k}: {e:.2e}")
        assert e < 1e-3, k
    for g, r, name in zip(model.last_preds, out["preds"], ["cat", "attr", "box"]):
        e = nerr(g.cpu().numpy(), r.detach().numpy())
        print(f"  running prediction {name}: {e:.2e}")
        assert e < 1e-3, name
    g = model.get_grads_dict()
    num = sum(float(((g[k].astype(np.float64) - grads[k]) ** 2).sum()) for k in grads)
    den = sum(float((grads[k] ** 2).sum()) for k in grads)
    rel = (num / den) ** 0.5
    print(f"  whole-gradient relative L2 error {rel:.2e}")
    assert rel < 5e-2
    after = model.get_weights_dict()
    assert stats
    e_stats = {k: nerr(after[k] - R.BN_MOMENTUM * w[k].astype(np.float64), ref - R.BN_MOMENTUM * w[k].astype(np.float64))
               for k, ref in stats.items()}
    k_worst = max(e_stats, key=e_stats.get)
    print(f"  BatchNorm moving statistics: worst {k_worst} {e_stats[k_worst]:.2e}")
    assert e_stats[k_worst] < 2e-3, k_worst


def test_model_fp32_c1205_vs_oracle(vocab):
    vocab(1205)
    dense.test_model_train_step_vs_oracle(2, 2, 20, 20, False, "COCO")


# ---- 5. plain DETR ---------------------------------------------------------------------------------------------------
def test_plain_detr_c1205_vs_oracle(vocab):
    vocab(1205)
    detr.test_plain_detr_train_step_vs_oracle()


# ---- 6. / 7. graph replay, step-0 ties -------------------------------------------------------------------------------
def test_graph_replay_c1205_equals_eager(tc_mode, vocab):
    vocab(1205)
    bench_path.test_graph_replay_equals_eager_and_draws_fresh_masks(tc_mode)


@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_step0_tie_structure_c1205(vocab, mode):
    vocab(1205)
    bench_path.test_step0_zero_queries_tie_structure(mode)


# ---- 8. inference tail -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_inference_tail_c1205(vocab, mode):
    """Early exit, and predict_indices' category tokens equal to torch's argmax of the model's own predictions."""
    from boosted_detr_b200 import _lib
    vocab(1205)
    tail.test_early_exit_returns_the_running_prediction_of_the_exit_block(mode)
    lib = _lib.load()
    lib.bdetr_set_mode(_lib.MODE_TF32 if mode == "tf32" else _lib.MODE_FP32)
    try:
        model, _, inputs = dense._model_and_data(N=2, B=2, rows=20, cols=20)
        assert model.num_categories == 1205
        feats = {"features": inputs["features"]}
        cat, _, _ = model.call(feats, training=False)
        tok_c, _, _ = model.predict_indices(feats)
        assert torch.equal(tok_c.reshape(-1).long().cpu(), cat.argmax(-1).reshape(-1).cpu())
    finally:
        lib.bdetr_set_mode(_lib.MODE_FP32)


# ---- 9. refusals above 2048 ------------------------------------------------------------------------------------------
def test_vocab_above_2048_is_refused(tc_mode):
    from boosted_detr_b200 import _lib
    from boosted_detr_b200.layers import Layer
    from boosted_detr_b200.prediction_heads import (BoxPredictionHead, MultiClassPredictionHead, SingleClassPredictionHead,
                                                    heads_forward_fused)
    C, A, B, T, Q = 2049, 3, 2, 20, 100
    rng = np.random.default_rng(9)
    Layer._rng = np.random.default_rng(11)
    dx = torch.from_numpy(_randn(rng, B, Q, D)).cuda()
    for cw, aw in ((C, A), (A, C)):
        heads = (SingleClassPredictionHead(cw, D, Q, name="cat"), MultiClassPredictionHead(aw, D, Q, name="attr"),
                 BoxPredictionHead(D, Q, name="box"))
        for hd in heads:
            hd.maybe_build([dx])
        before = [{k: v.clone() for k, v in hd._weights.items()} for hd in heads]
        with pytest.raises(_lib.BdetrError) as e:
            heads_forward_fused(heads, dx, True, None, 1.0)
        assert e.value.code == _lib.BDETR_E_UNSUPPORTED and "2048" in str(e.value)
        torch.cuda.synchronize()
        for hd, b0 in zip(heads, before):          # the moving statistics a training forward updates
            for k, v in hd._weights.items():
                assert torch.equal(v, b0[k]), f"{hd.name} {k} changed"

    lib = _lib.load()
    tr = _dev(*synth_targets(rng, B, T, C, A)[:3])
    pr = _dev(*synth_preds(rng, B, Q, C, A))
    nbytes = lib.bdetr_cost_targets_bytes(B, T, C, A)
    assert nbytes > 0
    prepared = torch.full((nbytes,), 0xA5, dtype=torch.uint8, device="cuda")
    rc = lib.bdetr_cost_targets_prepare(B, T, C, A, *[t.data_ptr() for t in tr], prepared.data_ptr(), None)
    assert rc == _lib.BDETR_E_UNSUPPORTED and b"2048" in lib.bdetr_last_error()
    cost = torch.full((B, T, Q), 7.0, device="cuda")
    rc = lib.bdetr_cost_matrix_prepared(B, T, Q, C, A, prepared.data_ptr(), *[t.data_ptr() for t in pr],
                                        W[0], W[1], W[2], cost.data_ptr(), None)
    assert rc == _lib.BDETR_E_UNSUPPORTED and b"2048" in lib.bdetr_last_error()
    torch.cuda.synchronize()
    assert (prepared == 0xA5).all() and (cost == 7.0).all()
