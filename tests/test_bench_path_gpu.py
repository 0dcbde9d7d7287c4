"""The path bench.py times is the path these tests check: tensor-core (tf32) mode, BASELINE config 2 size, dropout on,
CUDA-graph replay, multi-stream scheduling -- against the fp64 oracle and against the eager step.

Tolerances (north_star): losses / predictions within 1e-3 relative of the fp64 oracle in the reduced-precision mode;
bit-exact where the comparison is between two executions of the same kernels (graph replay vs eager step, concurrency
on vs off, identical query rows).  Gradients are compared with a tolerance because the weight-gradient GEMMs and the
LayerNorm parameter gradients accumulate with floating-point atomics (TMA reduce-add, atomicAdd) whose order varies."""
import numpy as np
import pytest
import torch

from test_dense_gpu import _model_and_data, nerr
from util import synth_targets

pytestmark = pytest.mark.gpu


@pytest.fixture()
def tc_mode():
    from boosted_detr_b200 import _lib
    lib = _lib.load()
    lib.bdetr_set_mode(_lib.MODE_TF32)
    yield
    lib.bdetr_set_mode(_lib.MODE_FP32)


def _masks_from_ctx(ctx, B, T, Q):
    out = []
    for c in ctx["loss"]:
        c4r = c["col4row"].cpu().numpy()
        m = np.zeros((B, T, Q), np.float64)
        bb, tt = np.nonzero(c4r >= 0)
        m[bb, tt, c4r[bb, tt]] = 1.0
        out.append(torch.from_numpy(m))
    return out


def test_config2_size_tf32_vs_fp64_oracle(tc_mode):
    """BASELINE config 2 (6 pairs, batch 16, 20x20 features, 100 queries, T = 20, C = 82, A = 3), tensor-core mode,
    dropout ON (seed 2024 like bench.py), eager step: loss vector, metric vectors and the running predictions of
    the last block within 1e-3 of the fp64 oracle evaluated with the SAME assignments (forced masks: a tf32-sized cost
    perturbation may legitimately flip a near-tie, which is reported, not hidden); gradients within the tf32 bar."""
    from oracle import reference_path as R
    N, B, T, Q = 6, 16, 20, 100
    model, w, inputs = _model_and_data(N=N, B=B, rows=20, cols=20, Q=Q, T=T)
    model.dropout_seed = 2024
    model.train_step(inputs)
    torch.cuda.synchronize()
    ctx = model.last_ctx_train
    masks = _masks_from_ctx(ctx, B, T, Q)
    tg = (inputs["category"], inputs["attribute"], inputs["bbox"], inputs["num_objects"])
    out, grads, stats = R.train_step_reference(w, inputs["features"], tg, N, 8, torch.float64, dropout_seed=2024,
                                               weights=R.model_weights(1.0), forced_masks=masks)
    free, _, _ = R.train_step_reference(w, inputs["features"], tg, N, 8, torch.float64, dropout_seed=2024,
                                        weights=R.model_weights(1.0))
    flips = sum(int((a.numpy() != b.numpy()).any(axis=(1, 2)).sum()) for a, b in zip(free["masks"], masks))
    print(f"config-2 size: images whose assignment differs from the fp64 oracle's own: {flips} of {N * B}")
    assert flips <= N * B // 10
    m = model.metric_tensors
    e_loss = nerr(m["loss"].cpu().numpy(), out["loss"].detach().numpy())
    print(f"loss vector {e_loss:.2e}")
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
    # BatchNorm moving statistics (fused heads: per-128-row partials): the increment over momentum * old value, i.e.
    # the batch statistic's share, so that the exact momentum term does not hide it
    after = model.get_weights_dict()
    assert stats
    e_stats = {k: nerr(after[k] - R.BN_MOMENTUM * w[k].astype(np.float64), ref - R.BN_MOMENTUM * w[k].astype(np.float64))
               for k, ref in stats.items()}
    k_worst = max(e_stats, key=e_stats.get)
    print(f"  BatchNorm moving statistics: worst {k_worst} {e_stats[k_worst]:.2e} over {len(stats)} tensors")
    assert e_stats[k_worst] < 2e-3, k_worst         # measured 4.4e-4 (B200)


def _snapshot(model):
    return {k: v.copy() for k, v in model.get_weights_dict().items()}


def test_graph_replay_equals_eager_and_draws_fresh_masks(tc_mode):
    """GraphedTrainStep.replay() == eager train_step, bit for bit, with the same dropout seed (forward outputs; the
    gradient within reduction-order noise); consecutive replays draw DIFFERENT masks (Keras Dropout draws a fresh mask
    per call, reference transformers.py:135,147), each equal to the eager step with that seed."""
    from boosted_detr_b200.graph import GraphedTrainStep
    model, w, inputs = _model_and_data(N=3, B=4, rows=20, cols=20)
    seed = 991
    w0 = _snapshot(model)
    eager = []
    for s in (seed, seed + 1):
        model.set_weights_dict(w0)
        model.dropout_seed = s
        model.train_step(inputs)
        torch.cuda.synchronize()
        eager.append(({k: v.clone() for k, v in model.metric_tensors.items()}, [p.clone() for p in model.last_preds],
                      model._flat[1].clone()))
    assert not torch.equal(eager[0][0]["loss"], eager[1][0]["loss"]), "two seeds must give two masks"
    model.set_weights_dict(w0)
    model.dropout_seed = seed + 17                      # warm-up / capture run with some other seed
    gs = GraphedTrainStep(model, inputs)
    for i, s in enumerate((seed, seed + 1)):
        model.set_weights_dict(w0)                      # BatchNorm moving statistics were touched by the warm-up steps
        if i == 0:
            model.dropout_seed = s                      # the second replay must pick seed + 1 up by itself
        assert model.dropout_seed == s
        gs.load(inputs)
        gs.replay()
        torch.cuda.synchronize()
        for k in ("loss", "Category_Loss", "Attribute_Loss", "Box_Loss", "Existence_Loss", "IOU"):
            assert torch.equal(gs.metrics[k], eager[i][0][k]), (i, k)
        ge = nerr(model._flat[1].cpu().numpy(), eager[i][2].cpu().numpy())
        print(f"replay {i}: metric vectors bit-identical to the eager step; gradient difference {ge:.2e}")
        assert ge < 1e-4                                # float atomics (split-K reduce-adds, column sums) in a different order


@pytest.mark.parametrize("lr0", [0.0, 0.05])
def test_prefetched_call_equals_plain_call(tc_mode, lr0):
    """The e2e path of bench.py: `gs(batch, prefetch=next_batch)` copies the next batch under the running step and queues
    its staging -> static copies and the next step's learning-rate / dropout-seed words BEHIND the running graph.  Three
    steps on three different pinned host batches, optimizer inside the graph, against three plain `gs(batch)` calls:
      lr0 = 0     the weights never move, so every step's logs must be BIT-identical (right batch, right dropout seed per step);
      lr0 = .05   a rate that changes every step: step 0 bit-identical, and after every call the device words hold exactly
                  the values the schedule prescribes (the primed path has already pushed the NEXT step's rate and seed).
                  Later logs are not compared: float-atomic noise in the weight gradients flips near-tied assignments."""
    from boosted_detr_b200.graph import GraphedTrainStep
    from boosted_detr_b200.optimizers import SGD, CosineDecayRestarts
    from util import synth_targets

    def batches(model, n):
        out = []
        for i in range(n):
            rng = np.random.default_rng(100 + i)
            cat, attr, box, num = synth_targets(rng, 4, 20, model.num_categories, model.num_attributes, attr_p=0.05)
            feats = np.tanh(rng.standard_normal((4, 20, 20, 256))).astype(np.float32)
            d = {"features": feats, "category": cat, "attribute": attr, "bbox": box, "num_objects": num.astype(np.int32)}
            out.append({k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in d.items()})
        return out

    results = []
    for use_prefetch in (False, True):
        model, w, inputs = _model_and_data(N=2, B=4, rows=20, cols=20)
        lr = CosineDecayRestarts(initial_learning_rate=lr0, first_decay_steps=2, m_mul=.95, alpha=0.1)
        model.compile(optimizer=SGD(learning_rate=lr, momentum=.9, nesterov=True, clipnorm=0.1))
        w0 = _snapshot(model)
        bs = batches(model, 3)
        model.dropout_seed = 5
        gs = GraphedTrainStep(model, bs[0])
        model.set_weights_dict(w0)
        it0, seed0 = model.optimizer.iterations, 4242
        model.dropout_seed = seed0
        logs, words = [], []
        for i, b in enumerate(bs):
            nxt = bs[i + 1] if (use_prefetch and i + 1 < len(bs)) else None
            logs.append(gs(b, prefetch=nxt))
            torch.cuda.synchronize()
            ahead = 1 if nxt is not None else 0            # the primed path has pushed the next step's words already
            assert float(model.optimizer._lr_dev) == np.float32(lr(it0 + i + ahead)), (use_prefetch, i)
            assert int(model._seed_dev) == seed0 + i + ahead, (use_prefetch, i)
        assert model.optimizer.iterations == it0 + 3 and model.dropout_seed == seed0 + 3
        results.append((logs, _snapshot(model)))
    (l0, w_plain), (l1, w_pref) = results
    assert l0[0] == l1[0], (l0[0], l1[0])                # same weights, same batch, same seed: bit-identical forward
    assert l0[0] != l0[1]                                # different batches really give different logs
    if lr0 == 0.0:
        assert l0 == l1, (l0, l1)
        worst = max(nerr(w_pref[k], w_plain[k]) for k in w_plain)
        print(f"prefetched path vs plain calls, 3 steps at lr 0: logs bit-identical, worst weight / statistic difference {worst:.2e}")
        assert worst < 1e-6


def test_concurrency_switch_does_not_change_results(tc_mode):
    """bdetr_set_concurrency(0/1) only changes which streams the kernels run on."""
    from boosted_detr_b200 import _lib
    lib = _lib.load()
    model, w, inputs = _model_and_data(N=3, B=4, rows=20, cols=20)
    w0 = _snapshot(model)
    res = []
    try:
        for on in (1, 0):
            lib.bdetr_set_concurrency(on)
            model.set_weights_dict(w0)
            model.dropout_seed = 31
            model.train_step(inputs)
            torch.cuda.synchronize()
            res.append(({k: v.clone() for k, v in model.metric_tensors.items()}, [p.clone() for p in model.last_preds],
                        model._flat[1].clone()))
    finally:
        lib.bdetr_set_concurrency(1)
    for k in res[0][0]:
        assert torch.equal(res[0][0][k], res[1][0][k]), k
    for a, b in zip(res[0][1], res[1][1]):
        assert torch.equal(a, b)
    assert nerr(res[0][2].cpu().numpy(), res[1][2].cpu().numpy()) < 1e-4


@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_step0_zero_queries_tie_structure(mode):
    """The reference initialises the shared queries to zeros (transformers.py:428-431), so at step 0 every query row
    enters the decoder identical.  Because the attention output [B,H,Lq,d] is re-read as [B,Lq,H*d] without a permute
    (quirk Q1, transformers.py:100), output row r is the concatenation of flat rows 8r..8r+7 of the [H*Lq, d] view: rows
    whose eight pieces come from the same heads stay identical, rows that straddle a head boundary do not -- the
    predictions fall into a few groups of exactly tied queries (NOT one group: SURVEY 7.2's "identity assignment" claim
    overlooked Q1).  What parity needs at this step: (1) queries the fp64 oracle ties stay BIT-identical through every
    kernel (no order-dependent arithmetic between rows), so the ties are real ties; (2) the solver breaks them exactly
    like scipy does on the same cost bits; (3) in fp32 mode the assignment equals the oracle's."""
    from scipy.optimize import linear_sum_assignment
    from boosted_detr_b200 import _lib
    from boosted_detr_b200.boosted_model import BoostedDETR
    from boosted_detr_b200.parameters import baseline_params
    from oracle import reference_path as R
    lib = _lib.load()
    lib.bdetr_set_mode(_lib.MODE_TF32 if mode == "tf32" else _lib.MODE_FP32)
    try:
        N = 2
        model = BoostedDETR(**baseline_params(1), attribute_weight=1.0, seed=0).build()
        model.dropout_seed = None                       # dropout masks differ per row: off for this check
        w = model.get_weights_dict()
        assert float(np.abs(w["DecoderPrep/init_decoder_features"]).max()) == 0.0
        rng = np.random.default_rng(5)
        B, T, Q = 4, 20, 100
        cat, attr, box, n = synth_targets(rng, B, T, model.num_categories, model.num_attributes)
        feats = np.tanh(rng.standard_normal((B, 20, 20, 256))).astype(np.float32)
        model.train_step({"features": feats, "category": cat, "attribute": attr, "bbox": box, "num_objects": n})
        out, _, _ = R.train_step_reference(w, feats, (cat, attr, box, n), N, 8, torch.float64, weights=R.model_weights(1.0))
        groups_seen = 0
        for i, c in enumerate(model.last_ctx_train["loss"]):
            ref_cat = out["per_block_preds"][i][0].detach().numpy()              # [B,Q,C] fp64
            got = [p.cpu().numpy() for p in c["pred"]]
            cost = c["cost"].cpu().numpy()
            c4r = c["col4row"].cpu().numpy()
            for b in range(B):
                # groups of queries the oracle ties (identical rows up to fp64 rounding of the row-independent GEMMs)
                key = np.round(ref_cat[b] / 1e-11).astype(np.int64)
                _, inv = np.unique(key, axis=0, return_inverse=True)
                inv = inv.reshape(-1)
                for gid in np.unique(inv):
                    rows = np.nonzero(inv == gid)[0]
                    if len(rows) < 2:
                        continue
                    groups_seen += 1
                    for arr in got:
                        assert (arr[b, rows] == arr[b, rows[:1]]).all(), f"block {i} image {b}: tied queries {rows[:4]}.. are not bit-identical"
                    assert (cost[b][:, rows] == cost[b][:, rows[:1]]).all()
                r_, c_ = linear_sum_assignment(cost[b, :n[b], :])
                assert (c4r[b, :n[b]] == c_).all(), f"block {i} image {b}: solver differs from scipy on its own tie-heavy cost matrix"
                if mode == "fp32":
                    ref_mask = out["masks"][i][b].numpy()
                    assert (ref_mask[np.arange(n[b]), c4r[b, :n[b]]] == 1).all(), f"block {i} image {b}: assignment differs from the oracle's"
        assert groups_seen >= B * N * 4, "expected several groups of tied queries per image at step 0"
    finally:
        lib.bdetr_set_mode(_lib.MODE_FP32)


def test_attention_core_at_config5_length(tc_mode):
    """Long-sequence attention at its design size (L = 20 020 = BASELINE config 5's 110 x 182 feature map), all heads,
    one image: a strided subsample of the query rows against an fp64 softmax over ALL 20 020 keys."""
    from boosted_detr_b200 import _lib
    from boosted_detr_b200.device import ptr, stream_ptr
    B, H, d, L = 1, 8, 32, 20020
    D = H * d
    rng = np.random.default_rng(20020)

    def tf32(x):
        u = x.astype(np.float32).view(np.uint32).astype(np.uint64)
        return ((u + 0x1000) & 0xFFFFE000).astype(np.uint32).view(np.float32)

    q = tf32(rng.standard_normal((B, L, D)) * 1.5)      # wider scores than N(0,1): the lazy rescale path is exercised
    k = tf32(rng.standard_normal((B, L, D)))
    v = tf32(rng.standard_normal((B, L, D)))
    dq, dk, dv = (torch.from_numpy(x).cuda() for x in (q, k, v))
    o = torch.full((B, H, L, d), float("nan"), device="cuda")
    lse = torch.full((B, H, L), float("nan"), device="cuda")
    _lib.call("bdetr_attention_core_fwd", B, H, L, L, d, ptr(dq), ptr(dk), ptr(dv), ptr(o), ptr(lse), stream_ptr())
    torch.cuda.synchronize()
    o, lse = o.cpu().numpy(), lse.cpu().numpy()
    assert np.isfinite(o).all() and np.isfinite(lse).all()
    rows = np.unique(np.concatenate([np.arange(0, L, 257), np.arange(L - 140, L), np.arange(0, 130)]))   # incl. ragged last tile
    for h in range(H):
        qh = q[0, rows, h * d:(h + 1) * d].astype(np.float64)
        kh = k[0, :, h * d:(h + 1) * d].astype(np.float64)
        vh = v[0, :, h * d:(h + 1) * d].astype(np.float64)
        s = qh @ kh.T / np.sqrt(d)
        mx = s.max(-1, keepdims=True)
        p = np.exp(s - mx)
        ref_o = (p / p.sum(-1, keepdims=True)) @ vh
        ref_l = (np.log(p.sum(-1)) + mx[:, 0]) / np.log(2.0)
        e_o, e_l = nerr(o[0, h, rows], ref_o), nerr(lse[0, h, rows], ref_l)
        assert e_o < 1e-3 and e_l < 1e-4, (h, e_o, e_l)
    print(f"attention core L={L}: {len(rows)} sampled rows x {H} heads within 1e-3 of the fp64 softmax")


def test_frozen_head_batchnorm_runs_in_inference_mode():
    """Keras: BatchNormalization of a frozen layer (trainable = False, reference notebook cell 30) uses its moving
    statistics and does not update them, even inside a training step; the oracle is told the same.  fp32 layer path
    (B*Q = 24 rows)."""
    _check_frozen_block0(tc=False)


def test_frozen_head_batchnorm_runs_in_inference_mode_fused(tc_mode):
    """The same on the tf32 fused path (B*Q = 200 rows), where frozen heads run with bn_training 0 / gw NULL and frozen
    blocks with gw / d_pos NULL: their gradient buffers stay zero."""
    _check_frozen_block0(tc=True)


def _check_frozen_block0(tc):
    """Block 0 frozen, one training step against the oracle told the same: frozen heads keep their moving statistics,
    no frozen variable is updated, block 1 and the shared queries match the oracle's gradients."""
    from oracle import reference_path as R
    N = 2
    if tc:
        # attribute weight 0: with the attribute term the gradient is ill-conditioned next to the .999 clip and a
        # tf32-sized perturbation moves it by O(1) (test_model_train_step_tf32)
        model, w, inputs = _model_and_data(N=N, B=2, rows=20, cols=20, Q=100, T=20, attribute_weight=0.0)
    else:
        model, w, inputs = _model_and_data(N=N, B=2, rows=5, cols=5, Q=12, T=5)
    for lst in (model.EncoderTransformerBlocks, model.DecoderBlocks, model.CategoryBlocks, model.AttributeBlocks, model.BoxBlocks):
        lst[0].trainable = False
    model.dropout_seed = None
    model.train_step(inputs)
    torch.cuda.synchronize()
    assert model._use_fused(torch.empty(inputs["features"].shape)) == tc
    tg = (inputs["category"], inputs["attribute"], inputs["bbox"], inputs["num_objects"])
    B, T, Q = inputs["category"].shape[0], inputs["category"].shape[1], model.num_object_preds
    masks = _masks_from_ctx(model.last_ctx_train, B, T, Q) if tc else None     # same assignment as the GPU (tf32 near-ties)
    out, grads, stats = R.train_step_reference(w, inputs["features"], tg, N, 8, torch.float64,
                                               weights=R.model_weights(0.0 if tc else 1.0), frozen_blocks=(0,),
                                               forced_masks=masks)
    bar_stats, bar_loss = (5e-5, 1e-4) if tc else (1e-5, 1e-5)          # tf32 measured 7.0e-6 / 2.4e-6 (B200)
    after = model.get_weights_dict()
    for k in w:
        if "Head_0/BatchNorm/moving" in k:
            assert (after[k] == w[k]).all(), f"{k}: a frozen head's moving statistics were updated"
        if "Head_1/BatchNorm/moving" in k:
            print(f"  {k}: {nerr(after[k], stats[k]):.2e}")
            assert nerr(after[k], stats[k]) < bar_stats, k
    e_loss = nerr(model.metric_tensors["loss"].cpu().numpy(), out["loss"].detach().numpy())
    print(f"  loss vector {e_loss:.2e}")
    assert e_loss < bar_loss
    g = model.get_grads_dict()
    frozen = [k for k in g if k.split("/")[0].endswith("_0")]
    assert frozen
    for k in frozen:
        assert (after[k] == w[k]).all(), f"{k}: a frozen variable was updated"
        if tc:      # the fused path computes no parameter gradient for a frozen block or head (gw / d_pos NULL)
            assert not np.any(g[k]), f"{k}: a frozen variable received a gradient"
    gmax = max(float(np.abs(v).max()) for v in grads.values())
    worst = (0.0, None)
    for k, ref in grads.items():
        if ("_1/" in k or k.startswith("DecoderPrep")) and "KeyProjection/bias" not in k:      # (key bias: mathematically zero)
            if tc:      # the tf32 gradient bar of test_model_train_step_tf32: relative L2 per tensor
                e = float(np.linalg.norm(g[k] - ref) / max(np.linalg.norm(ref), 1e-30))
            else:
                e = nerr(g[k], ref, 1e-6 * gmax)
            worst = max(worst, (e, k))
    print(f"  worst block-1 / query gradient: {worst[1]} {worst[0]:.2e}")
    assert worst[0] < (5e-2 if tc else 5e-4), worst[1]


def test_bucketed_optimizer_equals_whole_buffer_update(tc_mode):
    """SURVEY 8f rank 1: the clip + SGD-Nesterov update queued bucket by bucket behind each block's gradients (what
    bench.py runs, eager and under the CUDA graph) leaves the same weights as one update of the whole flat buffer.
    (Compared after ONE step: at random initialisation the predictions are nearly tied, and from the second step on a
    1e-7 weight difference can legitimately flip an assignment.)"""
    from boosted_detr_b200.graph import GraphedTrainStep
    from boosted_detr_b200.optimizers import SGD, CosineDecayRestarts
    from boosted_detr_b200.parallel import DataParallel
    model, w, inputs = _model_and_data(N=3, B=4, rows=20, cols=20)
    w0 = _snapshot(model)
    mk = lambda: SGD(learning_rate=CosineDecayRestarts(1e-2, 40, m_mul=.95, alpha=.1), momentum=.9, nesterov=True, clipnorm=0.1)
    res = {}
    for mode in ("whole", "bucketed", "graph"):
        model.set_weights_dict(w0)
        model.dropout_seed = 77
        model.grad_allreduce = model.grad_bucket_hook = None
        model.bucket_pipeline = None
        model.compile(optimizer=mk())
        if mode != "whole":
            DataParallel(model)                       # world size 1: the bucket pipeline only carries the optimizer
        if mode == "graph":
            gs = GraphedTrainStep(model, inputs)
            assert gs.optimizer_in_hook
            model.set_weights_dict(w0)
            model.optimizer._accum.zero_()
            model.optimizer.iterations = 0
            model.dropout_seed = 77
            gs(inputs)
        else:
            model.train_step(inputs)
        torch.cuda.synchronize()
        assert model.optimizer.iterations == 1
        res[mode] = model._flat[0].clone()
    start = np.concatenate([np.asarray(w0[n], np.float32).ravel() for n in model._index])      # (weights did move)
    assert float(np.abs(res["whole"].cpu().numpy()).sum()) != float(np.abs(start).sum())
    for mode in ("bucketed", "graph"):
        e = nerr(res[mode].cpu().numpy(), res["whole"].cpu().numpy())
        print(f"{mode} optimizer vs whole-buffer update after one step: {e:.2e}")
        # one step from identical weights (the forward is bit-reproducible, so the assignments agree); what differs is the
        # order of the floating-point atomics inside the gradient kernels
        assert e < 1e-6
