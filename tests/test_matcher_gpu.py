"""GPU parity of the matcher trio (K7 cost matrix, K8 assignment, K9 matched loss + gradient)
against the oracle (oracle/reference_path.py) and the real scipy matcher."""
import numpy as np
import pytest
import torch
from scipy.optimize import linear_sum_assignment

from util import synth_preds, synth_targets

pytestmark = pytest.mark.gpu

W = (1000.0, 1.0, 1.0, 100.0)     # w_cat, w_box, w_attr(model default 1.0), w_exist


def _dev(*arrs):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrs]


def _oracle_cost(tr, pr, w, dtype=torch.float32):
    from oracle import reference_path as R
    y_true = [torch.tensor(tr[0], dtype=dtype), torch.tensor(tr[1], dtype=dtype), torch.tensor(tr[2], dtype=dtype), tr[3]]
    y_pred = [torch.tensor(p, dtype=dtype) for p in pr]
    return R.weighted_cost(y_true, y_pred, (w[0], w[1], w[2], w[3]))[3].numpy()


def _ulp_diff(a, b):
    ai = a.view(np.int32).astype(np.int64)
    bi = b.view(np.int32).astype(np.int64)
    return np.abs(ai - bi)


@pytest.mark.parametrize("B,T,Q,C,A,w_attr", [(2, 20, 100, 82, 3, 1.0), (4, 20, 100, 82, 3, 0.0),
                                              (3, 20, 100, 48, 296, 1.0), (2, 100, 300, 82, 3, 1.0),
                                              (2, 5, 7, 5, 2, 100.0), (2, 33, 65, 33, 40, 1.0)])
def test_cost_matrix_vs_oracle(B, T, Q, C, A, w_attr):
    from boosted_detr_b200.losses_and_metrics import pairwise_cost
    rng = np.random.default_rng(B * 1000 + Q)
    tr = synth_targets(rng, B, T, C, A, attr_p=0.05)
    pr = synth_preds(rng, B, Q, C, A)
    got = pairwise_cost(_dev(*tr[:3]), _dev(*pr), W[0], W[1], w_attr).cpu().numpy()
    w = (W[0], W[1], w_attr, W[3])
    ref32 = _oracle_cost(tr, pr, w, torch.float32)
    ref64 = _oracle_cost(tr, pr, w, torch.float64)
    scale = np.abs(ref64).max()
    err = np.abs(got - ref64).max() / scale
    err_oracle = np.abs(ref32 - ref64).max() / scale
    ulps = _ulp_diff(got, ref32)
    print(f"cost[{B},{T},{Q}] C={C} A={A}: rel err vs fp64 {err:.2e} (oracle fp32 itself {err_oracle:.2e}); "
          f"ulp diff vs fp32 oracle max {ulps.max()} mean {ulps.mean():.3f} exact {np.mean(ulps == 0):.3f}")
    assert err < 1e-5            # fp32 tolerance stated by north_star
    assert np.isfinite(got).all()


def _scipy_expected(cost, n):
    B, T, Q = cost.shape
    c4r = np.full((B, T), -1, np.int32)
    for b in range(B):
        k = max(0, min(int(n[b]), T))
        r, c = linear_sum_assignment(cost[b, :k, :])
        c4r[b, r] = c
    return c4r


def _gpu_assign(cost, n):
    from boosted_detr_b200.losses_and_metrics import MatchingAssignment
    ma = MatchingAssignment()
    c4r, r4c, mask, assigned, status = ma.assign(*_dev(cost, n.astype(np.int32)))
    return c4r.cpu().numpy(), r4c.cpu().numpy(), mask.cpu().numpy(), assigned.cpu().numpy(), status.cpu().numpy()


def _check_assign(cost, n):
    cost = np.ascontiguousarray(cost, np.float32)
    c4r, r4c, mask, assigned, status = _gpu_assign(cost, n)
    exp = _scipy_expected(cost, n)
    assert (status == 0).all()
    bad = np.nonzero((c4r != exp).any(axis=1))[0]
    assert bad.size == 0, f"assignment differs from scipy for images {bad[:8]}: gpu {c4r[bad[0]]} scipy {exp[bad[0]]}"
    B, T, Q = cost.shape
    exp_mask = np.zeros_like(cost)
    bb, tt = np.nonzero(exp >= 0)
    exp_mask[bb, tt, exp[bb, tt]] = 1.0
    assert (mask == exp_mask).all()
    assert (assigned == exp_mask.max(axis=1)).all()
    inv = np.full((B, Q), -1, np.int32)
    inv[bb, exp[bb, tt]] = tt
    assert (r4c == inv).all()


# (20, 400) general solver, cost staged; (100, 400) general solver, unstaged; (130, 100) more targets than predictions,
# unstaged; (40, 307) register solver, staged, above 48 KB of dynamic shared memory; (20, 128) / (20, 129) the two
# register widths
LSAP_GENERAL = [(20, 400), (100, 400), (130, 100), (40, 307), (20, 128), (20, 129)]


@pytest.mark.parametrize("T,Q", [(20, 100), (100, 300), (7, 7), (33, 32), (64, 65), (100, 100)] + LSAP_GENERAL)
def test_lsap_bitexact_random(T, Q):
    rng = np.random.default_rng(T * 7 + Q)
    B = 48
    n = rng.integers(0, T + 1, B)
    n[0], n[1] = 0, T
    _check_assign(rng.random((B, T, Q)), n)
    _check_assign(rng.random((B, T, Q)) * 1000.0 + 3.0, n)


@pytest.mark.parametrize("T,Q", [(20, 100), (12, 12), (40, 50)] + LSAP_GENERAL)
def test_lsap_bitexact_ties(T, Q):
    rng = np.random.default_rng(T + Q)
    B = 64
    n = rng.integers(1, T + 1, B)
    _check_assign(np.round(rng.random((B, T, Q)) * 8) / 8, n)                 # quantised costs
    _check_assign(rng.integers(0, 3, (B, T, Q)).astype(np.float32), n)        # heavy ties
    _check_assign(np.tile(rng.random((B, T, 1)), (1, 1, Q)), n)               # identical columns (step-0 case)
    _check_assign(np.full((B, T, Q), 2.5), n)                                 # constant matrix -> identity
    dup = rng.random((B, T, Q))
    dup[:, :, Q // 2:Q // 2 * 2] = dup[:, :, :Q // 2]                         # duplicated columns
    _check_assign(dup, n)
    c = rng.integers(0, 4, (B, T, Q)).astype(np.float32)
    c[rng.random((B, T, Q)) < 0.15] = np.inf                                 # +inf entries are legal
    _check_assign(c, n)


def test_lsap_more_targets_than_predictions():
    rng = np.random.default_rng(5)
    B, T, Q = 16, 40, 12                                                     # scipy transposes internally
    n = rng.integers(0, T + 1, B)
    n[:4] = T
    _check_assign(rng.random((B, T, Q)), n)
    _check_assign(np.round(rng.random((B, T, Q)) * 4) / 4, n)


def _check_error_status(T, Q):
    """Per-image status and results next to invalid and infeasible images, with status words, index outputs and mask
    that start out holding garbage, and one image with more objects than target rows (it behaves like cost[b, :n])."""
    from boosted_detr_b200 import _lib
    from boosted_detr_b200.device import ptr, stream_ptr
    from boosted_detr_b200.losses_and_metrics import MatchingAssignment, raise_for_status
    rng = np.random.default_rng(9)
    B = 6
    cost = rng.random((B, T, Q)).astype(np.float32)
    n = np.full(B, T, np.int32)
    n[3] = 2
    n[5] = T + 3
    cost[1, 2, 3] = np.nan
    cost[2, 0, 0] = -np.inf
    cost[3, 4, 4] = np.nan            # beyond num_objects: ignored like cost[i,:n_i,:]
    cost[4, 1, :] = np.inf            # infeasible row
    dc, dn = _dev(cost, n)
    c4r = torch.full((B, T), 7, dtype=torch.int32, device="cuda")
    r4c = torch.full((B, Q), 7, dtype=torch.int32, device="cuda")
    mask = torch.full((B, T, Q), 7.0, device="cuda")
    assigned = torch.full((B, Q), 7.0, device="cuda")
    status = torch.full((B,), 12345, dtype=torch.int32, device="cuda")
    _lib.call("bdetr_lsap_assign", B, T, Q, ptr(dc), ptr(dn), ptr(c4r), ptr(r4c), ptr(mask), ptr(assigned), ptr(status),
              stream_ptr())
    c4r, r4c, mask, assigned, status = (t.cpu().numpy() for t in (c4r, r4c, mask, assigned, status))
    assert list(status) == [0, _lib.BDETR_E_INVALID_COST, _lib.BDETR_E_INVALID_COST, 0, _lib.BDETR_E_INFEASIBLE, 0]
    assert (c4r[1] == -1).all() and (c4r[4] == -1).all() and (r4c[1] == -1).all() and (r4c[4] == -1).all()
    for b in (0, 3, 5):
        r, c = linear_sum_assignment(cost[b, :n[b]])
        exp_c4r, exp_r4c, exp_mask = np.full(T, -1), np.full(Q, -1), np.zeros((T, Q), np.float32)
        exp_c4r[r], exp_r4c[c], exp_mask[r, c] = c, r, 1.0
        assert (c4r[b] == exp_c4r).all() and (r4c[b] == exp_r4c).all(), b
        assert (mask[b] == exp_mask).all() and (assigned[b] == exp_mask.max(axis=0)).all(), b
    with pytest.raises(ValueError, match="invalid numeric"):
        MatchingAssignment()(*_dev(cost, n))
    with pytest.raises(ValueError, match="infeasible"):
        raise_for_status(torch.tensor([0, _lib.BDETR_E_INFEASIBLE]))


def test_lsap_error_status():
    """Validation fused into the register solver's staging copy."""
    _check_error_status(6, 9)


@pytest.mark.parametrize("T,Q", [(20, 400), (100, 300)])
def test_lsap_error_status_separate_validate(T, Q):
    """The general solver (20, 400) and the register solver on an unstaged cost (100, 300), both behind the separate
    validate kernel and a memset of the status words."""
    _check_error_status(T, Q)


def test_end_to_end_assignment_on_gpu_cost():
    """GPU cost bits -> scipy  ==  GPU cost -> GPU solver; also reports flips vs the fp32 oracle cost."""
    from boosted_detr_b200.losses_and_metrics import pairwise_cost
    rng = np.random.default_rng(11)
    B, T, Q, C, A = 32, 20, 100, 82, 3
    tr = synth_targets(rng, B, T, C, A)
    pr = synth_preds(rng, B, Q, C, A)
    cost = pairwise_cost(_dev(*tr[:3]), _dev(*pr), W[0], W[1], W[2]).cpu().numpy()
    _check_assign(cost, tr[3])
    ref = _oracle_cost(tr, pr, W, torch.float32)
    a, b = _scipy_expected(cost, tr[3]), _scipy_expected(ref, tr[3])
    flips = int((a != b).sum())
    print(f"assignment flips GPU-cost vs oracle-cost: {flips} of {int((b >= 0).sum())}")
    assert flips <= 2


def test_step0_identical_predictions():
    """zero-initialised queries -> all Q predictions identical -> row i must go to column i."""
    from boosted_detr_b200.losses_and_metrics import pairwise_cost
    rng = np.random.default_rng(13)
    B, T, Q, C, A = 4, 20, 100, 82, 3
    tr = synth_targets(rng, B, T, C, A)
    pr = [np.repeat(p[:, :1], Q, axis=1) for p in synth_preds(rng, B, Q, C, A)]
    cost = pairwise_cost(_dev(*tr[:3]), _dev(*pr), W[0], W[1], W[2]).cpu().numpy()
    assert (cost == cost[:, :, :1]).all()
    c4r = _gpu_assign(cost, tr[3])[0]
    for b in range(B):
        assert (c4r[b, :tr[3][b]] == np.arange(tr[3][b])).all()
    _check_assign(cost, tr[3])


def test_cost_matrix_fwd_equals_prepared_path():
    """bdetr_cost_matrix_fwd -- the prepared path on a library-owned, grow-only scratch buffer -- gives the bits of
    bdetr_cost_targets_prepare + bdetr_cost_matrix_prepared.  The second, larger shape makes the buffer grow."""
    from boosted_detr_b200 import _lib
    from boosted_detr_b200.device import ptr, stream_ptr
    from boosted_detr_b200.losses_and_metrics import pairwise_cost
    for B, T, Q, C, A in [(2, 5, 7, 5, 2), (8, 100, 300, 1205, 3)]:
        rng = np.random.default_rng(T + C)
        tr = _dev(*synth_targets(rng, B, T, C, A, attr_p=0.05)[:3])
        pr = _dev(*synth_preds(rng, B, Q, C, A))
        want = pairwise_cost(tr, pr, W[0], W[1], W[2]).cpu().numpy()
        got = torch.full((B, T, Q), float("nan"), device="cuda")
        _lib.call("bdetr_cost_matrix_fwd", B, T, Q, C, A, *(ptr(t) for t in tr), *(ptr(t) for t in pr), W[0], W[1], W[2],
                  ptr(got), stream_ptr())
        got = got.cpu().numpy()
        assert np.isfinite(want).all()
        assert np.array_equal(got.view(np.int32), want.view(np.int32)), (B, T, Q, C, A)


# (2, 32, 100, 82, 3): the last T of the warp-per-row form; T > 32 runs one thread per row, with the attribute term
# inline for A <= 8 ((2, 100, 300, 82, 3) is BASELINE config 4) and a warp per row above ((2, 33, 65, 33, 9), and
# (2, 40, 100, 48, 296) at the Fashionpedia A); (1, 300, 300, 82, 8): more rows than the 256 threads of the CTA
@pytest.mark.parametrize("B,T,Q,C,A,w_attr", [(2, 20, 100, 82, 3, 1.0), (3, 20, 100, 48, 296, 1.0), (4, 9, 17, 6, 5, 0.0),
                                              (2, 32, 100, 82, 3, 1.0), (2, 100, 300, 82, 3, 1.0), (2, 100, 300, 82, 3, 0.0),
                                              (2, 33, 65, 33, 9, 1.0), (2, 40, 100, 48, 296, 1.0), (1, 300, 300, 82, 8, 1.0)])
def test_matched_loss_and_gradient_vs_oracle(B, T, Q, C, A, w_attr):
    """Matched losses, IoU metric and gradients against the fp64 oracle given the GPU's assignment.  Caught at T = 32: the
    accumulation check compared with the fp64 gradient element by element at rtol 1e-4, which fp32 arithmetic itself
    misses where box terms cancel (the fp32 oracle by 3.7e-4); it now compares with the first call's own gradient."""
    from oracle import reference_path as R
    from boosted_detr_b200.losses_and_metrics import MatchingLoss
    rng = np.random.default_rng(17 + B)
    tr = synth_targets(rng, B, T, C, A, attr_p=0.05)
    if T >= 32:         # the last image with every target row live, so that the last row (t = T - 1) is matched
        for x, f in zip(tr, synth_targets(rng, 1, T, C, A, attr_p=0.05, min_n=T)):
            x[-1] = f[0]
    pr = synth_preds(rng, B, Q, C, A, k_sum=2)
    pr[0][0, :5, 0] = 1.2          # saturate safe_clip on a few entries (zero gradient there)
    pr[0][0, 5:9, 0] = 0.0001
    w = (W[0], W[1], w_attr, W[3])
    ml = MatchingLoss(category_weight=w[0], box_weight=w[1], attribute_weight=w[2], exist_weight=w[3])
    d_tr, d_pr = _dev(*tr), _dev(*pr)
    losses, metrics = ml([d_tr, d_pr])
    ctx = ml.last_ctx
    mask = np.zeros((B, T, Q), np.float32)
    c4r = ctx["col4row"].cpu().numpy()
    bb, tt = np.nonzero(c4r >= 0)
    mask[bb, tt, c4r[bb, tt]] = 1.0
    # oracle with the same (GPU) assignment, fp64, autograd gradient of the summed total
    dt = torch.float64
    y_true = [torch.tensor(tr[0], dtype=dt), torch.tensor(tr[1], dtype=dt), torch.tensor(tr[2], dtype=dt), tr[3]]
    y_pred = [torch.tensor(p, dtype=dt, requires_grad=True) for p in pr]
    ref_losses, ref_iou, ref_mask, _ = R.matching_loss(y_true, y_pred, w, mask=torch.tensor(mask, dtype=dt))
    # and the oracle's own assignment must agree with the GPU's on this data -- or, where the GPU's fp32 cost and the
    # oracle's differ in their last bits at a near-tie (possible at T >= 100), be just as optimal under the fp64 cost
    _, _, own_mask, cost64 = R.matching_loss(y_true, [p.detach() for p in y_pred], w)
    own_mask = own_mask.numpy()
    if not (own_mask == mask).all():
        cost64 = cost64.numpy()
        tot_gpu, tot_own = (cost64 * mask).sum((1, 2)), (cost64 * own_mask).sum((1, 2))
        print(f"assignments differ at a near-tie: optimal totals {tot_own} (oracle) vs {tot_gpu} (GPU)")
        assert np.abs(tot_gpu - tot_own).max() <= 1e-6 * np.abs(tot_own).max()
    for k, name in enumerate(["total", "cat", "attr", "box", "exist"]):
        g = losses[k].cpu().numpy().astype(np.float64)
        r = ref_losses[k].detach().numpy()
        rel = np.abs(g - r).max() / max(np.abs(r).max(), 1e-30)
        print(f"{name}: rel {rel:.2e}")
        assert rel < 1e-5, name
    gi = metrics[0].cpu().numpy()
    assert gi.shape == (1, Q)
    assert np.abs(gi - ref_iou.detach().numpy()).max() < 1e-6
    ref_losses[0].sum().backward()
    d = [torch.zeros_like(t) for t in d_pr]
    ml.backward(ctx, d[0], d[1], d[2], gscale=1.0)
    for got, ref, name in zip(d, y_pred, ["d_cat", "d_attr", "d_box"]):
        r = ref.grad.numpy()
        g = got.cpu().numpy().astype(np.float64)
        rel = np.abs(g - r).max() / max(np.abs(r).max(), 1e-30)
        print(f"{name}: rel {rel:.2e} (max |ref| {np.abs(r).max():.3e})")
        assert rel < 1e-5, name
    # accumulate semantics + gscale: a second call with gscale 0.5 adds half of the first call's gradient
    first = [t.cpu().numpy() for t in d]
    ml.backward(ctx, d[0], d[1], d[2], gscale=0.5)
    for got, g1, name in zip(d, first, ["d_cat", "d_attr", "d_box"]):
        assert np.allclose(got.cpu().numpy(), 1.5 * g1, rtol=1e-6, atol=0), name


def test_matcher_stress_full_size_properties():
    """BASELINE config 4 (B=256, T=100, Q=300): size-independent properties + scipy on a sample."""
    from boosted_detr_b200.losses_and_metrics import pairwise_cost
    rng = np.random.default_rng(23)
    B, T, Q, C, A = 256, 100, 300, 82, 3
    tr = synth_targets(rng, B, T, C, A)
    pr = synth_preds(rng, B, Q, C, A)
    cost = pairwise_cost(_dev(*tr[:3]), _dev(*pr), W[0], W[1], W[2])
    c4r, r4c, mask, assigned, status = _gpu_assign(cost.cpu().numpy(), tr[3])
    cost = cost.cpu().numpy()
    assert (status == 0).all()
    n = tr[3]
    for b in range(B):
        cols = c4r[b, :n[b]]
        assert (cols >= 0).all() and len(set(cols.tolist())) == n[b]      # a matching
        assert (c4r[b, n[b]:] == -1).all()
    assert mask.sum() == n.sum() and (mask.sum(axis=2) <= 1).all() and (mask.sum(axis=1) <= 1).all()
    assert (assigned.sum(axis=1) == n).all()
    sample = rng.choice(B, 24, replace=False)
    exp = _scipy_expected(cost[sample], n[sample])
    assert (c4r[sample] == exp).all()
    # optimality certificate: the matched total equals scipy's optimum for every image
    for b in sample:
        r, c = linear_sum_assignment(cost[b, :n[b]])
        assert cost[b, r, c].sum() == cost[b, np.arange(n[b]), c4r[b, :n[b]]].sum()
