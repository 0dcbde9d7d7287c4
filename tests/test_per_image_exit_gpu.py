"""Per-image early exit (BoostedDETR.early_exit_per_image): every image leaves the forward at its own first confident
boundary, the images still running are gathered to the front of the batch and the later blocks run at that smaller batch.
Inference is independent per image, so every result must equal, bit for bit, the per-batch exit's running prediction of
the image's own exit block -- in eager calls and in GraphedInference's SWITCH graph."""
import numpy as np
import pytest
import torch

from test_dense_gpu import _model_and_data

pytestmark = pytest.mark.gpu

# (mode, N, B, rows, cols, Q): tf32 fused at config-2 size, tf32 fused at the reference default, the fp32 layer path,
# and fp16 mode at 84 x 84 tokens (the fp16 attention kernel serves every batch size there)
SHAPES = {
    "tf32_config2": ("tf32", 6, 16, 20, 20, 100),
    "tf32_reference": ("tf32", 4, 8, 18, 18, 96),
    "fp32_layers": ("fp32", 3, 4, 20, 20, 100),
    "fp16": ("fp16", 3, 4, 84, 84, 100),
}


@pytest.fixture()
def mode():
    from boosted_detr_b200 import _lib
    lib = _lib.load()

    def set_mode(m):
        lib.bdetr_set_mode({"fp32": _lib.MODE_FP32, "tf32": _lib.MODE_TF32, "fp16": _lib.MODE_FP16}[m])
    yield set_mode
    lib.bdetr_set_mode(_lib.MODE_FP32)


def _make(mode, name):
    m, N, B, rows, cols, Q = SHAPES[name]
    mode(m)
    model, _, inputs = _model_and_data(N=N, B=B, rows=rows, cols=cols, Q=Q)
    x = inputs["features"].copy()
    # images of different contrast: their confidences run apart, so thresholds can spread the exit blocks
    x *= np.linspace(0.25, 3.0, B, dtype=np.float32)[:, None, None, None]
    feats = {"features": x}
    fused = model._use_fused(torch.empty(x.shape))
    k_min = max(-(-128 // (rows * cols)), -(-128 // Q)) if fused else 1
    return model, feats, fused, k_min


def _eager(model, feats):
    out = [t.clone() for t in model.call(feats, training=False)]
    torch.cuda.synchronize()
    return out


def _reference(model, feats):
    """P[k] = the whole batch's running predictions after block k, c[:, k] = the per-image confidences at boundary k,
    both from the per-batch exit (threshold 0 stops right after min_blocks blocks)."""
    N = model.num_decoder_blocks
    model.early_exit_per_image = False
    P, c = [], []
    for k in range(N - 1):
        model.early_exit_threshold, model.early_exit_min_blocks = 0.0, k + 1
        P.append(_eager(model, feats))
        assert model.last_exit_block == k
        c.append(model.last_image_confidence.numpy().astype(np.float32).copy())
    model.early_exit_threshold = None
    P.append(_eager(model, feats))
    return P, np.stack(c, 1)                        # c [B, N - 1]


def _expect(c, thr, min_blocks, N, k_min):
    """Host model of the per-image exit: exit blocks, confidences, active counts (riders included)."""
    B = c.shape[0]
    t = np.float32(thr)
    e = np.full(B, N - 1, np.int32)
    conf = np.full(B, np.nan, np.float32)
    live = list(range(B))
    counts = [B] + [0] * (N - 1)
    for i in range(N - 1):
        if not live:
            break
        if i + 1 >= min_blocks:
            for b in live:
                conf[b] = c[b, i]
                if c[b, i] >= t:
                    e[b] = i
            live = [b for b in live if e[b] == N - 1]
        counts[i + 1] = max(len(live), k_min) if live else 0
    return e, conf, np.array(counts, np.int32)


def _cases(c, N, k_min, require_spread):
    """Threshold / min_blocks settings from the measured confidences: (spread) the most distinct exit blocks with N - 1
    among them, at least 3 when `require_spread`; (riders) fewer than k_min images left at some boundary; (same) every
    image at one boundary < N - 1; (never) a threshold no image reaches.  Where every image's confidence falls block by
    block (the reference-default model here), an image leaves at its first checked boundary or never: two exit blocks."""
    found, spread = {}, 0
    for mb in range(1, N):
        for t in sorted(set(c[:, mb - 1:].reshape(-1).tolist())):
            e, _, counts = _expect(c, t, mb, N, k_min)
            if N - 1 in e and len(set(e.tolist())) > spread:
                found["spread"], spread = (t, mb), len(set(e.tolist()))
            live = [int((e > i).sum()) for i in range(N - 1)]
            if any(0 < n < k_min or n == 1 for n in live) and len(set(e.tolist())) >= 2 and "riders" not in found:
                found["riders"] = (t, mb)
            if len(set(e.tolist())) == 1 and e[0] < N - 1 and "same" not in found:
                found["same"] = (t, mb)
    found["never"] = (2.0, 1)
    assert {"spread", "riders", "same"} <= set(found) and spread >= (3 if require_spread else 2), (found, c)
    return found


def _check_eager(model, feats, P, c, thr, mb, k_min):
    N, B = model.num_decoder_blocks, c.shape[0]
    e, conf, counts = _expect(c, thr, mb, N, k_min)
    model.early_exit_per_image = True
    model.early_exit_threshold, model.early_exit_min_blocks = thr, mb
    got = _eager(model, feats)
    assert np.array_equal(model.last_exit_blocks.numpy(), e)
    assert np.array_equal(model.last_image_confidence.numpy(), conf, equal_nan=True)
    assert np.array_equal(model.last_active_counts.numpy(), counts)
    assert model.last_exit_block == int(e.max())
    for b in range(B):
        for t in range(3):
            assert torch.equal(got[t][b], P[e[b]][t][b]), (b, int(e[b]), t)
    return got, e, counts


@pytest.mark.parametrize("shape", list(SHAPES))
def test_eager_per_image_equals_the_exit_blocks_predictions(mode, shape):
    from boosted_detr_b200 import _lib
    model, feats, fused, k_min = _make(mode, shape)
    if shape == "fp16":
        assert _lib.load().bdetr_attention_f16_workspace_bytes(1, 8, 7056, 7056, 32) > 0
    assert fused == (shape != "fp32_layers")
    N = model.num_decoder_blocks
    P, c = _reference(model, feats)
    cases = _cases(c, N, k_min, require_spread=shape == "tf32_config2")
    for name, (thr, mb) in cases.items():
        got, e, counts = _check_eager(model, feats, P, c, thr, mb, k_min)
        if name == "riders" and fused:
            assert any(0 < int((e > i).sum()) < counts[i + 1] for i in range(N - 1)), (e, counts)   # riders ran
        if name == "riders" and not fused:
            assert 1 in counts.tolist()
        if name == "same":                          # every image at one boundary: the per-batch exit's result
            model.early_exit_per_image = False
            assert all(torch.equal(a, b) for a, b in zip(got, _eager(model, feats)))
        if name == "never":                         # never reached: the no-exit result
            model.early_exit_per_image = False
            model.early_exit_threshold = None
            assert all(torch.equal(a, b) for a, b in zip(got, _eager(model, feats)))
            assert counts.tolist() == [c.shape[0]] * N


def _graph_equals_eager(model, feats, settings):
    from boosted_detr_b200.graph import GraphedInference
    x0 = feats["features"]
    x1 = np.tanh(np.random.default_rng(11).standard_normal(x0.shape)).astype(np.float32) * \
        np.linspace(3.0, 0.25, x0.shape[0], dtype=np.float32)[:, None, None, None]
    model.early_exit_per_image = True
    model.early_exit_threshold, model.early_exit_min_blocks = settings[0]
    gi = GraphedInference(model, {"features": x0})
    assert gi.per_image and gi.bodies == (model.num_decoder_blocks - 1) * (x0.shape[0] - gi.k_min + 1) + 1

    def one(x, thr, mb, host=False):
        model.early_exit_threshold, model.early_exit_min_blocks = thr, mb
        ref = _eager(model, {"features": x})
        state = (model.last_exit_blocks.clone(), model.last_image_confidence.clone(), model.last_active_counts.clone(),
                 model.last_exit_block)
        got = gi({"features": x}, return_host=host)
        torch.cuda.synchronize()
        if host:
            assert all(np.array_equal(g, r.cpu().numpy()) for g, r in zip(got, ref)), (thr, mb)
        else:
            assert all(torch.equal(g, r) for g, r in zip(got, ref)), (thr, mb)
        assert torch.equal(gi.last_exit_blocks, state[0])
        assert np.array_equal(gi.last_image_confidence.numpy(), state[1].numpy(), equal_nan=True)
        assert torch.equal(gi.last_active_counts, state[2])
        assert gi.last_exit_block == state[3]

    for thr, mb in settings:                        # thresholds and min_blocks change between replays, no recapture
        for x in (x0, x1, x0):
            one(x, thr, mb)
    junk = [torch.full((64, 1024, 1024), float(k), device="cuda") for k in range(4)]
    torch.cuda.synchronize()
    for x in (x0, x1):
        one(x, *settings[0], host=True)
    del junk
    return gi


@pytest.mark.parametrize("shape", ["tf32_config2", "fp16"])
def test_graph_per_image_equals_eager(mode, shape):
    model, feats, fused, k_min = _make(mode, shape)
    N = model.num_decoder_blocks
    P, c = _reference(model, feats)
    cases = _cases(c, N, k_min, require_spread=shape == "tf32_config2")
    settings = [cases["spread"], cases["riders"], cases["same"], cases["never"], (0.0, N - 1), (float(np.median(c)), 2)]
    _graph_equals_eager(model, feats, settings)


def test_skipped_blocks_do_nothing(mode, monkeypatch):
    """Every image leaves at boundary 1: the gather buffers only boundary 1 onwards would write stay NaN."""
    from boosted_detr_b200.boosted_model import BoostedDETR
    from boosted_detr_b200.graph import GraphedInference
    model, feats, _, _ = _make(mode, "tf32_reference")
    model.early_exit_per_image = True
    model.early_exit_threshold, model.early_exit_min_blocks = 0.0, 2
    seen = []
    begin = BoostedDETR._per_image_begin

    def nan_begin(self, f):
        st = begin(self, f)
        for t in (st["xp"][1], *st["cp"][1]):
            t.fill_(float("nan"))
        seen.append(st)
        return st
    monkeypatch.setattr(BoostedDETR, "_per_image_begin", nan_begin)
    eager = _eager(model, feats)
    assert model.last_exit_block == 1 and model.last_active_counts.tolist() == [8, 8, 0, 0]
    assert all(torch.isnan(t).all() for t in (seen[-1]["xp"][1], *seen[-1]["cp"][1]))
    monkeypatch.setattr(BoostedDETR, "_per_image_begin", begin)
    gi = GraphedInference(model, feats)
    st = gi._keep[1]
    for t in (st["xp"][1], *st["cp"][1]):
        t.fill_(float("nan"))
    got = gi(feats)
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(got, eager))
    assert gi.last_exit_block == 1 and gi.last_active_counts.tolist() == [8, 8, 0, 0]
    assert all(torch.isnan(t).all() for t in (st["xp"][1], *st["cp"][1]))


def test_refusals_and_training(mode):
    from boosted_detr_b200.graph import GraphedInference
    model, feats, _, _ = _make(mode, "tf32_reference")
    model.early_exit_threshold, model.early_exit_min_blocks = 0.5, 1
    model.early_exit_per_image = True
    gi = GraphedInference(model, feats)
    model.early_exit_per_image = False
    with pytest.raises(RuntimeError, match="early_exit_per_image"):
        gi(feats)
    gb = GraphedInference(model, feats)
    assert not gb.per_image
    model.early_exit_per_image = True
    with pytest.raises(RuntimeError, match="early_exit_per_image"):
        gb(feats)
    # training ignores the flag: same launches, same loss bits
    from boosted_detr_b200 import _lib
    lib = _lib.load()
    _, _, inputs = _model_and_data(N=4, B=8, rows=18, cols=18, Q=96)
    logs, launches = [], []
    for flag in (False, True):
        m, _, _ = _model_and_data(N=4, B=8, rows=18, cols=18, Q=96)
        m.early_exit_threshold, m.early_exit_per_image = 0.0, flag
        torch.cuda.synchronize()
        lib.bdetr_reset_launch_count()
        logs.append(m.train_step(inputs))
        launches.append(lib.bdetr_launch_count())
        assert m.last_exit_blocks is None
    assert launches[0] == launches[1]
    assert logs[0] == logs[1]
