"""GraphedInference (graph.py): BoostedDETR.call(training=False) as one graph launch, with the early exit decided on the
device by conditional graph nodes.  Every replay must equal the eager call bit for bit: predictions, and with an exit
threshold also `last_exit_block` and `last_image_confidence`."""
import numpy as np
import pytest
import torch

from test_dense_gpu import _model_and_data

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
def params(monkeypatch):
    """params(heads=None, C=None): every ModelParameters model gets that head count / C - 2 categories."""
    from boosted_detr_b200.parameters import ModelParameters

    def set_params(heads=None, C=None):
        if heads is not None:
            orig = ModelParameters.default_params

            def p(self, value=None):
                d = orig(self, value)
                d.update(num_encoder_heads=heads, num_decoder_heads=heads)
                return d
            monkeypatch.setattr(ModelParameters, "default_params", p)
        if C is not None:
            v = {"category": [f"cat_{i}" for i in range(C - 2)], "attribute": ["attr_0"]}
            monkeypatch.setattr(ModelParameters, "default_vocab", lambda self: v)
    return set_params


def _eager(model, inputs):
    out = [t.clone() for t in model.call(inputs, training=False)]
    torch.cuda.synchronize()
    return out


def _same(a, b):
    return all(torch.equal(x, y) for x, y in zip(a, b))


def _second_batch(x, seed=11):
    return np.tanh(np.random.default_rng(seed).standard_normal(x.shape)).astype(np.float32)


def _replays_equal_eager(model, key, x0):
    """Two batches replayed in turn (numpy, then a CUDA tensor, then a pinned tensor), then again after ~1 GB of
    unrelated allocations: every replay equals the eager call on the same batch."""
    from boosted_detr_b200.graph import GraphedInference
    x1 = _second_batch(x0)
    eager = [_eager(model, {key: x}) for x in (x0, x1)]
    gi = GraphedInference(model, {key: x0})
    feeds = [x0, torch.from_numpy(x1).cuda(), torch.from_numpy(x0).pin_memory(), x1]
    for k, x in enumerate(feeds):
        got = gi({key: x})
        torch.cuda.synchronize()
        assert _same(got, eager[k % 2]), f"replay {k}"
    junk = [torch.full((64, 1024, 1024), float(k), device="cuda") for k in range(4)]
    torch.cuda.synchronize()
    for k, x in enumerate((x0, x1)):
        got = gi({key: x}, return_host=True)
        assert all(np.array_equal(g, e.cpu().numpy()) for g, e in zip(got, eager[k])), f"after allocations, batch {k}"
    del junk
    assert gi.last_exit_block == model.num_decoder_blocks - 1
    return gi


def test_tf32_fused_config2_size(mode):
    mode("tf32")
    model, _, inputs = _model_and_data(N=6, B=4, rows=20, cols=20)
    assert model._use_fused(torch.empty(inputs["features"].shape))
    _replays_equal_eager(model, "features", inputs["features"])


def test_fp16_mode(mode):
    from boosted_detr_b200 import _lib
    mode("fp16")
    model, _, inputs = _model_and_data(N=2, B=4, rows=48, cols=40)
    assert _lib.load().bdetr_attention_f16_workspace_bytes(4, 8, 48 * 40, 48 * 40, 32) > 0
    _replays_equal_eager(model, "features", inputs["features"])


def test_fp32_layer_path(mode):
    mode("fp32")
    model, _, inputs = _model_and_data(N=2, B=2, rows=20, cols=20)
    assert not model._use_fused(torch.empty(inputs["features"].shape))
    _replays_equal_eager(model, "features", inputs["features"])


def test_four_heads(mode, params):
    mode("tf32")
    params(heads=4)
    model, _, inputs = _model_and_data(N=3, B=4, rows=20, cols=20)
    assert model.EncoderTransformerBlocks[0].num_attention_heads == 4
    _replays_equal_eager(model, "features", inputs["features"])


def test_c1205_column_slab_heads(mode, params):
    mode("tf32")
    params(C=1205)
    model, _, inputs = _model_and_data(N=2, B=4, rows=20, cols=20)
    assert model.num_categories == 1205
    _replays_equal_eager(model, "features", inputs["features"])


def test_backbone_neck(mode):
    from boosted_detr_b200.boosted_model import BoostedDETR
    from boosted_detr_b200.parameters import baseline_params
    mode("tf32")
    p = baseline_params(1)
    p.update(image_size=(12 * 32, 12 * 32))
    model = BoostedDETR(**p, seed=3, backbone_neck=True, backbone_channels=320).build()
    bf = np.random.default_rng(9).standard_normal((4, 12, 12, 320)).astype(np.float32)
    _replays_equal_eager(model, "backbone_features", bf)


# ---------------------------------------------------------------------------------------------------------------------
# Early exit on the device
@pytest.fixture()
def exit_model(mode):
    mode("tf32")
    model, _, inputs = _model_and_data(N=6, B=4, rows=20, cols=20)
    return model, {"features": inputs["features"]}


def _block_min_confidences(model, feats):
    """Float32 minimum image confidence after each boundary, from the eager early exit itself."""
    mins = []
    for k in range(model.num_decoder_blocks - 1):
        model.early_exit_threshold, model.early_exit_min_blocks = 0.0, k + 1
        _eager(model, feats)
        assert model.last_exit_block == k
        mins.append(np.float32(model.last_image_confidence.numpy().min()))
    return mins


def _expect_eager_bits(model, gi, feats):
    eager = _eager(model, feats)
    e_exit, e_conf = model.last_exit_block, model.last_image_confidence.clone()
    got = gi(feats)
    torch.cuda.synchronize()
    assert _same(got, eager)
    assert gi.last_exit_block == e_exit
    assert torch.equal(gi.last_image_confidence, e_conf)
    return e_exit


def test_early_exit_equals_eager(exit_model):
    from boosted_detr_b200.graph import GraphedInference
    model, feats = exit_model
    N = model.num_decoder_blocks
    mins = _block_min_confidences(model, feats)
    model.early_exit_threshold, model.early_exit_min_blocks = 2.0, 1
    gi = GraphedInference(model, feats)
    assert gi.segmented
    # never reached: every block runs
    assert _expect_eager_bits(model, gi, feats) == N - 1
    # always reached: exit after the minimum number of blocks
    for min_blocks in (1, 3):
        model.early_exit_threshold, model.early_exit_min_blocks = 0.0, min_blocks
        assert _expect_eager_bits(model, gi, feats) == min_blocks - 1
    # between two blocks' confidences
    order = sorted(set(float(m) for m in mins))
    assert len(order) >= 2, mins
    thr = 0.5 * (order[-2] + order[-1])
    model.early_exit_threshold, model.early_exit_min_blocks = thr, 1
    assert _expect_eager_bits(model, gi, feats) == next(i for i in range(N - 1) if mins[i] >= thr)
    # exactly a block's float32 minimum confidence: >= is inclusive
    k = int(np.argmax(mins))
    model.early_exit_threshold = float(mins[k])
    assert _expect_eager_bits(model, gi, feats) == k
    # a float64 threshold that is not a float32 value but rounds to that confidence
    thr64 = float(np.nextafter(np.float64(mins[k]), np.inf))
    assert thr64 != float(np.float32(thr64)) and np.float32(thr64) == mins[k]
    model.early_exit_threshold = thr64
    assert _expect_eager_bits(model, gi, feats) == k
    # and back to never reached on the same graph
    model.early_exit_threshold = 2.0
    assert _expect_eager_bits(model, gi, feats) == N - 1


def test_skipped_blocks_do_nothing(exit_model):
    from boosted_detr_b200.graph import GraphedInference
    model, feats = exit_model
    model.early_exit_threshold, model.early_exit_min_blocks = 0.0, 2
    gi = GraphedInference(model, feats)
    eager = _eager(model, feats)
    assert model.last_exit_block == 1
    for cums in gi._cums[2:]:
        for c in cums:
            c.fill_(float("nan"))
    got = gi(feats)
    torch.cuda.synchronize()
    assert gi.last_exit_block == 1 and _same(got, eager)
    for cums in gi._cums[2:]:
        for c in cums:
            assert torch.isnan(c).all()


@pytest.mark.parametrize("threshold", [None, 2.0])
def test_weights_can_be_swapped(exit_model, tmp_path, threshold):
    from boosted_detr_b200.graph import GraphedInference
    model, feats = exit_model
    other, _, _ = _model_and_data(N=6, B=4, rows=20, cols=20, seed=5)
    path = str(tmp_path / "other.npz")
    other.save_weights(path)
    model.early_exit_threshold, model.early_exit_min_blocks = threshold, 1
    gi = GraphedInference(model, feats)
    before = [t.clone() for t in gi(feats)]
    model.load_weights(path)
    eager = _eager(model, feats)
    assert not _same(before, eager)
    got = gi(feats)
    torch.cuda.synchronize()
    assert _same(got, eager)


def test_refusals(exit_model, mode):
    from boosted_detr_b200.graph import GraphedInference
    model, feats = exit_model
    gi = GraphedInference(model, feats)
    static = gi.static_in.clone()
    other = {"features": _second_batch(feats["features"])}
    with pytest.raises(ValueError, match="shape"):
        gi({"features": feats["features"][:, :10]})
    mode("fp32")
    with pytest.raises(RuntimeError, match="compute mode"):
        gi(other)
    mode("tf32")
    model.early_exit_threshold = 0.5
    with pytest.raises(RuntimeError, match="new GraphedInference"):
        gi(other)
    torch.cuda.synchronize()
    assert torch.equal(gi.static_in, static)
    gs = GraphedInference(model, feats)
    model.early_exit_threshold = None
    with pytest.raises(RuntimeError, match="new GraphedInference"):
        gs(other)


def test_early_exit_with_critical_stream(mode, monkeypatch):
    """BDETR_STREAM_PRIORITY=1 runs the encoder chain on a stream of its own: it is joined and forked again at every
    segment boundary like the others."""
    from boosted_detr_b200.graph import GraphedInference
    monkeypatch.setenv("BDETR_STREAM_PRIORITY", "1")
    mode("tf32")
    model, _, inputs = _model_and_data(N=3, B=4, rows=20, cols=20)
    feats = {"features": inputs["features"]}
    model.early_exit_threshold, model.early_exit_min_blocks = 2.0, 1
    gi = GraphedInference(model, feats)
    assert model._critical_stream() is not None
    assert _expect_eager_bits(model, gi, feats) == 2
    model.early_exit_threshold, model.early_exit_min_blocks = 0.0, 2
    assert _expect_eager_bits(model, gi, feats) == 1
