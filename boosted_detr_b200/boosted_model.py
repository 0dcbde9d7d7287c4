"""BoostedDETR — the reference's ModelComponents/boosted_model.py hot loop (call :170-267) on sm_100a.

Scope (SURVEY.md §8): the model starts at the BackboneNeck output.  `inputs` is a dict with
  'features'    [B, rows, cols, encoder_dim]  fp32   (replaces 'image'; backbone is out of scope)
  'category'    [B, T, C] one-hot  fp32              (the reference's Tokenization output)
  'attribute'   [B, T, A] multi-hot fp32
  'bbox'        [B, T, 4] COCO x,y,w,h, padded with -10
  'num_objects' [B] or [B,1] int
Values may be numpy arrays (copied host->device through pinned staging) or CUDA tensors.
The Keras surface is kept: BoostedDETR(**params), call(inputs, training), compile(optimizer), fit(ds),
train_step / test_step (which, as in the reference :269-270, also trains), per-block layer lists with
`trainable` flags, get_config().
"""
from __future__ import annotations

import ctypes
import os
import re

import numpy as np
import torch

from . import _lib
from .device import empty, f32, i32, ptr, require_cuda, stream_ptr, zeros
from .layers import Layer, dropout_key, dropout_site_key
from .losses_and_metrics import MatchingLoss, PreparedTargets, raise_for_status
from .prediction_heads import (BoxPredictionHead, MultiClassPredictionHead, SingleClassPredictionHead, heads_backward_fused,
                               heads_forward_fused)
from .transformers import (DecoderBlock, DecoderBlock_NoSelfAttention, DecoderPrep, ImageEncoderAttention, accumulate,
                           batch_sum_into, fused_path, make_fold, pos_projection)

# dropout site ids, one per Keras Dropout instance: block i -> 8*i + k
SITE_ENC_ATTN, SITE_ENC_FFN, SITE_DEC_SELF, SITE_DEC_CROSS, SITE_DEC_FFN = 0, 1, 2, 3, 4
BACKBONE_STRIDE = 32   # EfficientNetB4 include_top=False (reference backbone.py:28-31)


class BoostedDETR:
    def __init__(self, num_object_preds, image_size, num_encoder_blocks, num_encoder_heads, encoder_dim,
                 num_decoder_blocks, num_decoder_heads, decoder_dim, num_panoptic_heads=1, panoptic_dim=32,
                 vocab_dict=None, classification_only=False, attribute_weight=1.0, name="DETR",
                 feature_shape=None, seed=0, backbone_neck=False, backbone_channels=1792, **kwargs):
        self.name = name
        self.use_intermediate_predictions = True
        self.num_object_preds = num_object_preds
        self.image_size = tuple(image_size)
        self.num_encoder_blocks = num_encoder_blocks      # ignored by the reference too (:86, quirk Q5)
        self.num_encoder_heads = num_encoder_heads
        self.encoder_dim = encoder_dim
        self.num_decoder_blocks = num_decoder_blocks
        self.num_decoder_heads = num_decoder_heads
        self.decoder_dim = decoder_dim
        self.num_panoptic_heads = num_panoptic_heads
        self.panoptic_dim = panoptic_dim
        self.vocab_dict = vocab_dict or {"category": [], "attribute": []}
        self.classification_only = classification_only
        # vocab sizes include <PAD> and <OOV> (reference tokenizers.py:32-33)
        self.num_categories = len(self.vocab_dict["category"]) + 2
        self.num_attributes = len(self.vocab_dict["attribute"]) + 2
        self.feature_shape = tuple(feature_shape) if feature_shape else (
            self.image_size[0] // BACKBONE_STRIDE, self.image_size[1] // BACKBONE_STRIDE)

        Layer._rng = np.random.default_rng(seed)
        # SURVEY 8f rank 2: with backbone_neck=True the model starts one step earlier, at the EfficientNet output
        # inputs['backbone_features'] [B, rows, cols, backbone_channels] (reference boosted_model.py:195-196)
        from .backbone import BackboneNeck
        self.BackboneNeck = BackboneNeck(encoder_dim, name="BackboneNeck") if backbone_neck else None
        self.backbone_channels = backbone_channels
        N = num_decoder_blocks
        self.EncoderTransformerBlocks = [ImageEncoderAttention(1, num_encoder_heads, name=f"ImageEncoderAttention_{i}")
                                         for i in range(N)]
        self.DecoderPrep = DecoderPrep(num_object_preds, decoder_dim, name="DecoderPrep")
        self.DecoderBlocks = [DecoderBlock_NoSelfAttention(num_decoder_heads, name="DecoderBlock_0")]
        self.DecoderBlocks += [DecoderBlock(num_decoder_heads, name=f"DecoderBlock_{i}") for i in range(1, N)]
        self.CategoryBlocks = [SingleClassPredictionHead(self.num_categories, decoder_dim, num_object_preds,
                                                         name=f"CategoryPredictionHead_{i}") for i in range(N)]
        self.AttributeBlocks = [MultiClassPredictionHead(self.num_attributes, decoder_dim, num_object_preds,
                                                         name=f"AttributePredictionHead_{i}") for i in range(N)]
        self.BoxBlocks = [BoxPredictionHead(decoder_dim, num_object_preds, name=f"BoxPredictionHead_{i}")
                          for i in range(N)]
        self.loss_fn = MatchingLoss(category_weight=None, box_weight=0.0 if classification_only else None,
                                    attribute_weight=attribute_weight, exist_weight=None, name="MatchingLoss")
        self.optimizer = None
        self.dropout_seed = None          # None: dropout off (parity runs); int: hash-mask dropout, rate .1
        # Inference early exit (the reference's TODO, README.md:9): stop after the first boosted block (>= min blocks)
        # at which EVERY image's least confident query reaches the threshold; None = run all blocks.
        self.early_exit_threshold = None
        self.early_exit_min_blocks = 1
        self.last_exit_block = None
        # Per-image early exit (opt-in, needs a threshold and N >= 2): each image leaves at its own first confident boundary
        # and the blocks after it run without it (`_forward_per_image`).  After such a call: last_exit_blocks int32 [B],
        # last_image_confidence [B] (at the exit boundary, or the last boundary checked; NaN if none was) and
        # last_active_counts int32 [N] (images that ran each block, riders included).
        self.early_exit_per_image = False
        self.last_exit_blocks = self.last_active_counts = None
        self._exit_capture = None         # set by graph.GraphedInference while it captures the forward in segments
        self.step_count = 0
        self.num_replicas = 1
        self.grad_allreduce = None        # set by parallel.DataParallel (joins / performs the gradient all-reduce)
        self.grad_bucket_hook = None      # set by parallel.DataParallel: hook(block, lo, hi, events) as soon as a block's gradients are final
        self._flat = None
        self.metrics_names = ["loss", "Category_Loss", "Attribute_Loss", "Box_Loss", "Existence_Loss", "IOU"]

    # -- structure -----------------------------------------------------------------------------
    def layers(self):
        neck = [self.BackboneNeck] if self.BackboneNeck is not None else []
        return [*neck, *self.EncoderTransformerBlocks, self.DecoderPrep, *self.DecoderBlocks, *self.CategoryBlocks,
                *self.AttributeBlocks, *self.BoxBlocks]

    def get_config(self):
        return {k: getattr(self, k) for k in ("num_object_preds", "image_size", "num_encoder_blocks", "num_encoder_heads",
                                              "encoder_dim", "num_decoder_blocks", "num_decoder_heads", "decoder_dim",
                                              "num_panoptic_heads", "panoptic_dim", "vocab_dict")}

    def named_weights(self):
        for layer in self.layers():
            yield from layer.named_weights()

    def build(self, batch_size=2):
        """Creates all weights by running one tiny inference call (Keras builds lazily the same way)."""
        R, Cc = self.feature_shape
        if self.BackboneNeck is not None:
            self.call({"backbone_features": zeros(batch_size, R, Cc, self.backbone_channels)}, training=False)
        else:
            self.call({"features": zeros(batch_size, R, Cc, self.encoder_dim)}, training=False)
        self._flatten()
        return self

    def _flatten(self):
        """Moves trainable weights / gradients into two flat buffers (one memset, one all-reduce).  The slots are laid
        out in the order the backward finishes them -- boosted block N-1 first, block 0 (plus the shared query
        parameter) last -- so each block is one contiguous bucket that data-parallel runs can all-reduce while the
        backward of the earlier blocks is still running (`_buckets`: (block, first float, one-past-last float))."""
        N = self.num_decoder_blocks

        def block_of(name):
            m = re.match(r"[A-Za-z]+_(\d+)/", name)
            return int(m.group(1)) if m else 0                # DecoderPrep (shared queries): final only after block 0

        # BDETR_SPLIT_RANGES=1: two ranges per block (decoder / heads part goes out under encoder i's backward, encoder part
        # after it) instead of one.  Measured equal within noise at N = 1 / 2 / 8 (2.660 vs 2.642 ms at N = 8: twice as many
        # latency-bound all-reduces), so one range per block is the default.
        split_ranges = os.environ.get("BDETR_SPLIT_RANGES", "0") == "1"

        def part_of(name):
            # inside a block: decoder / heads variables first (their gradients are final long before the encoder's: the
            # decoder-side chains run ahead), encoder variables -- and the shared queries, final only at the very end --
            # last, so a block's bucket splits into two contiguous sub-ranges that can be all-reduced separately
            return 1 if (not split_ranges or name.startswith(("ImageEncoderAttention_", "DecoderPrep"))) else 0

        named = [(n, o, k) for n, o, k in self.named_weights() if k not in o._non_trainable]
        named.sort(key=lambda nok: (-block_of(nok[0]), part_of(nok[0])))      # stable: keeps the layer order inside a part
        self._index, off = {}, 0
        self._buckets, cur, start = [], None, 0
        self._split = {}                                      # block -> first float of its encoder part
        for n, o, k in named:
            blk = block_of(n)
            if cur is None:
                cur = blk
            if blk != cur:
                self._buckets.append((cur, start, off))
                self._split.setdefault(cur, off)
                cur, start = blk, off
            if part_of(n) == 1:
                self._split.setdefault(blk, off)
            w = o._weights[k]
            self._index[n] = (off, w.numel(), tuple(w.shape))
            off += (w.numel() + 3) // 4 * 4               # keep every tensor 16-byte aligned
        self._buckets.append((cur, start, off))
        self._split.setdefault(cur, off)
        assert [b for b, _, _ in self._buckets] == list(range(N - 1, -1, -1)), self._buckets
        # the ranges the bucket pipeline works on (all-reduce + optimizer update each): decoder part, encoder part per block
        self._ranges = []
        for b, lo, hi in self._buckets:
            mid = self._split[b]
            self._ranges += [r for r in ((lo, mid), (mid, hi)) if r[1] > r[0]]
        flat_w, flat_g, flat_tc = zeros(off), zeros(off), zeros(off)
        for n, o, k in named:
            o0, cnt, shp = self._index[n]
            flat_w[o0:o0 + cnt].copy_(o._weights[k].reshape(-1))
            o._weights[k] = flat_w[o0:o0 + cnt].view(shp)
            o._grads[k] = flat_g[o0:o0 + cnt].view(shp)
            if k.endswith("/kernel") or k in ("positional_encoding", "init_decoder_features"):
                o._shadow[k] = flat_tc[o0:o0 + cnt].view(shp)     # tf32-rounded copy read by the tcgen05 GEMMs
        self._flat = (flat_w, flat_g)
        self._flat_tc = flat_tc
        for layer in self.layers():
            layer.invalidate()

    def tensor_core_mode(self):
        return _lib.tc_mode()

    def refresh_shadow(self):
        """tensor-core mode: re-round the Dense kernels into their tf32 shadows (one pass over the flat buffer)."""
        if self._flat is not None and self.tensor_core_mode():
            _lib.call("bdetr_round_tf32", self._flat[0].numel(), ptr(self._flat[0]), ptr(self._flat_tc), stream_ptr())

    def num_parameters(self, include_non_trainable=True):
        return sum(o._weights[k].numel() for _, o, k in self.named_weights()
                   if include_non_trainable or k not in o._non_trainable)

    def get_weights_dict(self):
        return {n: o._weights[k].detach().cpu().numpy().copy() for n, o, k in self.named_weights()}

    def set_weights_dict(self, d):
        for n, o, k in self.named_weights():
            if n in d:
                o._weights[k].copy_(torch.from_numpy(np.ascontiguousarray(d[n], np.float32)).to(o._weights[k].device))

    def save_weights(self, path, naming="keras"):
        """Keras `Model.save_weights` by variable name (checkpoint.py: .npz, layer-name or TF object-graph keys)."""
        from .checkpoint import save_weights
        return save_weights(self, path, naming)

    def load_weights(self, source, strict=True):
        """Keras `Model.load_weights` (reference notebook cell 26) from an exported checkpoint (checkpoint.py)."""
        from .checkpoint import load_weights
        if self._flat is None:
            self.build()
        return load_weights(self, source, strict)

    def get_grads_dict(self):
        return {n: o._grads[k].detach().cpu().numpy().copy() for n, o, k in self.named_weights() if k in o._grads}

    def zero_grads(self):
        if self._flat is not None:
            self._flat[1].zero_()
        else:
            for _, o, k in self.named_weights():
                if k in o._grads:
                    o._grads[k].zero_()

    # -- inputs --------------------------------------------------------------------------------
    def _h2d(self, name, x, dtype, dst=None):
        """host array -> pinned staging slot -> HBM, async on the current stream (counted in self.h2d_bytes).
        Each (name, shape) has TWO staging slots used alternately, and a slot is only rewritten after the event recorded
        behind its previous H2D copy has completed -- the host may run ahead of the device (no sync in the step), and a
        single slot could be overwritten with batch k+1 while the copy of batch k was still queued."""
        tdt = torch.int32 if dtype == "i32" else torch.float32
        if isinstance(x, torch.Tensor) and x.is_pinned() and x.dtype == tdt and x.is_contiguous():
            # caller-owned pinned memory: copied straight from it (no staging memcpy -- 82 MB per step at config 5); as
            # with any non_blocking copy the caller must not rewrite the buffer before the step's stream has passed it
            self.h2d_bytes += x.numel() * x.element_size()
            if dst is None:
                return x.to(require_cuda(), non_blocking=True)
            dst.copy_(x.reshape(dst.shape), non_blocking=True)
            return dst
        arr = x.numpy() if isinstance(x, torch.Tensor) else np.asarray(x)
        arr = np.ascontiguousarray(arr, dtype=np.int32 if dtype == "i32" else np.float32)
        stage = getattr(self, "_staging", None)
        if stage is None:
            stage = self._staging = {}
        key = (name, arr.shape)
        if key not in stage:
            stage[key] = {"buf": [torch.empty(arr.shape, dtype=tdt).pin_memory() for _ in range(2)],
                          "ev": [None, None], "next": 0}
        st = stage[key]
        slot = st["next"]
        st["next"] = slot ^ 1
        if st["ev"][slot] is not None:
            st["ev"][slot].synchronize()                       # the copy that last read this slot has run
        st["buf"][slot].numpy()[...] = arr
        self.h2d_bytes += arr.nbytes
        if dst is None:
            out = st["buf"][slot].to(require_cuda(), non_blocking=True)
        else:
            dst.copy_(st["buf"][slot].reshape(dst.shape), non_blocking=True)
            out = dst
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        st["ev"][slot] = ev
        return out

    def _to_device(self, name, x, dtype):
        """host array -> pinned staging -> HBM (async on the current stream); CUDA tensors pass through."""
        if isinstance(x, torch.Tensor) and x.is_cuda:
            return i32(x) if dtype == "i32" else f32(x)
        return self._h2d(name, x, dtype)

    def _prepare(self, inputs, training):
        self.h2d_bytes = 0
        self._neck_ctx = None
        if self.BackboneNeck is not None and "backbone_features" in inputs:
            bf = self._to_device("backbone_features", inputs["backbone_features"], "f32")
            feats, self._neck_ctx = self.BackboneNeck.forward([bf], training)
        else:
            feats = self._to_device("features", inputs["features"], "f32")
        y_true = None
        if training:
            y_true = [self._to_device("category", inputs["category"], "f32"),
                      self._to_device("attribute", inputs["attribute"], "f32"),
                      self._to_device("bbox", inputs["bbox"], "f32"),
                      self._to_device("num_objects", inputs["num_objects"], "i32").reshape(-1)]
        return feats, y_true

    def _keys(self, i):
        """Per-site halves of the dropout keys of boosted block i.  The step's seed lives in device memory
        (`_seed_dev`, refreshed by `push_dropout_seed` before every eager step / graph replay) and the kernels combine the
        two, so a captured graph draws new masks on every replay like Keras Dropout (reference transformers.py:135,147)."""
        if self.dropout_seed is None:
            return None
        k = lambda s: dropout_site_key(8 * i + s)
        return {"enc": [(k(SITE_ENC_ATTN), k(SITE_ENC_FFN))], "dec": (k(SITE_DEC_SELF), k(SITE_DEC_CROSS), k(SITE_DEC_FFN))}

    def push_dropout_seed(self):
        """Queues the 4-byte H2D copy of the current `dropout_seed` on the current stream (pinned 16-slot ring: the host
        may run a few steps ahead of the device)."""
        if self.dropout_seed is None:
            return
        if getattr(self, "_seed_dev", None) is None:
            self._seed_dev = torch.zeros(1, dtype=torch.int32, device=require_cuda())
            self._seed_host = torch.zeros(16, dtype=torch.int32).pin_memory()
            self._seed_slot = 0
        slot = self._seed_slot = (self._seed_slot + 1) % 16
        self._seed_host.numpy().view(np.uint32)[slot] = self.dropout_seed & 0xFFFFFFFF
        self._seed_dev.copy_(self._seed_host[slot:slot + 1], non_blocking=True)

    def advance_dropout_seed(self):
        if self.dropout_seed is not None:
            self.dropout_seed = (self.dropout_seed + 1) & 0xFFFFFFFF

    def _side_stream(self):
        if getattr(self, "_side", None) is None:
            self._side = torch.cuda.Stream()
        return self._side

    def _loss_streams(self, n):
        if not _lib.load().bdetr_get_concurrency():
            return [self._side_stream()] * n
        cur = getattr(self, "_loss_s", [])
        while len(cur) < n:
            cur.append(torch.cuda.Stream())
        self._loss_s = cur
        return cur[:n]

    def _block_streams(self, n, backward=False):
        """One side stream per boosted block (decoder / heads / matching of block i; their backward).  Backward: the
        chains are needed by the sequential encoder chain in the order N-1, N-2, ... -- their stream priorities follow
        that order (pending CTAs of a higher-priority kernel are placed first when SM slots free up)."""
        if not _lib.load().bdetr_get_concurrency():
            return [torch.cuda.current_stream()] * n
        key = "_blk_bw" if backward else "_blk_s"
        cur = getattr(self, key, [])
        use_prio = os.environ.get("BDETR_STREAM_PRIORITY", "0") == "1"
        while len(cur) < n:
            prio = 0
            if backward and use_prio:
                rank = n - 1 - len(cur)                       # 0 = needed first (block N-1)
                prio = min(-1, -4 + rank)                     # -4, -3, -2, -1, -1, ...
            cur.append(torch.cuda.Stream(priority=prio))
        setattr(self, key, cur)
        return cur[:n]

    def _critical_stream(self):
        """The sequential encoder chain runs on a highest-priority stream: it is the step's critical path, and its
        ~100-CTA kernels otherwise queue for SM slots behind the decoder / heads / matcher kernels of other blocks."""
        if not _lib.load().bdetr_get_concurrency() or os.environ.get("BDETR_STREAM_PRIORITY", "0") != "1":
            return None
        if getattr(self, "_crit", None) is None:
            self._crit = torch.cuda.Stream(priority=-5)
        return self._crit

    def _aux_streams(self):
        """Four extra streams: two for the attribute / box heads (the three heads of a block are independent
        chains of short kernels), one for the batch-invariant decoder self-attention, one for the decoder chain."""
        if not _lib.load().bdetr_get_concurrency():
            return [torch.cuda.current_stream()] * 4          # A/B switch: everything in order on one stream
        if getattr(self, "_aux", None) is None:
            self._aux = [torch.cuda.Stream() for _ in range(4)]
        return self._aux

    # -- timeline of one captured step (tests/trace_step.py): timing events that survive CUDA-graph capture -------
    def _mark(self, label, stream=None):
        tr = getattr(self, "_trace", None)
        if tr is None:
            return
        ev = torch.cuda.Event(enable_timing=True, external=True)
        ev.record(stream if stream is not None else torch.cuda.current_stream())
        tr.append((label, ev))

    # -- inference early exit ---------------------------------------------------------------------
    def _early_exit(self, i, cums):
        """True when inference may stop after boosted block i.  Confidence of a query = max class probability of the
        running prediction / (i + 2) (the running prediction after block i is a sum of i + 2 softmax vectors: block 0
        counts twice, quirk Q2); an image is confident when its least confident query is.  One 4*B-byte D2H + sync."""
        if self.early_exit_threshold is None or i + 1 < self.early_exit_min_blocks or i + 1 >= self.num_decoder_blocks:
            return False
        cat, attr = cums[0], cums[1]
        B, Q, C = cat.shape
        conf, iconf = empty(B, Q), empty(B)
        _lib.call("bdetr_inverse_tokenize", B, Q, C, attr.shape[-1], ptr(cat), None, None, None, ptr(conf), ptr(iconf),
                  1.0 / (i + 2), stream_ptr())
        if getattr(self, "_exit_host", None) is None or self._exit_host.numel() != B:
            self._exit_host = torch.empty(B, dtype=torch.float32).pin_memory()
        self._exit_host.copy_(iconf, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        self.last_image_confidence = self._exit_host.clone()
        return bool((self._exit_host >= self.early_exit_threshold).all())

    def _exit_boundary(self, i, cums, streams):
        """True when the inference forward stops after boosted block i (`_early_exit`).  While graph.GraphedInference
        captures the forward in segments, the decision is a captured kernel instead and every block is issued: it ends
        the current segment there, after joining `streams` (every stream the forward has forked), and begins the next."""
        if self._exit_capture is None:
            return self._early_exit(i, cums)
        self._exit_capture.boundary(i, cums, streams)
        return False

    # -- per-image early exit ---------------------------------------------------------------------
    def _exit_words(self):
        """Device words the plan kernel reads: threshold (float32; eager compares float32 confidences with it in float32),
        [min_blocks, threshold set].  Refilled on the current stream when the settings changed, never inside a capture."""
        if getattr(self, "_exit_dev", None) is None:
            self._exit_dev = (torch.zeros(1, dtype=torch.float32, device=require_cuda()),
                              torch.zeros(2, dtype=torch.int32, device=require_cuda()))
            self._exit_dev_words = None
        words = (float(np.float32(self.early_exit_threshold)), int(self.early_exit_min_blocks))
        if words != self._exit_dev_words and not torch.cuda.is_current_stream_capturing():
            self._exit_dev[0].fill_(words[0])
            self._exit_dev[1][0:1].fill_(words[1])
            self._exit_dev[1][1:2].fill_(1)
            self._exit_dev_words = words
        return self._exit_dev

    def _per_image_begin(self, feats):
        """Prologue of the per-image forward at the full batch B, and what it carries across the boundaries: the gather
        buffers of x and of the three running predictions (two sets, boundary i writes set i % 2), the outputs and the
        plan state.  The path chosen at B is kept for the whole call; on the fused path the batch never drops below
        k_min = the fewest images that fill one 128-row GEMM tile (`_use_fused`)."""
        B, R, Cc, D = feats.shape
        N, Q, C, A = self.num_decoder_blocks, self.num_object_preds, self.num_categories, self.num_attributes
        L = R * Cc
        if self._use_fused(feats):
            st = self._fused_prologue(feats, None, False, False, None, 0.0)
            st.update(fused=True, streams=[st["pre_s"], *st["bstreams"]], k_min=max(-(-128 // L), -(-128 // Q)))
        else:
            st = self._layer_prologue(feats, None, False)
            st.update(fused=False, streams=list(st["aux"]), k_min=1)
        nbytes = _lib.load().bdetr_image_exit_state_bytes(B, N)
        st.update(B=B, xp=[empty(B, R, Cc, D) for _ in range(2)], cp=[[empty(B, Q, n) for n in (C, A, 4)] for _ in range(2)],
                  out=[empty(B, Q, n) for n in (C, A, 4)], conf_q=empty(B, Q), iconf=empty(B), words=self._exit_words(),
                  state=torch.empty(nbytes // 4, dtype=torch.int32, device=feats.device))
        return st

    def _per_image_block(self, st, i, k, switch=0):
        """Block i at batch k (block 0: the prologue's input; later blocks: the first k rows of the gather buffers),
        every stream joined into the caller's, then boundary i: the image confidences of the k running slots, the plan
        (`switch` = the graph's SWITCH handle for block i + 1, 0 in eager calls) and the compaction.  After the last
        block the compaction writes every remaining image out instead."""
        N, B = self.num_decoder_blocks, st["B"]
        if i == 0:
            x, cums = st["x"], None
        else:
            x, cums = st["xp"][(i - 1) & 1][:k], [c[:k] for c in st["cp"][(i - 1) & 1]]
        main = st["main"]
        if st["fused"]:
            x, cums, _ = self._fused_block(st, i, x, cums)
            st["heads_ev"], st["pre_ev"] = None, [None] * N     # joined below: later blocks need no event of this one
        else:
            x, cums = self._layer_block(st, i, x, cums)
        capturing = torch.cuda.is_current_stream_capturing()
        for s in st["streams"]:
            with torch.cuda.stream(s):
                forked = not capturing or torch.cuda.is_current_stream_capturing()   # (a body forks only the streams it uses)
            if forked:
                main.wait_stream(s)
        st["blocks"].clear()                                 # no block context outlives its block
        _, Q, C = cums[0].shape
        A = cums[1].shape[-1]
        cin, out = _lib.PTR3(*[c.data_ptr() for c in cums]), _lib.PTR3(*[o.data_ptr() for o in st["out"]])
        state = ptr(st["state"])
        if i == N - 1:
            _lib.call("bdetr_image_exit_compact", B, N, i, k, Q, C, A, x[0].numel(), None, ctypes.byref(cin), None, None,
                      ctypes.byref(out), state, stream_ptr())
            return
        _lib.call("bdetr_inverse_tokenize", k, Q, C, A, ptr(cums[0]), None, None, None, ptr(st["conf_q"]), ptr(st["iconf"]),
                  1.0 / (i + 2), stream_ptr())
        thr, ints = st["words"]
        _lib.call("bdetr_image_exit_plan", B, N, st["k_min"], i, k, ptr(st["iconf"]), ptr(thr), ptr(ints[0:1]), ptr(ints[1:2]),
                  switch, state, stream_ptr())
        cout = _lib.PTR3(*[c.data_ptr() for c in st["cp"][i & 1]])
        _lib.call("bdetr_image_exit_compact", B, N, i, k, Q, C, A, x[0].numel(), ptr(x), ctypes.byref(cin),
                  ptr(st["xp"][i & 1]), ctypes.byref(cout), ctypes.byref(out), state, stream_ptr())

    def _forward_per_image(self, feats):
        """Inference with the per-image early exit.  After each boundary one small D2H of the plan's head words (the
        number of images that run the next block, the per-block counts, exit blocks and confidences) and one
        synchronisation -- the per-batch exit also syncs once per boundary -- then the next block is issued at that size."""
        N = self.num_decoder_blocks
        st = self._per_image_begin(feats)
        B = st["B"]
        head = 1 + N + 2 * B
        if getattr(self, "_pi_host", None) is None or self._pi_host.numel() != head:
            self._pi_host = torch.empty(head, dtype=torch.int32).pin_memory()
        k = B
        for i in range(N):
            self._per_image_block(st, i, k)
            self.last_exit_block = i
            if i == N - 1:
                break
            self._pi_host.copy_(st["state"][:head], non_blocking=True)
            torch.cuda.current_stream().synchronize()
            k = int(self._pi_host[0])
            if k == 0:
                break
        h = self._pi_host.clone()
        self.last_active_counts, self.last_exit_blocks = h[1:1 + N], h[1 + N:1 + N + B]
        self.last_image_confidence = h[1 + N + B:].view(torch.float32)
        return st["out"], {"blocks": [], "loss": [], "y_true": None}

    # -- fused tensor-core path -------------------------------------------------------------------
    def _use_fused(self, feats):
        """Tensor-core mode, model width 256, every layer already built (the very first call builds the layers lazily
        in the reference's execution order, which fixes the seeded initial weights -- it runs the layer-level path) and
        enough rows per GEMM for one 128-row tile."""
        if self._flat is None or not fused_path(self.encoder_dim) or self.decoder_dim != 256:
            return False
        B, R, Cc, _ = feats.shape
        return B * R * Cc >= 128 and B * self.num_object_preds >= 128 and os.environ.get("BDETR_FUSED", "1") == "1"

    def _forward_fused(self, feats, y_true, training):
        """Same hot loop as `forward` on the fused entry points (include/bdetr.h "Fused tensor-core path"):
            aux2   positional tables pos W + b of every block (batch-invariant) and the decoder self-attention of blocks
                   >= 1 hoisted out of the batch -- both depend on the weights only and run ahead of everything
            main   encoder i: grouped q/k/v projection -> attention -> out-proj+LN -> DenseRelu -> DenseLinear+LN
            dec    decoder i (q projection beside the grouped k/v projection -> attention -> out-proj+LN -> FFN),
                   the three heads in one call, then the matching of block i on its own stream"""
        N = self.num_decoder_blocks
        use_dropout = training and self.dropout_seed is not None
        if use_dropout and not torch.cuda.is_current_stream_capturing():
            self.push_dropout_seed()
        seed_dev = self._seed_dev if use_dropout else None
        rate = 0.1 if use_dropout else 0.0
        caller = torch.cuda.current_stream()
        crit = self._critical_stream()
        if crit is not None:
            crit.wait_stream(caller)
            with torch.cuda.stream(crit):
                out = self._forward_fused_on(feats, y_true, training, use_dropout, seed_dev, rate)
            caller.wait_stream(crit)
            return out
        return self._forward_fused_on(feats, y_true, training, use_dropout, seed_dev, rate)

    def _forward_fused_on(self, feats, y_true, training, use_dropout, seed_dev, rate):
        N = self.num_decoder_blocks
        st = self._fused_prologue(feats, y_true, training, use_dropout, seed_dev, rate)
        main, pre_s, bstreams = st["main"], st["pre_s"], st["bstreams"]
        x, cums = st["x"], None
        for i in range(N):
            x, cums, bs = self._fused_block(st, i, x, cums)
            with torch.cuda.stream(bs):
                self.last_exit_block = i
                if not training:
                    if self._exit_boundary(i, cums, [main, pre_s, *bstreams]):
                        break
                    if self._exit_capture is not None:
                        # a new graph segment has begun behind a join of every stream: events recorded in the previous
                        # segments cannot be waited on, and the join already orders everything after them
                        st["heads_ev"], st["pre_ev"] = None, [None] * N
        for bs in bstreams:
            main.wait_stream(bs)
        main.wait_stream(pre_s)
        if training:
            main.wait_stream(st["side"])
        self._mark("fwd joined (main)")
        return cums, {"blocks": st["blocks"], "loss": st["loss_ctxs"], "y_true": y_true, "fused": True}

    def _fused_prologue(self, feats, y_true, training, use_dropout, seed_dev, rate):
        """Everything of `_forward_fused_on` before block 0, at the full batch: the rounded input, the target digest, and
        the weight-only work (positional tables, tiled queries, hoisted decoder self-attention) on the aux2 stream."""
        N = self.num_decoder_blocks
        main = torch.cuda.current_stream()
        side = self._side_stream() if training else None
        aux = self._aux_streams()
        pre_s = aux[2]
        self.refresh_shadow()
        x = torch.empty_like(feats)                        # the block input feeds tcgen05 GEMMs: round it too
        _lib.call("bdetr_round_tf32", feats.numel(), ptr(feats), ptr(x), stream_ptr())
        B, R, Cc, D = feats.shape
        prepared = None
        if training:
            side.wait_stream(main)
            with torch.cuda.stream(side):
                prepared = PreparedTargets(y_true)
            for bs in self._block_streams(N):
                bs.wait_stream(side)
        # ---- weight-only work, ahead of the image-dependent chains ------------------------------------------------
        q0 = self.DecoderPrep._weights["init_decoder_features"]
        q0_tc = self.DecoderPrep._shadow.get("init_decoder_features", q0)
        pre_s.wait_stream(main)
        tabs, pre_self, pre_ev = [], [], []
        with torch.cuda.stream(pre_s):
            dec0 = self.DecoderPrep.tile_queries(B)         # block 0's decoder input: the tiled queries (:445-447)
            for i in range(N):
                enc, dec_l = self.EncoderTransformerBlocks[i], self.DecoderBlocks[i]
                for nm in ("SelfAttentionBlock", "JointAttentionBlock", "FeedForwardBlock"):
                    if hasattr(dec_l, nm):
                        getattr(dec_l, nm).rate = rate
                blk = enc.EncoderBlocks[0]
                blk.SelfAttentionBlock.rate = blk.FeedForwardBlock.rate = rate
                tabs.append(pos_projection(enc.pos_tc(), [(blk.SelfAttentionBlock.AttentionLayer, "QueryProjection"),
                                                          (blk.SelfAttentionBlock.AttentionLayer, "KeyProjection"),
                                                          (dec_l.JointAttentionBlock.AttentionLayer, "KeyProjection")]))
                keys = self._keys(i) if use_dropout else None
                if i >= 1:
                    pre_self.append(dec_l.SelfAttentionBlock.forward_hoisted(q0, q0_tc, B, training, keys["dec"][0] if keys else 0, seed_dev))
                else:
                    pre_self.append(None)
                ev = torch.cuda.Event()
                ev.record(pre_s)
                pre_ev.append(ev)
        # decoder i / heads i / matching i hang off encoder i's output only (plus the running prediction of block i-1):
        # every block gets its own side stream, so decoder i overlaps heads i-1 and the matchings
        return {"main": main, "side": side, "pre_s": pre_s, "bstreams": self._block_streams(N), "x": x, "B": B, "L": R * Cc,
                "D": D, "training": training, "use_dropout": use_dropout, "seed_dev": seed_dev, "y_true": y_true,
                "prepared": prepared, "tabs": tabs, "pre_self": pre_self, "pre_ev": pre_ev, "dec0": dec0, "heads_ev": None,
                "blocks": [], "loss_ctxs": []}

    def _fused_block(self, st, i, x, cums):
        """Boosted block i of the fused path on x [k, R, Cc, D] (k <= the prologue's batch: the tiled queries and the hoisted
        self-attention are the same for every image, so their first k rows serve).  Returns (encoder output, running
        predictions, the block's stream, on which they are final)."""
        training, use_dropout, seed_dev = st["training"], st["use_dropout"], st["seed_dev"]
        main, L, D = st["main"], st["L"], st["D"]
        k = x.shape[0]
        keys = self._keys(i) if use_dropout else None
        enc, dec_l = self.EncoderTransformerBlocks[i], self.DecoderBlocks[i]
        dkeys = keys["dec"] if keys else (0, 0, 0)
        if st["pre_ev"][i] is not None:
            main.wait_event(st["pre_ev"][i])
        (x, pos), c_enc = enc.forward([x], training, keys["enc"] if keys else None, seed_dev, tabs=st["tabs"][i][:2])
        self._mark(f"fwd enc{i} done (main)")
        bs = st["bstreams"][i]
        bs.wait_stream(main)
        with torch.cuda.stream(bs):
            fold = make_fold(pos=pos.view(L, D), tab_k=st["tabs"][i][2], pos_tc=enc.pos_tc())
            dec_in = st["dec0"] if i == 0 else st["pre_self"][i][0]
            if k != dec_in.shape[0]:
                dec_in = dec_in[:k]
            dec, c_dec = dec_l.forward_fused(x.view(k, L, D), fold, dec_in, training, dkeys, seed_dev)
            self._mark(f"fwd dec{i} done (dec)")
            mult = 2.0 if i == 0 else 1.0                 # block 0 is counted twice (reference :222-229)
            heads = (self.CategoryBlocks[i], self.AttributeBlocks[i], self.BoxBlocks[i])
            if st["heads_ev"] is not None:
                bs.wait_event(st["heads_ev"])             # the running prediction of block i-1
            cums, c_heads = heads_forward_fused(heads, dec, training, cums, mult)
            st["heads_ev"] = torch.cuda.Event()
            st["heads_ev"].record(bs)
            self._mark(f"fwd heads{i} done (dec)")
            st["blocks"].append({"enc": c_enc, "dec": c_dec, "self": None if i == 0 else st["pre_self"][i][1], "heads": c_heads,
                                 "dec0": st["dec0"]})
            if training:
                st["loss_ctxs"].append(self.loss_fn.forward(st["y_true"], cums, st["prepared"]))
                self._mark(f"fwd loss{i} done (side)")
        return x, cums, bs

    def _trainable_flags(self):
        N = self.num_decoder_blocks
        enc = [self.EncoderTransformerBlocks[i].trainable for i in range(N)]
        dec = [self.DecoderBlocks[i].trainable for i in range(N)]
        heads = [any(h[i].trainable for h in (self.CategoryBlocks, self.AttributeBlocks, self.BoxBlocks)) for i in range(N)]
        return enc, dec, heads, self.DecoderPrep.trainable

    def _backward_fused(self, ctx, gscale=1.0):
        caller = torch.cuda.current_stream()
        crit = self._critical_stream()
        if crit is not None:
            crit.wait_stream(caller)
            with torch.cuda.stream(crit):
                self._backward_fused_on(ctx, gscale)
            caller.wait_stream(crit)
            return None
        return self._backward_fused_on(ctx, gscale)

    def _backward_fused_on(self, ctx, gscale=1.0):
        """Backward of `_forward_fused`.  Work nothing trainable depends on is skipped (the reference's boosted
        training regime freezes whole blocks, Boosted_DETR_COCO.ipynb cell 30): no parameter gradients for frozen
        layers, no data gradients into blocks below the first trainable one."""
        lib = _lib.load()
        # parameter-gradient side chains are joined once per block (bdetr_join below), not inside every layer call
        lib.bdetr_set_deferred_join(1 if os.environ.get("BDETR_DEFER_JOIN", "1") == "1" else 0)
        try:
            return self._backward_fused_body(ctx, gscale)
        finally:
            lib.bdetr_set_deferred_join(0)

    def _backward_fused_body(self, ctx, gscale):
        N = self.num_decoder_blocks
        first = ctx["loss"][0]
        B, T, Q, C, A = first["dims"]
        enc_tr, dec_tr, heads_tr, prep_tr = self._trainable_flags()
        # does anything trainable sit at or below encoder i (on the chain x_0 -> enc_0 -> enc_1 -> ...)?
        below = [any(enc_tr[:i + 1]) for i in range(N)]
        neck_ctx = getattr(self, "_neck_ctx", None)
        neck_tr = neck_ctx is not None and self.BackboneNeck.trainable
        if neck_tr:
            below = [True] * N                      # the neck sits below every encoder block
        # Gradient of the running prediction of block i = sum of the loss gradients of blocks i .. N-1 (every later block's
        # prediction contains it).  The N loss backward kernels only need forward quantities, so they all run at once,
        # each into its own slice of one zeroed buffer, and one suffix-sum kernel turns the slices into the running
        # gradients; after that the heads / decoder backward of ALL blocks are independent chains (one stream each) --
        # only the encoder chain on the main stream is sequential.
        nC, nA, nB = B * Q * C, B * Q * A, B * Q * 4
        per = nC + nA + nB
        RG = zeros(N, per)
        r_of = lambda i: (RG[i, :nC].view(B, Q, C), RG[i, nC:nC + nA].view(B, Q, A), RG[i, nC + nA:].view(B, Q, 4))
        main = torch.cuda.current_stream()
        aux = self._aux_streams()
        pre_s = aux[2]
        bstreams = self._block_streams(N, backward=True)
        keep = [RG]
        pre_s.wait_stream(main)
        for i in range(N):
            bstreams[i].wait_stream(main)
            with torch.cuda.stream(bstreams[i]):
                self.loss_fn.backward(ctx["loss"][i], *r_of(i), gscale)
        for i in range(1, N):
            bstreams[0].wait_stream(bstreams[i])
        with torch.cuda.stream(bstreams[0]):
            _lib.call("bdetr_suffix_sum", N, per, ptr(RG), stream_ptr())
            self._mark("bwd loss gradients done (dec)")
        for i in range(1, N):
            bstreams[i].wait_stream(bstreams[0])
        g_q0 = self.DecoderPrep._grads["init_decoder_features"]
        d_encs, evs, self_evs, grad_evs = [None] * N, [None] * N, [None] * N, [None] * N

        def decoder_side(i):
            blk = ctx["blocks"][i]
            dec_l = self.DecoderBlocks[i]
            enc = self.EncoderTransformerBlocks[i]
            dec_s = bstreams[i]
            with torch.cuda.stream(dec_s):
                self_tr = i >= 1 and dec_l.SelfAttentionBlock.trainable
                need_d_dec = prep_tr or self_tr
                need_d_enc = below[i]
                need_dec = dec_tr[i] or need_d_dec or need_d_enc
                d_dec = None
                if heads_tr[i] or need_dec:
                    heads = (self.CategoryBlocks[i], self.AttributeBlocks[i], self.BoxBlocks[i])
                    d_dec = heads_backward_fused(heads, blk["heads"], list(r_of(i)), need_dx=need_dec)
                self._mark(f"bwd heads{i} done (dec)")
                d_dec_in = d_enc = None
                if need_dec:
                    L, D = blk["dec"]["joint"]["dims"][2], blk["dec"]["joint"]["dims"][3]
                    g_pos = enc._grads["positional_encoding"].view(L, D)
                    d_dec_in, d_enc = dec_l.backward_fused(blk["dec"], d_dec, d_pos=g_pos if enc.trainable else None,
                                                           need_d_dec=need_d_dec, need_d_enc=need_d_enc)
                ev = torch.cuda.Event()
                ev.record(dec_s)                                          # data gradients of block i's decoder side are final
                evs[i] = ev
                if d_dec_in is not None:
                    pre_s.wait_stream(dec_s)
                    with torch.cuda.stream(pre_s):                       # query-parameter side: queries only
                        if i == 0:
                            if prep_tr:
                                batch_sum_into(d_dec_in, g_q0)
                        else:
                            dec_l.SelfAttentionBlock.backward_hoisted(blk["self"], d_dec_in, g_q0 if prep_tr else None)
                            _lib.call("bdetr_join", stream_ptr())
                with torch.cuda.stream(pre_s):
                    sev = torch.cuda.Event()
                    sev.record(pre_s)
                self_evs[i] = sev
                _lib.call("bdetr_join", stream_ptr())                    # parameter gradients of decoder i / heads i
                gev = torch.cuda.Event()
                gev.record(dec_s)
                grad_evs[i] = gev
                d_encs[i] = d_enc
                self._mark(f"bwd dec{i} done (dec)")
                keep.extend([d_dec, d_dec_in, d_enc])

        decoder_side(N - 1)
        for i in reversed(range(N)):
            if i > 0:
                decoder_side(i - 1)          # enqueued before encoder i: encoder i accumulates its input gradient into d_enc[i-1]
            main.wait_event(evs[i])
            self._mark(f"bwd enc{i} may start (main)")
            if self.grad_bucket_hook is not None and self._flat is not None:
                # decoder / heads variables of block i are final once the decoder-side chain (grad_evs) and the hoisted
                # self-attention (self_evs) have passed: that sub-range goes out while encoder i's backward runs
                _, lo, hi = self._buckets[N - 1 - i]
                if self._split[i] > lo:
                    self.grad_bucket_hook(i, lo, self._split[i], [self_evs[i], grad_evs[i]])
            enc = self.EncoderTransformerBlocks[i]
            d_out = d_encs[i]                # gradient of encoder i's output: decoder i's k/v paths (+ encoder i+1, accumulated)
            if d_out is not None and (enc.trainable or (i > 0 and below[i - 1]) or (i == 0 and neck_tr)):
                Bf, L, D = d_out.shape
                R, Cc = self.feature_shape
                need_dx = (i > 0 and below[i - 1]) or (i == 0 and neck_tr)
                tgt = d_encs[i - 1] if (need_dx and i > 0) else None
                if tgt is not None:
                    main.wait_event(evs[i - 1])                       # d_enc[i-1] must exist before it is accumulated into
                d_x0 = enc.backward(ctx["blocks"][i]["enc"], d_out.view(Bf, R, Cc, D), d_x=None if tgt is None else tgt.view(Bf, R, Cc, D),
                                    acc=tgt is not None, need_dx=need_dx)
                if i == 0 and neck_tr:
                    self.BackboneNeck.backward(neck_ctx, d_x0)       # parameter gradients of the neck (the backbone is frozen)
                    keep.append(d_x0)
            self._mark(f"bwd enc{i} done (main)")
            if self.grad_bucket_hook is not None and self._flat is not None:
                _, lo, hi = self._buckets[N - 1 - i]
                hook_evs = [self_evs[i], grad_evs[i]]
                if i == 0:
                    hook_evs = [e for e in self_evs if e is not None] + [grad_evs[0]]
                # encoder i's parameter-gradient chains are joined INTO the consumer's stream (bucket pipeline), not into
                # this one: the encoder chain keeps running.  Only the encoder part of the bucket is left (its positional
                # table also collects decoder i's key-path gradient; block 0's part holds the shared queries).
                if hi > self._split[i]:
                    self.grad_bucket_hook(i, self._split[i], hi, hook_evs, join_from=torch.cuda.current_stream())
        _lib.call("bdetr_join", stream_ptr())
        for bs in bstreams:
            main.wait_stream(bs)
        main.wait_stream(pre_s)
        self._mark("bwd joined (main)")
        return None

    # -- forward -------------------------------------------------------------------------------
    def forward(self, feats, y_true, training):
        """The hot loop (reference :199-246).  Returns (y_pred, ctx).

        Scheduling.  Encoder block i+1 only needs encoder block i's output, while decoder i, the heads of block i
        and its matching loss hang off that output as a side chain.  The kernels are short and at most ~100 CTAs
        wide, so the step is latency-bound: the chains run on separate streams (captured as parallel branches
        of the CUDA graph):
            main     encoder 0 -> encoder 1 -> ... -> encoder N-1
            dec      (after encoder i) DecoderPrep -> decoder i -> heads i        [cums chain, in block order]
            aux0/1   attribute / box head of block i (forked from and joined into dec)
            aux2     decoder self-attention of block i >= 1 (queries only: no dependency on the image at all)
            side     cost matrix -> per-image assignment -> matched loss of block i (forked from dec)
        and everything is joined into main before returning."""
        if not training and self.early_exit_per_image and self.early_exit_threshold is not None and self.num_decoder_blocks >= 2:
            return self._forward_per_image(feats)
        if self._use_fused(feats):
            return self._forward_fused(feats, y_true, training)
        N = self.num_decoder_blocks
        st = self._layer_prologue(feats, y_true, training)
        main, aux, dec_s = st["main"], st["aux"], st["dec_s"]
        x, cums = st["x"], None
        for i in range(N):
            x, cums = self._layer_block(st, i, x, cums)
            with torch.cuda.stream(dec_s):
                self.last_exit_block = i
                if not training and self._exit_boundary(i, cums, [main, *aux]):
                    break
                if training:
                    ls = st["loss_streams"][i]
                    ls.wait_stream(dec_s)
                    with torch.cuda.stream(ls):
                        st["loss_ctxs"].append(self.loss_fn.forward(y_true, cums, st["prepared"]))
                        self._mark(f"fwd loss{i} done (side)")
        main.wait_stream(dec_s)
        main.wait_stream(aux[2])
        if training:
            main.wait_stream(st["side"])
            for ls in st["loss_streams"]:
                main.wait_stream(ls)
        self._mark("fwd joined (main)")
        return cums, {"blocks": st["blocks"], "loss": st["loss_ctxs"], "y_true": y_true}

    def _layer_prologue(self, feats, y_true, training):
        """Everything of the layer-level `forward` before block 0: the (rounded) input and the target digest."""
        N = self.num_decoder_blocks
        use_dropout = training and self.dropout_seed is not None
        if use_dropout and not torch.cuda.is_current_stream_capturing():
            self.push_dropout_seed()
        seed_dev = self._seed_dev if use_dropout else None
        x = feats
        main = torch.cuda.current_stream()
        side = self._side_stream() if training else None
        aux = self._aux_streams()
        if self.tensor_core_mode():
            self.refresh_shadow()
            x = torch.empty_like(feats)                        # the block input feeds tcgen05 GEMMs: round it too
            _lib.call("bdetr_round_tf32", feats.numel(), ptr(feats), ptr(x), stream_ptr())
        prepared, loss_streams = None, None
        if training:                                           # one target batch, N matchings: digest the targets once
            side.wait_stream(main)
            with torch.cuda.stream(side):
                prepared = PreparedTargets(y_true)
            # The matching of block i (cost -> per-image assignment -> matched loss) only depends on block i's running
            # prediction, and the sequential solver dominates it (~0.2 ms on near-tied early-training predictions), so
            # every block gets its own stream: the six matchings overlap instead of forming a 1.2 ms chain.
            loss_streams = self._loss_streams(N)
            for ls in loss_streams:
                ls.wait_stream(side)
        return {"main": main, "side": side, "aux": aux, "dec_s": aux[3], "x": x, "training": training, "use_dropout": use_dropout,
                "seed_dev": seed_dev, "prepared": prepared, "loss_streams": loss_streams, "blocks": [], "loss_ctxs": []}

    def _layer_block(self, st, i, x, cums):
        """Boosted block i of the layer-level path on x [k, R, Cc, D] (any k).  Returns (encoder output, running
        predictions), final on the dec stream."""
        training, use_dropout, seed_dev = st["training"], st["use_dropout"], st["seed_dev"]
        main, aux, dec_s = st["main"], st["aux"], st["dec_s"]
        keys = self._keys(i) if use_dropout else None
        enc = self.EncoderTransformerBlocks[i]
        for blk in enc.EncoderBlocks:
            blk.SelfAttentionBlock.rate = blk.FeedForwardBlock.rate = 0.1 if use_dropout else 0.0
        dec_l = self.DecoderBlocks[i]
        for nm in ("SelfAttentionBlock", "JointAttentionBlock", "FeedForwardBlock"):
            if hasattr(dec_l, nm):
                getattr(dec_l, nm).rate = 0.1 if use_dropout else 0.0
        dkeys = keys["dec"] if keys else (0, 0, 0)
        pre_self, dec0 = None, None
        # (not on the very first call: layers build lazily in execution order, and the weight-initialisation
        # order -- hence the seeded initial weights -- must not depend on this scheduling choice)
        if hasattr(dec_l, "SelfAttentionBlock") and dec_l.SelfAttentionBlock.built:
            aux[2].wait_stream(main)
            with torch.cuda.stream(aux[2]):
                dec0 = self.DecoderPrep.tile_queries(x.shape[0], like=x)
                pre_self = dec_l.SelfAttentionBlock.forward([dec0, dec0, dec0], training, dkeys[0], seed_dev)
        (x, pos), c_enc = enc.forward([x], training, keys["enc"] if keys else None, seed_dev)
        self._mark(f"fwd enc{i} done (main)")
        dec_s.wait_stream(main)
        with torch.cuda.stream(dec_s):
            prep_out, c_prep = self.DecoderPrep.forward([x, pos], training, dec=dec0)
            if pre_self is not None:
                dec_s.wait_stream(aux[2])
            dec, c_dec = dec_l.forward(list(prep_out), training, dkeys, pre_self=pre_self, seed_dev=seed_dev)
            self._mark(f"fwd dec{i} done (dec)")
            mult = 2.0 if i == 0 else 1.0                 # block 0 is counted twice (reference :222-229)
            if cums is not None and training:
                cums = [c.clone() for c in cums]          # each block's loss keeps its own running prediction
            heads = (self.CategoryBlocks[i], self.AttributeBlocks[i], self.BoxBlocks[i])
            c_heads, new_cums = [], []
            for h, head in enumerate(heads):              # three independent chains: one stream each
                st_h = dec_s if h == 0 else aux[h - 1]
                if st_h is not dec_s:
                    st_h.wait_stream(dec_s)
                with torch.cuda.stream(st_h):
                    _, c = head.forward([dec], training, cum=None if cums is None else cums[h], mult=mult)
                c_heads.append(c)
                new_cums.append(c["cum"])
            dec_s.wait_stream(aux[0])
            dec_s.wait_stream(aux[1])
            self._mark(f"fwd heads{i} done (dec)")
            st["blocks"].append({"enc": c_enc, "prep": c_prep, "dec": c_dec, "heads": c_heads})
        return x, new_cums

    def backward(self, ctx, gscale=1.0):
        """Gradient of gscale * sum_b sum_i total_b^(i) w.r.t. every trainable weight (accumulated).

        Same scheduling idea as forward: the loss / heads / decoder backward of ALL blocks only depends on the
        running prediction gradient, not on the encoder backward, so that chain runs ahead on the `dec` stream
        (heads on aux0/1, decoder self-attention backward on aux2) and hands (d_enc_value, d_enc_key) of block i
        to the encoder chain on the main stream through an event."""
        if ctx.get("fused"):
            return self._backward_fused(ctx, gscale)
        N = self.num_decoder_blocks
        first = ctx["loss"][0]
        B, T, Q, C, A = first["dims"]
        r_cat, r_attr, r_box = zeros(B, Q, C), zeros(B, Q, A), zeros(B, Q, 4)
        main = torch.cuda.current_stream()
        aux = self._aux_streams()
        dec_s = aux[3]
        keep = [r_cat, r_attr, r_box]            # buffers used on other streams stay alive until the final join
        dec_s.wait_stream(main)
        d_x_next = None
        # The two chains are ENQUEUED interleaved, block by block (decoder side of block i, then encoder i on main):
        # stream semantics do not care, but a captured graph is scheduled roughly in node-creation order, and with the
        # whole decoder-side chain created first the encoder chain of block N-1 sat idle behind it (measured: +0.5 ms).
        for i in reversed(range(N)):
            blk = ctx["blocks"][i]
            with torch.cuda.stream(dec_s):
                self.loss_fn.backward(ctx["loss"][i], r_cat, r_attr, r_box, gscale)
                self._mark(f"bwd loss{i} done (dec)")
                # the three heads are independent: category on this stream, attribute / box beside it
                aux[0].wait_stream(dec_s)
                aux[1].wait_stream(dec_s)
                d_dec = self.CategoryBlocks[i].backward(blk["heads"][0], r_cat)
                with torch.cuda.stream(aux[0]):
                    d_dec_a = self.AttributeBlocks[i].backward(blk["heads"][1], r_attr)
                with torch.cuda.stream(aux[1]):
                    d_dec_b = self.BoxBlocks[i].backward(blk["heads"][2], r_box)
                dec_s.wait_stream(aux[0])
                dec_s.wait_stream(aux[1])
                accumulate(d_dec_a, d_dec)
                accumulate(d_dec_b, d_dec)
                self._mark(f"bwd heads{i} done (dec)")
                # decoder: FFN + cross-attention here; the self-attention backward (queries only) and the
                # query-parameter gradient go to aux2
                d_ev, d_s, d_ek = self.DecoderBlocks[i].backward(blk["dec"], d_dec, defer_self=True)
                aux[2].wait_stream(dec_s)
                with torch.cuda.stream(aux[2]):
                    d_q = self.DecoderBlocks[i].backward_self(blk["dec"], d_s)
                    self.DecoderPrep.backward_queries(d_q)
                    self_ev = torch.cuda.Event()
                    self_ev.record(aux[2])
                ev = torch.cuda.Event()
                ev.record(dec_s)
                self._mark(f"bwd dec{i} done (dec)")
                keep += [d_dec, d_dec_a, d_dec_b, d_s, d_q, d_ev, d_ek]
            main.wait_event(ev)
            self._mark(f"bwd enc{i} may start (main)")
            if d_x_next is not None:
                accumulate(d_x_next.reshape(d_ev.shape), d_ev)
            enc = self.EncoderTransformerBlocks[i]
            L, D = d_ev.shape[1], d_ev.shape[2]
            g_pos = enc._grads["positional_encoding"].view(L, D)
            d_x4 = self.DecoderPrep.backward(blk["prep"], d_ev, None, d_ek, g_pos)
            d_x_next = enc.backward(blk["enc"], d_x4)
            self._mark(f"bwd enc{i} done (main)")
            if self.grad_bucket_hook is not None and self._flat is not None:
                # every gradient of boosted block i is final once this stream (encoder i, and through the hand-off
                # event decoder i / heads i) and the self-attention stream have passed this point: its bucket can be
                # all-reduced underneath the backward of blocks i-1 .. 0
                _, lo, hi = self._buckets[N - 1 - i]
                self.grad_bucket_hook(i, lo, hi, [self_ev])
        if getattr(self, "_neck_ctx", None) is not None and self.BackboneNeck.trainable and d_x_next is not None:
            self.BackboneNeck.backward(self._neck_ctx, d_x_next)
        main.wait_stream(dec_s)
        main.wait_stream(aux[2])
        self._mark("bwd joined (main)")
        return d_x_next

    # -- keras surface -------------------------------------------------------------------------
    def call(self, inputs, training=False):
        feats, y_true = self._prepare(inputs, training)
        y_pred, ctx = self.forward(feats, y_true, training)
        self.last_ctx = ctx
        if training:
            self._collect_metrics(ctx)
        return y_pred

    __call__ = call

    def _collect_metrics(self, ctx):
        """add_loss / add_metric bookkeeping (reference :250-260).  Runs on the matcher's side stream so that the
        backward does not wait for it; `_join_metrics` orders the caller's stream after it."""
        B = ctx["loss"][0]["dims"][0]
        main = torch.cuda.current_stream()
        side = self._side_stream() if _lib.load().bdetr_get_concurrency() else main
        side.wait_stream(main)
        with torch.cuda.stream(side):
            tot = zeros(5, B)
            for c in ctx["loss"]:
                accumulate(c["losses"], tot)
            iou = ctx["loss"][-1]["iou"]
            # one [6] vector of the Keras-style batch means and one status vector: a single small D2H each per step
            self.metric_means = torch.cat([tot.mean(dim=1), iou.mean().reshape(1)])
            self.status_all = torch.stack([c["status"] for c in ctx["loss"]]).reshape(-1)
        self.losses = [tot[0]]                                # add_loss(loss) (reference :250)
        self.metric_tensors = {"loss": tot[0], "Category_Loss": tot[1], "Attribute_Loss": tot[2], "Box_Loss": tot[3],
                               "Existence_Loss": tot[4], "IOU": iou.unsqueeze(0)}
        return self.metric_tensors

    def _join_metrics(self):
        if _lib.load().bdetr_get_concurrency():
            torch.cuda.current_stream().wait_stream(self._side_stream())

    def host_logs(self):
        """Metric means + matcher status to the host: two small pinned copies, one synchronisation."""
        if getattr(self, "_host_buf", None) is None or self._host_buf[1].numel() != self.status_all.numel():
            self._host_buf = (torch.empty(6, dtype=torch.float32).pin_memory(),
                              torch.empty(self.status_all.numel(), dtype=torch.int32).pin_memory())
        hm, hs = self._host_buf
        hm.copy_(self.metric_means, non_blocking=True)
        hs.copy_(self.status_all, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        raise_for_status(hs)
        return {k: float(hm[j]) for j, k in enumerate(self.metrics_names)}

    def compile(self, optimizer=None, **kwargs):
        self.optimizer = optimizer
        if optimizer is not None and self._flat is None:
            self.build()
        return self

    def train_step(self, inputs, return_host=True):
        if self._flat is None:
            self.build()
        feats, y_true = self._prepare(inputs, True)
        self.zero_grads()
        y_pred, ctx = self.forward(feats, y_true, True)
        self.last_ctx_train, self.last_preds = ctx, y_pred
        m = self._collect_metrics(ctx)
        pipe = getattr(self, "bucket_pipeline", None)
        in_hook = self.optimizer is not None and pipe is not None and pipe.bucket_optimizer and ctx.get("fused")
        if in_hook:                               # the update runs bucket by bucket behind each block's all-reduce
            self.optimizer._ensure_bucket_tables(self)
            pipe.opt_lr = (self.optimizer.current_lr(), None)
        try:
            self.backward(ctx, gscale=1.0 / self.num_replicas)
        finally:
            if pipe is not None:
                lr_used, pipe.opt_lr = pipe.opt_lr, None
        self._join_metrics()
        if self.grad_allreduce is not None:
            self.grad_allreduce(self._flat[1])
        if in_hook:
            self.optimizer.finish_step(lr_used[0])
        elif self.optimizer is not None:
            self.optimizer.apply(self)
        self.step_count += 1
        self.advance_dropout_seed()
        if not return_host:
            return m
        return self.host_logs()

    def test_step(self, inputs):
        return self.train_step(inputs)          # reference :269-270 (quirk Q8: validation also trains)

    def fit(self, dataset, epochs=1, steps_per_epoch=None, verbose=0, **kwargs):
        history = {k: [] for k in self.metrics_names}
        for _ in range(epochs):
            sums, n = {k: 0.0 for k in self.metrics_names}, 0
            for step, batch in enumerate(dataset):
                if steps_per_epoch is not None and step >= steps_per_epoch:
                    break
                logs = self.train_step(batch)
                for k in sums:
                    sums[k] += logs[k]
                n += 1
                if verbose:
                    print(f"step {step}: " + " ".join(f"{k}={v:.4f}" for k, v in logs.items()))
            for k in sums:
                history[k].append(sums[k] / max(n, 1))
        return history

    def predict_indices(self, inputs):
        """Numeric half of InverseTokenization (reference tokenizers.py:130-135) on the device: (category tokens [B,Q,1],
        attribute tokens [B,Q,A] = multi-hot * arange(A), boxes)."""
        from .tokenizers import InverseTokenization
        cat, attr, box = self.call(inputs, training=False)
        tok_c, tok_a = InverseTokenization(self.vocab_dict).tokens([cat, attr])
        return tok_c, tok_a, box
