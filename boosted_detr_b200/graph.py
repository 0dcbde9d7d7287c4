"""CUDA-graph replay of the training step: the whole fwd + matcher + bwd chain is ~600 small kernels, so at
BASELINE config 2 the step is launch-bound; one graph launch replaces the Python/ctypes launch sequence.
GraphedInference does the same for BoostedDETR.call(training=False), with the early exit decided on the device."""
from __future__ import annotations

import ctypes
import time

import numpy as np
import torch

from . import _lib
from .device import empty, ptr, require_cuda, stream_ptr
from .losses_and_metrics import raise_for_status


class GraphedTrainStep:
    """Captures model.forward + backward for fixed shapes.  __call__(inputs) copies the batch into the static
    input buffers (H2D from pinned staging when given numpy), replays, and returns the metric tensors."""

    def __init__(self, model, example_inputs, warmup=3):
        self.model = model
        if model._flat is None:
            model.build()
        self.static = {}
        feats, y_true = model._prepare(example_inputs, True)
        self.static = {"features": feats.clone(), "category": y_true[0].clone(), "attribute": y_true[1].clone(),
                       "bbox": y_true[2].clone(), "num_objects": y_true[3].clone()}
        self.h2d_bytes = sum(t.numel() * t.element_size() for t in self.static.values())
        if model.optimizer is not None:
            model.optimizer.prepare(model)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self._step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        if getattr(model, "_trace", None) is not None:
            model._trace.clear()                   # keep only the marks of the captured step
        with torch.cuda.graph(self.graph):
            model._mark("step start (main)")
            self.metrics, self.status = self._step(capturing=True)
            model._mark("step end (main)")
        torch.cuda.synchronize()

    def _step(self, capturing=False):
        m = self.model
        s = self.static
        m.zero_grads()
        y_true = [s["category"], s["attribute"], s["bbox"], s["num_objects"]]
        _, ctx = m.forward(s["features"], y_true, True)
        metrics = m._collect_metrics(ctx)
        pipe = getattr(m, "bucket_pipeline", None)
        # the optimizer update belongs to the graph whenever the gradients are final inside it (single GPU, or the
        # bucketed all-reduce); its learning rate is read from device memory (see SGD.capture / pre_replay).  With a
        # bucket pipeline the update of block i's variables is queued right behind that block's all-reduce.
        self.optimizer_in_graph = m.optimizer is not None and (m.grad_allreduce is None or m.grad_bucket_hook is not None)
        self.optimizer_in_hook = bool(self.optimizer_in_graph and pipe is not None and pipe.bucket_optimizer and ctx.get("fused"))
        if self.optimizer_in_hook:
            pipe.opt_lr = (0.0, ptr(m.optimizer._lr_dev)) if capturing else None
        try:
            m.backward(ctx, gscale=1.0 / m.num_replicas)
        finally:
            if pipe is not None:
                pipe.opt_lr = None
        m._join_metrics()
        if m.grad_bucket_hook is not None and m.grad_allreduce is not None:
            m.grad_allreduce(m._flat[1])          # joins the bucketed all-reduces issued inside the backward (captured too)
        if self.optimizer_in_graph and capturing and not self.optimizer_in_hook:
            m.optimizer.capture(m)
        return metrics, m.status_all

    def load(self, inputs):
        """Host batch -> (pinned staging) -> static device buffers, async on the current stream."""
        m = self.model
        m.h2d_bytes = 0
        for k in ("features", "category", "attribute", "bbox", "num_objects"):
            x, dst = inputs[k], self.static[k]
            dtype = "i32" if k == "num_objects" else "f32"
            if isinstance(x, torch.Tensor) and x.is_cuda:
                if x.data_ptr() != dst.data_ptr():
                    dst.copy_(x.reshape(dst.shape), non_blocking=True)
            elif isinstance(x, torch.Tensor) and x.is_pinned() and x.dtype == dst.dtype and x.is_contiguous():
                dst.copy_(x.reshape(dst.shape), non_blocking=True)       # already in pinned host memory: no staging copy
                m.h2d_bytes += x.numel() * x.element_size()
            else:
                m._h2d(k, x, dtype, dst=dst)

    def _pre(self):
        """The per-step device words the captured kernels read (learning rate, dropout seed), queued on the current stream."""
        m = self.model
        if self.optimizer_in_graph:
            m.optimizer.pre_replay()
        m.push_dropout_seed()

    def replay(self):
        m = self.model
        if not getattr(self, "_primed", False):   # (already queued behind the previous launch by __call__(prefetch=...))
            self._pre()
        self._primed = False
        self.graph.replay()
        if m.grad_allreduce is not None and m.grad_bucket_hook is None:
            m.grad_allreduce(m._flat[1])          # non-overlapped mode: one all-reduce after the graph
        if m.optimizer is not None and not self.optimizer_in_graph:
            m.optimizer.apply(m)
        m.step_count += 1
        m.advance_dropout_seed()

    # -- input prefetch ---------------------------------------------------------------------------------------------
    def prefetch(self, inputs):
        """Starts the H2D copy of the NEXT batch into a second set of device buffers on a copy stream, so that it runs
        underneath the step that is executing; `__call__(inputs)` with the same object then only does device-to-device
        copies.  The caller keeps `inputs` (pinned host tensors) alive and unmodified until that call."""
        if not hasattr(self, "_staging"):
            self._staging = {k: torch.empty_like(v) for k, v in self.static.items()}
            self._copy_stream = torch.cuda.Stream()
            self._staged_ev, self._staging_free = torch.cuda.Event(), torch.cuda.Event()
            self._staging_free.record(torch.cuda.current_stream())
            self._staged_for = None
        cs = self._copy_stream
        cs.wait_event(self._staging_free)                 # the previous staging -> static copy has run
        with torch.cuda.stream(cs):
            for k, dst in self._staging.items():
                x = inputs[k]
                if not (isinstance(x, torch.Tensor) and (x.is_cuda or x.is_pinned())):
                    self.model._h2d(k, x, "i32" if k == "num_objects" else "f32", dst=dst)
                else:
                    dst.copy_(x.reshape(dst.shape), non_blocking=True)
            self._staged_ev.record(cs)
        self._staged_for = inputs

    def _take_prefetched(self):
        main = torch.cuda.current_stream()
        main.wait_event(self._staged_ev)
        for k, dst in self.static.items():
            dst.copy_(self._staging[k], non_blocking=True)
        self._staging_free.record(main)
        self._staged_for = None

    def __call__(self, inputs, return_host=True, prefetch=None):
        """One training step on `inputs`.  `prefetch` = the batch of the FOLLOWING step (optional): its H2D copy runs on a
        copy stream underneath this step, and everything else the next launch needs -- the staging -> static input copies
        and the next step's learning-rate / dropout-seed words -- is queued on the main stream right BEHIND this step's
        graph while the host would otherwise sit in the logs' synchronisation.  The next call then only launches the graph
        (the host-side issue of ~8 small copies, ~50 us, no longer sits between two steps)."""
        if getattr(self, "_primed_for", None) is inputs and inputs is not None:
            pass                                  # inputs and per-step words are already in place
        elif getattr(self, "_staged_for", None) is inputs and inputs is not None:
            self._take_prefetched()
        else:
            self.load(inputs)
        self._primed_for = None
        self.replay()
        if prefetch is not None:
            self.prefetch(prefetch)
            if self.optimizer_in_graph or self.model.optimizer is None:
                # stream order keeps this behind the running graph, which still reads the current batch and words
                self._take_prefetched()
                self._pre()
                self._primed, self._primed_for = True, prefetch
        if not return_host:
            return self.metrics
        return self.model.host_logs()


def _is_capturing(stream):
    with torch.cuda.stream(stream):
        return torch.cuda.is_current_stream_capturing()


class GraphedInference:
    """Captures BoostedDETR.call(training=False) for one input shape and compute mode.  `__call__(inputs)` copies
    `features` (or `backbone_features` for a model with a backbone neck) into a static input buffer, replays and returns
    the three running predictions [cat, attr, box].  Those tensors are static buffers: the next call overwrites them
    (clone them to keep a result).  Inputs may be CUDA tensors, pinned host tensors or numpy arrays (through the model's
    pinned staging), as in GraphedTrainStep.load.

    The capture shape is fixed by `model.early_exit_threshold` at construction:
      None      one graph around the forward, with its multi-stream schedule across blocks as is;
      a number  the forward captured in segments (S0 = prologue + block 0, Sk = block k + the device-side exit decision
                after it, E = the output select), stitched by the library into
                    S0 -> IF(h0){S1} -> IF(h1){S2} -> ... -> E
                so the blocks after the exit block do not run (include/bdetr.h "Graph-captured inference").  The threshold
                and `early_exit_min_blocks` live in device words: a change takes effect at the next call, without a new
                capture.  Switching between None and a number needs a new GraphedInference.
      a number, with `model.early_exit_per_image` (and N >= 2): the per-image exit, captured as
                    S0 -> SWITCH(h0){S1@k_min .. S1@B} -> ... -> SWITCH(h_{N-2}){S_{N-1}@k_min .. S_{N-1}@B}
                where Si@k is block i at batch k plus boundary i's plan and compaction (the final write-out in block
                N - 1); the plan of boundary i picks the body of block i + 1 that matches the images still running.
                Changing `early_exit_per_image` after the capture needs a new GraphedInference.
    `last_exit_block` and `last_image_confidence` (and in the per-image mode `last_exit_blocks` and `last_active_counts`)
    are read from the device on first access after a call and equal what the eager call leaves on the model
    (`last_image_confidence` is None when no block boundary was checked by the per-batch exit)."""

    def __init__(self, model, example_inputs, warmup=2):
        self.model = model
        if model._flat is None:
            model.build()
        lib = _lib.load()
        self.mode = lib.bdetr_get_mode()
        self.key = "backbone_features" if model.BackboneNeck is not None and "backbone_features" in example_inputs else "features"
        self.shape = tuple(example_inputs[self.key].shape)
        self.static_in = torch.empty(self.shape, dtype=torch.float32, device=require_cuda())
        self.segmented = model.early_exit_threshold is not None
        N, B, Q = model.num_decoder_blocks, self.shape[0], model.num_object_preds
        self.per_image_flag = bool(model.early_exit_per_image)
        self.per_image = self.segmented and self.per_image_flag and N >= 2
        self.load(example_inputs)
        self._exit_graph = None
        if self.segmented and not self.per_image:
            # device words the decide kernels read: threshold (float32), min_blocks, threshold set; the exit block; the
            # image confidences of every boundary
            self._thr_dev = torch.zeros(1, dtype=torch.float32, device=require_cuda())
            self._int_dev = torch.zeros(2, dtype=torch.int32, device=require_cuda())
            self._exit_dev = torch.full((1,), N - 1, dtype=torch.int32, device=require_cuda())
            self._conf_dev = torch.zeros(max(N - 1, 1), B, dtype=torch.float32, device=require_cuda())
            self._conf_q, self._iconf = empty(B, Q), empty(B)
            self._words = None
            self.out = [empty(B, Q, n) for n in (model.num_categories, model.num_attributes, 4)]
        saved_thr, saved_trace = model.early_exit_threshold, getattr(model, "_trace", None)
        model._trace = None                        # no timing-event nodes: a conditional body may not hold event nodes
        try:
            model.early_exit_threshold = None      # warm-up: every block, no host-side exit
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(warmup):
                    cums = self._forward()[0]
                if self.per_image:                 # every kernel of every body size runs once outside the capture
                    # with a threshold no image reaches, boundary 0 keeps all B slots in order, so block 1 may run at
                    # any k <= B (its plan reads the first k slots of boundary 0's order)
                    model.early_exit_threshold = 2.0
                    st = model._per_image_begin(model._prepare({self.key: self.static_in}, False)[0])
                    model._per_image_block(st, 0, B)
                    for k in range(st["k_min"], B + 1):
                        model._per_image_block(st, 1, k)
                    self.k_min = st["k_min"]
                    del st
                elif self.segmented:               # load the decide / select kernels outside the capture
                    self._cums = [cums] * N
                    if N > 1:
                        self._decide(0, cums, 0)
                    self._select()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            model.early_exit_threshold = saved_thr
            t0 = time.perf_counter()
            if self.per_image:
                self._capture_switch()
            elif self.segmented:
                self._capture_segments()
            else:
                self.graph = torch.cuda.CUDAGraph(keep_graph=True)
                with torch.cuda.graph(self.graph):
                    self.out, self._keep = self._forward()
            t1 = time.perf_counter()
            if self.segmented:
                segs = (ctypes.c_void_p * len(self._segs))(*[g.raw_cuda_graph() for g in self._segs])
                build = lib.bdetr_switch_graph_build if self.per_image else lib.bdetr_exit_graph_build
                _lib.check(build(self._exit_graph, segs, len(self._segs)))
            else:
                self.graph.instantiate()
            torch.cuda.synchronize()
            self.capture_seconds, self.instantiate_seconds = t1 - t0, time.perf_counter() - t1
        finally:
            model.early_exit_threshold, model._trace = saved_thr, saved_trace
            model._exit_capture = None
        self._host = None
        self._read = None

    def _forward(self):
        feats, _ = self.model._prepare({self.key: self.static_in}, False)
        cums, ctx = self.model.forward(feats, None, False)
        return cums, (feats, ctx)

    # -- segmented capture ------------------------------------------------------------------------------------------
    def _capture_segments(self):
        m = self.model
        lib = _lib.load()
        N = m.num_decoder_blocks
        handles = (ctypes.c_ulonglong * max(N - 1, 1))()
        g = ctypes.c_void_p()
        _lib.check(lib.bdetr_exit_graph_create(N - 1, ctypes.byref(g), handles))
        self._exit_graph, self._handles = g, list(handles)[:N - 1]
        self._pool = torch.cuda.graph_pool_handle()
        self._origin = torch.cuda.Stream()
        self._origin.wait_stream(torch.cuda.current_stream())
        self._segs, self._cums = [], []
        with torch.cuda.stream(self._origin):
            self._begin_segment()
            m._exit_capture = self
            try:
                cums, self._keep = self._forward()
            finally:
                m._exit_capture = None
            assert len(self._cums) == N and self._cums[-1] is cums
            self._segs[-1].capture_end()
            self._begin_segment()
            self._select()
            self._segs[-1].capture_end()

    def _capture_switch(self):
        """S0 = prologue + block 0 + boundary 0, then block i at every batch k_min .. B, one body each, into one pool:
        bodies of one SWITCH never run together and SWITCH i ends before SWITCH i + 1 begins, so memory a body frees
        may serve the bodies captured after it.  What later bodies read (the gather buffers, outputs, plan state,
        positional tables, hoisted self-attention) lives in the prologue's state, kept until close()."""
        m = self.model
        lib = _lib.load()
        N, B = m.num_decoder_blocks, self.shape[0]
        self._pool = torch.cuda.graph_pool_handle()
        self._origin = torch.cuda.Stream()
        self._origin.wait_stream(torch.cuda.current_stream())
        self._segs = []
        handles = (ctypes.c_ulonglong * (N - 1))()
        g = ctypes.c_void_p()
        _lib.check(lib.bdetr_switch_graph_create(N - 1, B - self.k_min + 1, ctypes.byref(g), handles))
        self._exit_graph, self._handles = g, list(handles)
        with torch.cuda.stream(self._origin):
            self._begin_segment()
            feats, _ = m._prepare({self.key: self.static_in}, False)
            st = m._per_image_begin(feats)
            m._per_image_block(st, 0, B, self._handles[0])
            self._segs[-1].capture_end()
            for i in range(1, N):
                for k in range(self.k_min, B + 1):
                    self._begin_segment()
                    m._per_image_block(st, i, k, self._handles[i] if i < N - 1 else 0)
                    self._segs[-1].capture_end()
        self.out, self._keep = st["out"], (feats, st)
        self.bodies = len(self._segs)

    def _begin_segment(self):
        g = torch.cuda.CUDAGraph(keep_graph=True)
        g.capture_begin(pool=self._pool)
        self._segs.append(g)

    def _decide(self, i, cums, handle):
        """Image confidences of boundary i, exactly as BoostedDETR._early_exit computes them, and the decision kernel."""
        N = self.model.num_decoder_blocks
        B, Q, C = cums[0].shape
        _lib.call("bdetr_inverse_tokenize", B, Q, C, cums[1].shape[-1], ptr(cums[0]), None, None, None, ptr(self._conf_q),
                  ptr(self._iconf), 1.0 / (i + 2), stream_ptr())
        _lib.call("bdetr_early_exit_decide", B, i, N, ptr(self._iconf), ptr(self._thr_dev), ptr(self._int_dev[0:1]),
                  ptr(self._int_dev[1:2]), handle, ptr(self._exit_dev), ptr(self._conf_dev[i]), stream_ptr())

    def _select(self):
        m = self.model
        B, Q = self.out[0].shape[:2]
        srcs = (ctypes.c_void_p * (3 * len(self._cums)))(*[c.data_ptr() for cums in self._cums for c in cums])
        _lib.call("bdetr_select_exit_predictions", len(self._cums), B, Q, m.num_categories, m.num_attributes, srcs,
                  ptr(self._exit_dev), ptr(self.out[0]), ptr(self.out[1]), ptr(self.out[2]), stream_ptr())

    def boundary(self, i, cums, streams):
        """Called by the forward after boosted block i (BoostedDETR._exit_boundary) while the segments are captured:
        queues the decision for block i + 1 on the stream that produced `cums`, joins every forked stream into the
        capture's origin stream, ends segment i and begins segment i + 1 there, and forks the same streams again."""
        self._cums.append(cums)
        if i + 1 >= self.model.num_decoder_blocks:
            return
        self._decide(i, cums, self._handles[i])
        origin, forked = self._origin, []
        for s in [torch.cuda.current_stream(), *streams]:
            if s != origin and s not in forked and _is_capturing(s):
                origin.wait_stream(s)
                forked.append(s)
        with torch.cuda.stream(origin):
            self._segs[-1].capture_end()
            self._begin_segment()
        for s in forked:
            s.wait_stream(origin)

    def _push_words(self):
        """Queues the exit settings on the current stream when they changed (fills, no host buffer involved).  Eager
        compares the float32 confidences with the threshold in float32: it is rounded to float32 once, here."""
        m = self.model
        words = (float(np.float32(m.early_exit_threshold)), int(m.early_exit_min_blocks))
        if words != self._words:
            self._thr_dev.fill_(words[0])
            self._int_dev[0:1].fill_(words[1])
            self._int_dev[1:2].fill_(1)
            self._words = words

    # -- calls ------------------------------------------------------------------------------------------------------
    def _check(self, inputs):
        m = self.model
        if self.key not in inputs:
            raise KeyError(f"GraphedInference was captured for inputs['{self.key}']")
        shape = tuple(inputs[self.key].shape)
        if shape != self.shape:
            raise ValueError(f"GraphedInference was captured for {self.key} of shape {self.shape}, got {shape}: "
                             "capture a new GraphedInference for this shape")
        mode = _lib.load().bdetr_get_mode()
        if mode != self.mode:
            raise RuntimeError(f"GraphedInference was captured in compute mode {self.mode}, the library is in mode {mode}: "
                               "capture a new GraphedInference in this mode")
        if (m.early_exit_threshold is not None) != self.segmented:
            raise RuntimeError("early_exit_threshold changed between None and a number since the capture: the early exit "
                               "needs a differently shaped graph, capture a new GraphedInference")
        if bool(m.early_exit_per_image) != self.per_image_flag:
            raise RuntimeError("early_exit_per_image changed since the capture: the per-image exit needs a differently "
                               "shaped graph, capture a new GraphedInference")

    def load(self, inputs):
        """Host or device input -> the static input buffer, async on the current stream."""
        x, dst = inputs[self.key], self.static_in
        m = self.model
        m.h2d_bytes = 0
        if isinstance(x, torch.Tensor) and x.is_cuda:
            if x.data_ptr() != dst.data_ptr():
                dst.copy_(x.reshape(dst.shape), non_blocking=True)
        elif isinstance(x, torch.Tensor) and x.is_pinned() and x.dtype == dst.dtype and x.is_contiguous():
            dst.copy_(x.reshape(dst.shape), non_blocking=True)
            m.h2d_bytes += x.numel() * x.element_size()
        else:
            m._h2d(self.key, x, "f32", dst=dst)

    def replay(self):
        if self.per_image:
            self.model._exit_words()
            _lib.check(_lib.load().bdetr_exit_graph_launch(self._exit_graph, stream_ptr()))
        elif self.segmented:
            self._push_words()
            _lib.check(_lib.load().bdetr_exit_graph_launch(self._exit_graph, stream_ptr()))
        else:
            self.graph.replay()
        self._read = None

    def __call__(self, inputs, return_host=False):
        self._check(inputs)
        self.load(inputs)
        self.replay()
        if not return_host:
            return self.out
        if self._host is None:
            self._host = [torch.empty(t.shape, dtype=t.dtype).pin_memory() for t in self.out]
        for h, t in zip(self._host, self.out):
            h.copy_(t, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return [h.numpy().copy() for h in self._host]

    def _exit_state(self):
        if self._read is None:
            m = self.model
            N = m.num_decoder_blocks
            if self.per_image:
                B = self.shape[0]
                h = self._keep[1]["state"][:1 + N + 2 * B].cpu()
                exits = h[1 + N:1 + N + B]
                self._read = (int(exits.max()), h[1 + N + B:].view(torch.float32), exits, h[1:1 + N])
            elif not self.segmented:
                self._read = (N - 1, None)
            else:
                e = int(self._exit_dev.item())
                # the boundaries eager checks: min_blocks - 1 .. N - 2, up to the exit
                last = e if e < N - 1 else N - 2
                conf = self._conf_dev[last].cpu() if last >= max(self._words[1] - 1, 0) else None
                self._read = (e, conf)
        return self._read

    @property
    def last_exit_block(self):
        return self._exit_state()[0]

    @property
    def last_image_confidence(self):
        return self._exit_state()[1]

    @property
    def last_exit_blocks(self):
        return self._exit_state()[2] if self.per_image else None

    @property
    def last_active_counts(self):
        return self._exit_state()[3] if self.per_image else None

    def close(self):
        if self._exit_graph is not None:
            _lib.check(_lib.load().bdetr_exit_graph_destroy(self._exit_graph))
            self._exit_graph = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
