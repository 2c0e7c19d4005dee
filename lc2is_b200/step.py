"""One pre-allocated pass of the whole head hot path (what ``Engine.train_loop`` /
``eval_loop`` do around the head, engine.py:75-101 and :145-163), chained through the C ABI on
the current stream with no host synchronisation and no allocation inside the step:

    pack / count labels -> [DP: all-reduce n_valid] -> K0 proto_normalize -> K1 cosine_logits_fwd ->
    K2 upsample+CE fwd/bwd + K3 argmax/confusion matrix (one kernel at x16; the 'outputs' map of final.py:44) ->
    mean_scale -> K1b cosine_logits_bwd -> finalize_loss -> [DP: all-reduce gradient bucket, behind the next step]

Used by bench.py and usable as the data-parallel engine shim (SURVEY 8f-4).
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib, dp
from ._lib import BF16, F32, check, lib, ptr, stream_ptr


class _Block:
    """Everything ONE step accumulates into, in one flat buffer whose head is zeroed with a single fill:
        [ grad bucket: grad_t (C*D) | loss_sum as fp32 (1) | pad ] [ grad_low (B*C*h*w) ]
        [ scalars: double loss_sum | int64 n_valid | float gscale | float loss | pad ]
        [ logits-backward workspace: its accumulators (zeroed too: LC2IS_BWD_WS_ZEROED) | the rest ]
    HeadStep keeps TWO of them and alternates, so that the gradient-bucket all-reduce of step i can stay in flight
    while step i+1 zero-fills and fills the other one."""

    def __init__(self, B, C, D, h, w, dev):
        nb = C * D + 1
        nb_pad = (nb + 3) // 4 * 4
        ngl = B * C * h * w
        ngl_pad = (ngl + 3) // 4 * 4
        ws_off = (nb_pad + ngl_pad + 8 + 63) // 64 * 64                                  # 256-byte aligned
        ws_bytes = max(int(lib.lc2is_cosine_logits_bwd_workspace(B, h * w, D, 1, C)), 256)
        ws_zero = int(lib.lc2is_cosine_logits_bwd_workspace_zeroed(B, h * w, D, 1, C))
        self.acc32 = torch.zeros(ws_off + (ws_bytes + 3) // 4, dtype=torch.float32, device=dev)
        self.zero_fill = self.acc32[:ws_off + (ws_zero + 3) // 4]                         # zeroed as fp32: 16-byte stores
        self.bwd_ws = self.acc32[ws_off:]
        acc = self.acc32.view(torch.uint8)
        f32 = self.acc32[: nb_pad + ngl_pad]
        self.bucket = dp.GradBucket([(1, C, D), (1,)], dev, flat=f32[:nb])
        self.grad_t = self.bucket.views[0]
        self.grad_low = f32[nb_pad:nb_pad + ngl].view(B, C, h, w)
        o = 4 * (nb_pad + ngl_pad)
        # scalars: [0:8] double loss_sum | [8:16] int64 n_valid | [16:20] float gscale | [20:24] float loss
        self.scalars = acc[o:o + 32]
        self.loss_sum = self.scalars[0:8].view(torch.float64)
        self.n_valid = self.scalars[8:16].view(torch.int64)
        self.gscale = self.scalars[16:20].view(torch.float32)
        self.loss = self.scalars[20:24].view(torch.float32)


class _Join:
    """`wait()`: the current stream waits for what was enqueued on the exchange stream UP TO the creation of this object
    (an event recorded there) - not for collectives issued later on the same stream (no host sync)."""

    def __init__(self, stream):
        self.event = torch.cuda.Event()
        self.event.record(stream)

    def wait(self):
        torch.cuda.current_stream().wait_event(self.event)


class HeadStep:
    """Pre-allocated device-resident step.  Per call: loss / n_valid / grad_v / grad_t of the batch; the confusion
    matrix ACCUMULATES over calls (``reset_metrics()`` clears it, ``global_confmat()`` returns it summed over the
    ranks - integer sums commute, so an evaluation pass needs ONE int64 all-reduce at its end, SURVEY 8d config 3).

    Data-parallel order of a call (weak scaling, one process per GPU):
        [bucket all-reduce of the PREVIOUS call, async] -> zero-fill -> pack labels -> [n_valid all-reduce, async] ->
        K0 -> K1 -> K2+K3 -> [wait n_valid] -> K1b -> [wait the previous bucket; its loss]
    The valid-count all-reduce hides behind K0 / K1 / K2+K3 and the gradient-bucket all-reduce of call i behind the whole
    of call i+1 (two accumulator blocks alternate), so no collective is exposed inside a pass; ``flush()`` all-reduces the
    last call's bucket.  ``loss`` / ``n_valid`` / ``grad_t`` / ``grad_low`` are those of the most recent call and - with a
    process group - complete after ``flush()``.

    ``capture(v, t, labels)`` records one call into a CUDA graph (static input addresses; one graph per input set and
    accumulator block) and returns a callable that replays it: one cudaGraphLaunch instead of ~12 kernel launches and
    two collectives enqueued from Python."""

    def __init__(self, B: int, h: int, w: int, H: int, W: int, C: int, D: int = 512, ignore_index: int = 0,
                 logit_scale: float = 1.0, normalize: bool = True, backward: bool = True,
                 v_dtype=torch.bfloat16, device: Optional[torch.device] = None, distributed: bool = False,
                 extra_bucket_floats: int = 0) -> None:
        dev = device or torch.device("cuda", torch.cuda.current_device())
        self.B, self.h, self.w, self.H, self.W, self.C, self.D = B, h, w, H, W, C, D
        self.hw = h * w
        self.ignore_index, self.logit_scale, self.normalize, self.backward = ignore_index, logit_scale, normalize, backward
        self.v_dtype = v_dtype
        self.distributed = distributed and dp.is_dist()
        Cp = _lib.class_pad(C)
        M = B * self.hw
        e = lambda *s, dt=torch.float32: torch.empty(*s, dtype=dt, device=dev)
        self.t_hat = e(1, Cp, D, dt=torch.bfloat16)
        self.inv_t = e(1, C)
        # bf16 V + normalize: the row normalisation runs inside the logits GEMM and the backward takes the raw V
        # (lc2is_cosine_logits_fwd with d_v_hat = NULL, LC2IS_BWD_RAW_V) - no v_hat round trip
        self.fuse_norm = bool(normalize and v_dtype == torch.bfloat16)
        self.v_hat = None if self.fuse_norm else e(M, D, dt=torch.bfloat16)
        self.inv_v = e(M)
        self.logits = e(B, C, h, w)
        # the route the lc2is_step_* stages take for this geometry: packed labels + packed-label K2 / K3 (split), at x16
        # K2 and K3 as ONE kernel (fused, k23_rc_kernel)
        self.split = bool(lib.lc2is_ce_split_supported(h, w, H, W))
        self.labels_packed = e(B, H, W, dt=torch.uint16) if self.split else None
        self.fused = bool(self.split and lib.lc2is_ce_argmax_fused_supported(C, h, w, H, W))
        self.grad_v = e(B, self.hw, D, dt=torch.bfloat16)
        self._blocks = [_Block(B, C, D, h, w, dev), _Block(B, C, D, h, w, dev)]
        self._cur = 0
        # gradients of upstream parameters that ride in the same all-reduce (TextToPatch: BASELINE config 4's 2.93 MB
        # bucket): callers write them into `extra` before the next call / flush()
        self.extra = [torch.zeros(extra_bucket_floats, dtype=torch.float32, device=dev) for _ in range(2)] \
            if extra_bucket_floats else None
        self._pending = None           # block whose bucket has not been all-reduced yet (distributed only)
        # the exchange steps go through ncclAllReduce on a stream of their own, forked / joined with events: plain
        # stream-ordered launches that overlap the head kernels and can be captured into the step's CUDA graph
        # (a process group that is not NCCL: torch.distributed's collectives instead - not capturable on this stack)
        self.comm = None
        if self.distributed:
            from . import nccl
            self.comm = nccl.default_comm(dev)
        self._xs = torch.cuda.Stream(device=dev) if self.comm is not None else None
        self.confmat = torch.zeros(C, C, dtype=torch.int64, device=dev)        # this rank's counts, accumulated
        self._confmat_global = torch.zeros(C, C, dtype=torch.int64, device=dev) if self.distributed else None
        self.k2_events = None          # optional (start, stop) CUDA events around the K2 call
        self._open = None
        self.timers = None             # optional {name: [(start, stop) CUDA events]} per section (bench --kernel-times)

    # ---- the most recent call's results ---------------------------------------------------------------------
    @property
    def _blk(self) -> _Block:
        return self._blocks[self._cur]

    @property
    def loss(self) -> torch.Tensor:
        """Mean loss of the most recent call (data-parallel: over the GLOBAL batch, valid after flush())."""
        blk = self._blk
        if self.distributed:
            return (blk.bucket.views[1] / blk.n_valid).reshape(1)       # all-reduced loss sum / all-reduced count
        return blk.loss

    n_valid = property(lambda self: self._blk.n_valid)
    grad_t = property(lambda self: self._blk.grad_t)
    grad_low = property(lambda self: self._blk.grad_low)
    loss_sum = property(lambda self: self._blk.loss_sum)
    bucket = property(lambda self: self._blk.bucket)

    def _mark(self, name: str) -> None:
        """Close the running timed section and open `name` (None = just close).  No-op unless self.timers is a dict."""
        if self.timers is None:
            return
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        if self._open is not None:
            self.timers.setdefault(self._open[0], []).append((self._open[1], ev))
        self._open = (name, ev) if name is not None else None

    def reset_metrics(self) -> None:
        self.confmat.zero_()

    def global_confmat(self) -> torch.Tensor:
        """The accumulated confusion matrix summed over all ranks (ONE int64 all-reduce; bit-identical to the
        single-GPU matrix).  Without a process group: the local matrix."""
        if not self.distributed:
            return self.confmat
        self._confmat_global.copy_(self.confmat)
        if self.comm is not None:
            self.comm.all_reduce_(self._confmat_global)
        else:
            dp.allreduce_confmat_(self._confmat_global)
        return self._confmat_global

    def _allreduce_async(self, *tensors):
        """SUM all-reduce of the tensors, asynchronous to the current stream; -> objects with .wait()."""
        if self.comm is None:
            return [dp.allreduce_sum_async(t) for t in tensors]
        self._xs.wait_stream(torch.cuda.current_stream())
        if len(tensors) == 1:
            self.comm.all_reduce_(tensors[0], self._xs)
        else:
            self.comm.all_reduce_many_(tensors, self._xs)
        return [_Join(self._xs)]

    # ---- data-parallel exchange of a finished block ------------------------------------------------------------
    def _start_exchange(self, k: int):
        """All-reduce block k's gradient bucket (+ the upstream gradients riding with it) asynchronously."""
        if self.extra is not None:
            return self._allreduce_async(self._blocks[k].bucket.flat, self.extra[k])
        return self._allreduce_async(self._blocks[k].bucket.flat)

    def _finish_exchange(self, k: int, works) -> None:
        for wk in works:
            wk.wait()                                             # stream-level wait, no host sync

    def flush(self) -> None:
        """Complete the most recent call: all-reduce its gradient bucket (distributed only; enqueued, no host sync)."""
        if self._pending is not None:
            k, self._pending = self._pending, None
            self._finish_exchange(k, self._start_exchange(k))

    def capture(self, v: torch.Tensor, t: torch.Tensor, labels: torch.Tensor):
        """Record ``self(v, t, labels)`` for the NEXT accumulator block into CUDA graphs; returns ``replay()``.
        The tensors' addresses are baked in (refill them in place).  Graphs alternate blocks like eager calls do, so
        capture one per (input set, block) in the order they will be replayed and replay them in that order.

        Single GPU: the whole call is ONE graph.  Data-parallel: the kernels between the exchange steps are three graphs
        (labels | logits + CE/argmax | backward) and the two ncclAllReduce launches stay eager on the exchange stream -
        a single graph holding the NCCL nodes and their cross-stream edges took as long to LAUNCH as the step takes to run
        (0.37 ms of host time per replay against 0.004 ms for the kernel-only graph)."""
        assert self.timers is None and self.k2_events is None, "no event timers inside a captured step"
        k = self._cur ^ 1
        pending = self._pending
        side = torch.cuda.Stream()

        def record(fn):
            g = torch.cuda.CUDAGraph()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                with torch.cuda.graph(g, stream=side, capture_error_mode="thread_local"):
                    fn()
            torch.cuda.current_stream().wait_stream(side)
            return g
        if not self.distributed:
            graphs = [record(lambda: self._enqueue(v, t, labels, k, pending))]
        else:
            graphs = [record(lambda: self._part_labels(labels, k)), record(lambda: self._part_forward(v, t, labels, k)),
                      record(lambda: self._part_backward(v, labels, k))]
        # capturing does not execute: leave the bookkeeping as if the call had not happened
        nxt_pending = k if self.distributed else None

        def replay():
            assert self._cur == (k ^ 1) and self._pending == pending, "replay graphs in the order they were captured"
            if not self.distributed:
                graphs[0].replay()
            else:
                graphs[0].replay()
                w_valid = self._allreduce_async(self._blocks[k].n_valid)
                works_prev = self._start_exchange(pending) if pending is not None else None
                graphs[1].replay()
                for wk in w_valid:
                    wk.wait()
                graphs[2].replay()
                if works_prev is not None:
                    self._finish_exchange(pending, works_prev)
            self._cur, self._pending = k, nxt_pending
        replay.graphs = graphs
        replay.block = k
        # the graphs of a rotation are captured back to back: advance the bookkeeping so that the next capture
        # records the other block (and this block's pending exchange)
        self._cur, self._pending = k, nxt_pending
        return replay

    def __call__(self, v: torch.Tensor, t: torch.Tensor, labels: torch.Tensor) -> None:
        """v [B,hw,D] (bf16/fp32), t [C,D] fp32, labels [B,H,W] int64 - all on the device.  Enqueues everything on
        the current stream; no host synchronisation."""
        k = self._cur ^ 1
        self._enqueue(v, t, labels, k, self._pending)
        self._cur = k
        self._pending = k if self.distributed else None

    def _enqueue(self, v, t, labels, k: int, pending) -> None:
        # exchange stream: this call's valid count first (K1b needs it; 8 bytes), then the previous call's gradient bucket -
        # both run next to K0 / K1 and are done before the fused kernel has taken every SM's registers (an NCCL kernel
        # that is launched later than that only starts when the fused kernel ends, and is then exposed)
        self._part_labels(labels, k)
        w_valid = self._allreduce_async(self._blocks[k].n_valid) if self.distributed else None
        works_prev = self._start_exchange(pending) if pending is not None else None
        self._part_forward(v, t, labels, k)
        self._mark("K1b backward")
        if w_valid is not None:
            for wk in w_valid:
                wk.wait()                                         # stream-level wait, no host sync
        self._part_backward(v, labels, k)
        if works_prev is not None:
            self._finish_exchange(pending, works_prev)
        self._mark(None)

    def _part_labels(self, labels, k: int) -> None:
        """zero-fill of block k + everything that depends on the labels only (packing, valid count)."""
        B, C, h, w, H, W = self.B, self.C, self.h, self.w, self.H, self.W
        blk = self._blocks[k]
        self._mark("zero-fill")
        blk.zero_fill.zero_()                                    # bucket, grad_low, scalars, K1b accumulators: one fill
        glow = ptr(blk.grad_low) if self.backward else None
        self._mark("label prepass / count")
        # un-scaled gradients accumulate into grad_low on the split routes; 1/N_valid is applied by K1b, so the
        # valid-count all-reduce hides behind K0 / K1 / K2
        check(lib.lc2is_step_ce_labels(ptr(labels), B, C, h, w, H, W, self.ignore_index, ptr(self.labels_packed),
                                       ptr(blk.n_valid), glow, stream_ptr()), "step_ce_labels")

    def _fuse(self, v) -> bool:
        return self.fuse_norm and v.dtype == torch.bfloat16

    def _part_forward(self, v, t, labels, k: int) -> None:
        """K0 -> K1 -> K2 (+ K3 in the same kernel at x16)."""
        st = stream_ptr()
        B, hw, D, C, h, w, H, W = self.B, self.hw, self.D, self.C, self.h, self.w, self.H, self.W
        blk = self._blocks[k]
        glow = ptr(blk.grad_low) if self.backward else None
        self._mark("K0+K1 logits")
        check(lib.lc2is_proto_normalize(ptr(t), 1, C, D, int(self.normalize), ptr(self.t_hat), ptr(self.inv_t), st),
              "proto_normalize")
        fuse = self._fuse(v)
        if not fuse and self.v_hat is None:
            self.v_hat = torch.empty(B * hw, D, dtype=torch.bfloat16, device=v.device)
        check(lib.lc2is_cosine_logits_fwd(ptr(v), BF16 if v.dtype == torch.bfloat16 else F32, B, hw, D,
                                          ptr(self.t_hat), 1, C, int(self.normalize), self.logit_scale,
                                          None if fuse else ptr(self.v_hat), ptr(self.inv_v), ptr(self.logits), st),
              "cosine_logits_fwd")
        self._mark("K2 upsample+CE")
        if self.k2_events is not None:
            self.k2_events[0].record()
        check(lib.lc2is_step_ce(ptr(self.logits), ptr(labels), ptr(self.labels_packed), B, C, h, w, H, W,
                                self.ignore_index, ptr(blk.loss_sum), glow, ptr(self.confmat), st), "step_ce")
        if self.k2_events is not None:
            self.k2_events[1].record()

    def _part_backward(self, v, labels, k: int) -> None:
        """1 / N_valid -> K1b -> K3 (where it is a separate kernel) -> the loss."""
        st = stream_ptr()
        B, hw, D, C, h, w, H, W = self.B, self.hw, self.D, self.C, self.h, self.w, self.H, self.W
        blk = self._blocks[k]
        fuse = self._fuse(v)
        if self.distributed:
            check(lib.lc2is_mean_scale(ptr(blk.n_valid), 1.0, ptr(blk.gscale), st), "mean_scale")
        else:
            # single GPU: the loss sum is complete (K2 has run), so the loss leaves with the gradient scale in one launch
            check(lib.lc2is_mean_scale_finalize(ptr(blk.n_valid), 1.0, ptr(blk.gscale), ptr(blk.loss_sum), ptr(blk.loss), st),
                  "mean_scale_finalize")
        if self.backward:
            check(lib.lc2is_cosine_logits_bwd_ex(ptr(blk.grad_low), F32, ptr(self.logits),
                                                 ptr(v) if fuse else ptr(self.v_hat),
                                                 ptr(self.inv_v), ptr(self.t_hat), ptr(self.inv_t), B, hw, D, 1, C,
                                                 int(self.normalize), self.logit_scale, ptr(blk.gscale),
                                                 ptr(self.grad_v), BF16, ptr(blk.grad_t), ptr(blk.bwd_ws), st,
                                                 _lib.BWD_WS_ZEROED | (_lib.BWD_RAW_V if fuse else 0)),
                  "cosine_logits_bwd")
        self._mark("K3 argmax+confmat")
        check(lib.lc2is_step_argmax(ptr(self.logits), ptr(labels), ptr(self.labels_packed), B, C, h, w, H, W,
                                    ptr(self.confmat), st), "step_argmax")       # (nothing on the fused route)
        self._mark("finalize")
        if self.distributed:
            blk.bucket.views[1].copy_(blk.loss_sum)              # fp32 copy of the loss sum rides in the bucket


class HostStep:
    """The same pass through ``lc2is_head_step_host``: HOST (pinned) buffers in, host results out,
    H2D / D2H copies inside the call (bench.py's `e2e`).

    ``hs(v, t, labels)`` blocks until the results are in ``out_loss / out_n_valid / out_confmat``.
    ``hs.submit(v, t, labels)`` / ``hs.wait()`` keep up to ``depth`` steps in flight (each with its own
    workspace and output buffers), so the copy of the next batch overlaps the kernels of the previous one, like a
    prefetching data loader; ``wait()`` returns the oldest step's (loss, n_valid, confmat).  ``hs.prefetch(labels)``
    starts the host-side packing of the next batch's labels in the background (otherwise submit() packs them itself,
    blocking the caller for that long)."""

    class _Slot:
        def __init__(self, nbytes, B, H, W, C, dev, host_pack):
            self.ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            self.out_loss = torch.zeros(1, dtype=torch.float32).pin_memory()
            self.out_n_valid = torch.zeros(1, dtype=torch.int64).pin_memory()
            self.out_confmat = torch.zeros(C, C, dtype=torch.int64).pin_memory()
            self.event = None
            self.keep = None

    def __init__(self, B: int, h: int, w: int, H: int, W: int, C: int, D: int = 512, ignore_index: int = 0,
                 logit_scale: float = 1.0, backward: bool = True, device: Optional[torch.device] = None,
                 pipelined: bool = True, host_pack: bool = True, depth: int = 2,
                 raw_images: Optional[int] = None) -> None:
        dev = device or torch.device("cuda", torch.cuda.current_device())
        self.args = (B, h, w, D, C, H, W)
        self.ignore_index, self.logit_scale, self.backward = ignore_index, logit_scale, backward
        nbytes = int(lib.lc2is_head_step_workspace(B, h * w, D, C, H, W))
        # pinned scratch for the host-side int64 -> 1- / 2-byte narrowing of the labels (split geometries)
        self.host_pack = bool(host_pack and lib.lc2is_ce_split_supported(h, w, H, W) and C < 0x7fff)
        # raw_images: how many of the batch's LAST label maps cross PCIe as int64 (packed on the device) while the host
        # threads narrow the others; None = measure this host's packing rate and H2D rate once and balance the two
        # routes (0 on a host with enough cores; everything raw when the host threads are slower than the 8-byte copy)
        self.label_bytes = int(lib.lc2is_host_label_bytes(C)) if self.host_pack else 8
        self.calibration = None
        if not self.host_pack:
            self.n_raw = B
        elif raw_images is not None:
            self.n_raw = max(0, min(B, int(raw_images)))
        else:
            self.n_raw = self._calibrate_split(B, h * w, D, H, W, C, dev)
        if self.n_raw >= B:
            self.host_pack, self.label_bytes = False, 8
        self.slots = [HostStep._Slot(nbytes, B, H, W, C, dev, self.host_pack) for _ in range(max(1, depth))]
        # pinned scratch for the packed labels: one more than the steps in flight, so that the labels of the NEXT batch
        # can be packed (prefetch) while all slots are busy
        # (host form: 1 byte per label for C <= 254, else the packed uint16 form - lc2is_host_label_bytes)
        self._scratch = [torch.empty(B, H, W, self.label_bytes, dtype=torch.uint8).pin_memory()
                         for _ in range(len(self.slots) + 1)] if self.host_pack else []
        self._scr_next = 0
        self._prefetched = None                     # (labels data_ptr, scratch index, pack handle)
        self.copy_stream = torch.cuda.Stream(device=dev) if pipelined else None
        n_raw = self.n_raw if self.host_pack else B
        self.h2d_bytes = B * h * w * D * 2 + C * D * 4 + (B - n_raw) * H * W * self.label_bytes + n_raw * H * W * 8
        self.d2h_bytes = 4 + 8 + C * C * 8
        self._next, self._inflight = 0, []
        self._set_outputs(self.slots[0])

    def _calibrate_split(self, B, hw, D, H, W, C, dev) -> int:
        """Time one host packing pass over a batch of labels and one pinned H2D copy, then pick the number of raw
        images that minimises max(host packing time, copy time) of a step.  Ranks of a node calibrate together (each
        sees its share of the cores / DRAM / PCIe)."""
        import time
        import torch.distributed as dist
        lb = self.label_bytes
        # label buffers rotate over more than a last-level cache (the real maps come from DRAM); the copy has its own
        # source: lines the cores have just touched copy several times slower
        n_rot = max(1, min(4, (96 << 20) // (B * H * W * 8) + 1))
        labs = [torch.zeros(B, H, W, dtype=torch.int64).pin_memory() for _ in range(n_rot)]
        src = torch.zeros(B * H * W, dtype=torch.int64).pin_memory()
        out = torch.empty(B * H * W * lb, dtype=torch.uint8).pin_memory()
        d_buf = torch.empty(B * H * W, dtype=torch.int64, device=dev)
        if dist.is_available() and dist.is_initialized():
            dist.barrier()
        t_pack, t_copy = float("inf"), float("inf")
        for i in range(2 * n_rot):
            lab = labs[i % n_rot]
            t0 = time.perf_counter()
            check(lib.lc2is_pack_labels_host(ptr(lab), lab.numel(), C, self.ignore_index, ptr(out)), "lc2is_pack_labels_host")
            t_pack = min(t_pack, time.perf_counter() - t0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            d_buf.copy_(src, non_blocking=True)
            e1.record()
            e1.synchronize()
            t_copy = min(t_copy, e0.elapsed_time(e1) * 1e-3)
        bw = B * H * W * 8 / t_copy                                   # bytes / s
        best = self.pick_raw_images(B, B * hw * D * 2, H * W * lb, H * W * 8, 1.1 * t_pack / B, bw)
        self.calibration = {"pack_ms": t_pack * 1e3, "h2d_gbs": bw / 1e9, "n_raw": best, "threads": int(lib.lc2is_pack_threads())}
        return best

    @staticmethod
    def pick_raw_images(B: int, v_bytes: int, packed_img_bytes: int, raw_img_bytes: int, pack_s_per_img: float,
                        h2d_bytes_per_s: float) -> int:
        """How many of the B label maps should cross PCIe as int64: a step lasts max(host packing of the others, H2D copy
        of everything).  The model ignores the contention between the two routes, so stay all-packed (0) unless the
        gain is clear (> 10 %), and take the smallest split within 5 % of the optimum."""
        def step_time(r):
            copy_t = (v_bytes + (B - r) * packed_img_bytes + r * raw_img_bytes) / h2d_bytes_per_s
            return max(pack_s_per_img * (B - r), copy_t)
        t_opt = min(step_time(r) for r in range(B + 1))
        if step_time(0) <= 1.1 * t_opt:
            return 0
        return min(r for r in range(B + 1) if step_time(r) <= 1.05 * t_opt)

    def _set_outputs(self, s) -> None:
        self.out_loss, self.out_n_valid, self.out_confmat = s.out_loss, s.out_n_valid, s.out_confmat

    def _take_scratch(self, h_labels):
        """-> (scratch tensor | None, flags): LC2IS_STEP_LABELS_PREPACKED if `h_labels` were prefetched."""
        if not self.host_pack:
            return None, 0
        if self._prefetched is not None and self._prefetched[0] == h_labels.data_ptr():
            _, k, handle = self._prefetched
            self._prefetched = None
            check(lib.lc2is_pack_labels_host_end(handle), "lc2is_pack_labels_host_end")
            return self._scratch[k], 1                       # h_scratch holds the first B - n_raw label maps
        if self._prefetched is not None:                      # a prefetch for other labels: let it finish, drop it
            check(lib.lc2is_pack_labels_host_end(self._prefetched[2]), "lc2is_pack_labels_host_end")
            self._prefetched = None
        k = self._scr_next
        self._scr_next = (k + 1) % len(self._scratch)
        return self._scratch[k], 0

    def prefetch(self, h_labels: torch.Tensor) -> None:
        """Start packing the labels of the NEXT batch on the library's host threads (returns at once); the following
        submit() / call with the same tensor uses the packed copy.  A data loader's prefetch."""
        import ctypes
        if not self.host_pack or self._prefetched is not None:
            return
        B, h, w, D, C, H, W = self.args
        k = self._scr_next
        self._scr_next = (k + 1) % len(self._scratch)
        handle = ctypes.c_void_p()
        check(lib.lc2is_pack_labels_host_begin(ptr(h_labels), (B - self.n_raw) * H * W, C, self.ignore_index,
                                               ptr(self._scratch[k]), ctypes.byref(handle)), "lc2is_pack_labels_host_begin")
        self._prefetched = (h_labels.data_ptr(), k, handle)
        self._prefetch_keep = h_labels

    def _check_inputs(self, h_v, h_labels) -> None:
        assert h_v.dtype == torch.bfloat16 and not h_v.is_cuda and not h_labels.is_cuda

    def __call__(self, h_v: torch.Tensor, h_t: torch.Tensor, h_labels: torch.Tensor) -> None:
        B, h, w, D, C, H, W = self.args
        self._check_inputs(h_v, h_labels)
        assert not self._inflight, "wait() for the submitted steps first"
        s = self.slots[0]
        scratch, flags = self._take_scratch(h_labels)
        check(lib.lc2is_head_step_host(ptr(h_v), ptr(h_t), ptr(h_labels), B, h, w, D, C, H, W, self.ignore_index,
                                       self.logit_scale, int(self.backward), ptr(s.out_loss),
                                       ptr(s.out_n_valid), ptr(s.out_confmat), ptr(s.ws), stream_ptr(),
                                       self.copy_stream.cuda_stream if self.copy_stream is not None else None,
                                       ptr(scratch), self.n_raw if self.host_pack else 0, flags),
              "lc2is_head_step_host")
        self._set_outputs(s)

    def submit(self, h_v: torch.Tensor, h_t: torch.Tensor, h_labels: torch.Tensor) -> None:
        import ctypes
        B, h, w, D, C, H, W = self.args
        self._check_inputs(h_v, h_labels)
        assert self.copy_stream is not None, "submit() needs pipelined=True (a copy stream)"
        assert len(self._inflight) < len(self.slots), "all slots are in flight: wait() first"
        s = self.slots[self._next]
        self._next = (self._next + 1) % len(self.slots)
        ev = ctypes.c_void_p()
        scratch, flags = self._take_scratch(h_labels)
        check(lib.lc2is_head_step_host_submit(ptr(h_v), ptr(h_t), ptr(h_labels), B, h, w, D, C, H, W, self.ignore_index,
                                              self.logit_scale, int(self.backward), ptr(s.out_loss),
                                              ptr(s.out_n_valid), ptr(s.out_confmat), ptr(s.ws), stream_ptr(),
                                              self.copy_stream.cuda_stream, ptr(scratch),
                                              self.n_raw if self.host_pack else 0, flags, ctypes.byref(ev)),
              "lc2is_head_step_host_submit")
        s.event, s.keep = ev, (h_v, h_t, h_labels)          # host buffers must outlive the step
        self._inflight.append(s)

    def close(self) -> None:
        """Drain the steps in flight and a label prefetch that was never consumed (its worker threads write into this
        object's pinned scratch), so that the buffers can be freed."""
        if getattr(self, "_prefetched", None) is not None:
            handle = self._prefetched[2]
            self._prefetched = None
            check(lib.lc2is_pack_labels_host_end(handle), "lc2is_pack_labels_host_end")
        while getattr(self, "_inflight", None):
            self.wait()

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def wait(self):
        s = self._inflight.pop(0)
        check(lib.lc2is_head_step_host_wait(s.event), "lc2is_head_step_host_wait")
        s.event, s.keep = None, None
        self._set_outputs(s)
        return s.out_loss, s.out_n_valid, s.out_confmat
