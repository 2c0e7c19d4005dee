#!/usr/bin/env python
"""bench.py - the head hot path on N B200s (one process per GPU; torchrun for N > 1).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle)

A "step" is one pass of the hot path over one synthetic batch (BASELINE.json configs[1]):
B=16 images per GPU at 512^2, D=512, C=150, bf16 GEMM operands / fp32 accumulate:
cosine logits (K0+K1) -> fused bilinear-upsample + softmax-CE fwd/bwd (K2) -> logits backward
(K1b) -> argmax / confusion matrix / mIoU (K3); with N > 1 the valid-pixel count and the head-gradient bucket are
all-reduced over NCCL every step (the bucket behind the next step) and the int64 confusion matrix once per pass
(weak scaling).  After the timed primary step short secondary legs measure BASELINE configs 3, 4, 5 and the x4
geometry (`secondary` in the JSON line).  Prints ONE JSON line (rank 0).

    python bench.py --dump-outputs DIR ...   # also write what the last timed step computed (rank 0) as DIR/<name>.npy

The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "ADE20K-shape 512^2 images/sec (logits+loss+mIoU)"
UNIT = "images/s"
GEOM = {"A": (32, 32, 512), "B": (128, 128, 512), "5": (64, 64, 1024)}   # (h, w, H = W): SURVEY 8 G-A aux head x16,
#                                   G-B main head x4; "5" = BASELINE config 5 (1024^2, use --classes 847 --batch 8)
L2_BYTES = 126 * 1024 * 1024
DUMP_BYTES = 60 * 10 ** 6          # --dump-outputs: array data of all files together, so that they stay under 64 MB


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=None)
    p.add_argument("--warmup", type=int, default=None)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--geometry", default="A", choices=list(GEOM))
    p.add_argument("--batch", type=int, default=16, help="images per GPU")
    p.add_argument("--classes", type=int, default=150)
    p.add_argument("--no-backward", action="store_true")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--kernel-times", action="store_true", help="extra pass: per-section CUDA-event times (not the timed run)")
    p.add_argument("--no-graph", action="store_true", help="time eager launches instead of CUDA-graph replays")
    p.add_argument("--no-secondary", action="store_true", help="skip the cfg3 / G-B / cfg4 / cfg5 legs")
    p.add_argument("--legs", default="cfg3_eval,G-B,cfg4,cfg5", help="comma-separated secondary legs to run")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write the outputs of the last timed step (loss, n_valid, logits, grad_v, grad_t) and the pass's "
                        "confusion matrix as DIR/<name>.npy (float32 / float64)")
    a = p.parse_args()
    if a.steps is not None and a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        p.error("--dump-outputs writes the outputs of --impl b200")
    return a


def write_outputs(arrays, out_dir, budget=DUMP_BYTES, seed=0):
    """Write every tensor of `arrays` (name -> tensor) as out_dir/<name>.npy: floating point as float32, integers as
    float64 (exact below 2**53).  Smallest first, each array gets an equal share of what is left of `budget` bytes; an
    array larger than its share is written as a seeded sample of its flattened elements (sorted positions, the same
    for the same shape on every run)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    items = sorted(arrays.items(), key=lambda kv: kv[1].numel())
    left = budget
    for i, (name, t) in enumerate(items):
        t = t.detach().cpu()
        t = t.float() if t.is_floating_point() else t.double()
        share = left // (len(items) - i)
        if t.numel() * t.element_size() > share:
            g = torch.Generator().manual_seed(seed)
            idx = torch.randint(t.numel(), (share // t.element_size(),), generator=g).unique()
            t = t.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())
        left -= t.numel() * t.element_size()


def workload_name(a, h, w):
    H = GEOM[a.geometry][2]
    return (f"cfg{'5' if a.geometry == '5' else '2'}: text_patch logits + fused upsample/softmax-CE fwd/bwd + argmax/confmat mIoU, "
            f"B={a.batch}/GPU, {h}x{w}->{H}x{H} (x{H // h}), D=512, C={a.classes}, ignore_index=0")


# --------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Polls NVML (SM clock, throttle reasons) while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.002)

    def result(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:  # noqa: BLE001
            return local_rank
    return local_rank


# --------------------------------------------------------------------------------------------
def cpu_reference_time(B, h, w, C, steps, warmup, threads=None):
    """Times oracle.head_step (the reference's lines on CPU, fp32) on a B-image sample."""
    import torch
    from lc2is_b200 import synthetic
    from oracle import head_oracle as O
    if threads:
        torch.set_num_threads(threads)
    v = synthetic.make_patch_embeddings(B, h * w, 512, dtype=torch.float32)
    t = synthetic.make_prototypes(C, 512)
    labels = synthetic.make_labels(B, 512, 512, C)
    for _ in range(warmup):
        O.head_step(v, t, labels, ignore_index=0, n_cls=C, hw_shape=(h, w))
    t0 = time.perf_counter()
    for _ in range(steps):
        O.head_step(v, t, labels, ignore_index=0, n_cls=C, hw_shape=(h, w))
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return dt, torch.get_num_threads()


def run_reference(a):
    """--impl reference: the reference's own CPU implementation of the path (the oracle: reference lines
    restated with live torch ops; the reference is pure Python and cannot run as shipped - SURVEY 0) on
    all host threads, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    h, w, HW_ = GEOM[a.geometry]
    steps = a.steps if a.steps is not None else 5
    warmup = a.warmup if a.warmup is not None else 1
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    Bs = 2
    t1, _ = cpu_reference_time(Bs, h, w, a.classes, 1, 0, cores)          # probe
    if t1 * (steps + warmup) > 150 and Bs > 1:
        Bs = 1
    dt, thr = cpu_reference_time(Bs, h, w, a.classes, steps, warmup, cores)
    val = Bs / dt
    sample = f"{Bs} images per step of the same workload (oracle.head_step, fp32, torch CPU)"
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(a, h, w), "global_batch": a.gpus * a.batch, "parallelism": f"dp{a.gpus}",
                   "backward": not a.no_backward},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": thr, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
def _device_ms(fn, world, dev, dist):
    """CUDA-event time of fn() on the current stream, barrier + synchronize on both sides, max over ranks."""
    import torch
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    tm = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    return float(tm)


def _step_leg(name, geometry, B, C, world, rank, dev, dist, steps=10, warmup=3, extra_bucket_floats=0, note=""):
    """A short secondary leg: HeadStep at another BASELINE configuration / geometry (device-resident inputs, eager calls,
    two rotating input sets larger than L2 where the shape allows)."""
    import torch
    from lc2is_b200 import synthetic
    from lc2is_b200.step import HeadStep
    h, w, HW_ = GEOM[geometry]
    H = W = HW_
    sets = []
    for i in range(2):
        v = synthetic.make_patch_embeddings(B, h * w, 512, seed=synthetic.SEED + 13 * (rank * 2 + i)).to(dev)
        lab = synthetic.make_labels(B, H, W, C, seed=synthetic.SEED + 13 * (rank * 2 + i), ignore_frac=0.1).to(dev)
        sets.append((v, lab))
    t = synthetic.make_prototypes(C, 512).to(dev)
    step = HeadStep(B, h, w, H, W, C, 512, ignore_index=0, device=dev, distributed=world > 1,
                    extra_bucket_floats=extra_bucket_floats)
    for i in range(warmup):
        step(sets[i % 2][0], t, sets[i % 2][1])
    step.flush()
    step.global_confmat()                                     # warm-up of the pass-end collective too (first use of a message
    step.reset_metrics()                                      # size sets NCCL channels up: 40 ms at 8 GPUs for 5.7 MB)

    def run():
        for i in range(steps):
            step(sets[i % 2][0], t, sets[i % 2][1])
        step.flush()
        step.global_confmat()
    ms = _device_ms(run, world, dev, dist)
    step.timers = {}
    for i in range(4):
        step(sets[i % 2][0], t, sets[i % 2][1])
    step.flush()
    torch.cuda.synchronize()
    sect = {k: round(statistics.mean(s.elapsed_time(e) for s, e in v) * 1e3, 1) for k, v in step.timers.items()}
    out = {"workload": f"{name}: B={B}/GPU, {h}x{w}->{H}x{H} (x{H // h}), C={C}, D=512", "steps": steps,
           "ms_per_step": ms / steps, "value": world * B * steps / (ms * 1e-3), "unit": "images/s" if H == 512 else f"{H}^2 images/s",
           "section_us": sect, "loss": float(step.loss), "fused_k2k3": bool(step.fused), "split": bool(step.split)}
    if extra_bucket_floats:
        out["bucket_bytes"] = 4 * (C * 512 + 1 + extra_bucket_floats)
    if note:
        out["note"] = note
    del step, sets
    torch.cuda.empty_cache()
    return out


def _cfg3_leg(world, rank, dev, dist, peak, n_images=2000, C=150, H=512):
    """BASELINE config 3: full-val-size eval (2000 images of 512^2) sharded over the ranks: argmax + confusion matrix of
    MATERIALISED [n,C,512,512] fp32 logits (k3_full_kernel; reference metrics.py:127-134 on the tensor engine.py:162-163
    concatenates), ONE int64 all-reduce at the end - and the fused-from-low-resolution form ([n,C,32,32] -> x16)."""
    import torch
    from lc2is_b200 import dp, ops, synthetic
    lo, hi = dp.shard_range(n_images, rank, world)
    n_local = hi - lo
    chunk = 16
    g = torch.Generator(device=dev).manual_seed(1024 + rank)
    low = torch.randn(chunk, C, 32, 32, generator=g, device=dev) * 0.05
    logits = torch.nn.functional.interpolate(low, size=(H, H), mode="bilinear")      # one 2.5 GB chunk, reused (>> L2)
    labs = [synthetic.make_labels(chunk, H, H, C, seed=synthetic.SEED + 7 * (rank * 3 + i), ignore_frac=0.1).to(dev)
            for i in range(3)]
    cm = torch.zeros(C, C, dtype=torch.int64, device=dev)

    def run_full():
        cm.zero_()
        done = 0
        i = 0
        while done < n_local:
            nb = min(chunk, n_local - done)
            ops.argmax_confmat(logits[:nb], labs[i % 3][:nb], confmat=cm)
            done += nb
            i += 1
        dp.allreduce_confmat_(cm)
    run_full()
    ms_full = _device_ms(run_full, world, dev, dist)
    total_full = int(cm.sum())
    pred_ref = logits.argmax(1)
    cm_ref = torch.zeros_like(cm)
    # bit-exact check of this rank's first chunk against torch.argmax + bincount on the same materialised logits
    cm1 = torch.zeros_like(cm)
    ops.argmax_confmat(logits, labs[0], confmat=cm1)
    cm_ref += torch.bincount((labs[0] * C + pred_ref).flatten(), minlength=C * C).view(C, C)
    exact = bool(torch.equal(cm1, cm_ref))

    def run_low():
        cm.zero_()
        done = 0
        i = 0
        while done < n_local:
            nb = min(chunk, n_local - done)
            ops.argmax_confmat(low[:nb], labs[i % 3][:nb], confmat=cm, size=(H, H), mode="bilinear")
            done += nb
            i += 1
        dp.allreduce_confmat_(cm)
    run_low()
    ms_low = _device_ms(run_low, world, dev, dist)
    total_low = int(cm.sum())
    bytes_img = C * H * H * 4 + H * H * 8
    gbs = n_local * bytes_img / (ms_full * 1e-3) / 1e9       # this rank's stream (ranks run the same amount +-1 image)
    out = {"workload": f"cfg3: {n_images} images of {H}^2, C={C}, fp32 logits, sharded over {world} rank(s) "
                       f"({n_local} on rank 0), one int64 all-reduce",
           "materialised": {"kernel": "k3_full_kernel<float,true>", "ms": ms_full, "images_per_s": n_images / (ms_full * 1e-3),
                            "algorithmic_bytes_per_image": bytes_img, "achieved_gbs_per_gpu": gbs, "hbm_frac": gbs / peak,
                            "ideal_images_per_s_per_gpu": peak * 1e9 / bytes_img},
           "fused_from_lowres_x16": {"kernel": "k3_strip_kernel<16,false>", "ms": ms_low,
                                     "images_per_s": n_images / (ms_low * 1e-3)},
           "check": {"confmat_total_materialised": total_full, "confmat_total_lowres": total_low,
                     "expected_total": n_images * H * H, "first_chunk_equals_torch_argmax_bincount": exact}}
    del logits, low, labs
    torch.cuda.empty_cache()
    return out


def run_b200(a):
    import torch
    import torch.distributed as dist
    from lc2is_b200 import _lib, dp, synthetic
    from lc2is_b200.step import HeadStep, HostStep

    rank, world, local_rank = dp.init_distributed()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: lc2is_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    steps = a.steps if a.steps is not None else 200
    warmup = a.warmup if a.warmup is not None else 20
    warmup = max(warmup, 3)
    h, w, HW_ = GEOM[a.geometry]
    B, C, D, H, W = a.batch, a.classes, 512, HW_, HW_
    backward = not a.no_backward

    # ---- inputs: rotate over enough distinct sets that a step's inputs never sit in the 126 MB L2 (an even number:
    # the step alternates two accumulator blocks and the captured graphs bake in (input set, block))
    set_bytes = B * h * w * D * 2 + B * H * W * 8
    nset = max(2, -(-2 * L2_BYTES // set_bytes))
    nset += nset % 2
    t_host = synthetic.make_prototypes(C, D)
    host_sets = []
    for i in range(nset):
        hv = synthetic.make_patch_embeddings(B, h * w, D, seed=synthetic.SEED + 97 * (rank * nset + i)).pin_memory()
        hl = synthetic.make_labels(B, H, W, C, seed=synthetic.SEED + 97 * (rank * nset + i), ignore_frac=0.1).pin_memory()
        host_sets.append((hv, hl))
    dev_sets = [(hv.to(dev), hl.to(dev)) for hv, hl in host_sets]
    t_dev = t_host.to(dev)
    t_pin = t_host.pin_memory()

    step = HeadStep(B, h, w, H, W, C, D, ignore_index=0, backward=backward, device=dev, distributed=world > 1)

    def barrier():
        if world > 1:
            dist.barrier()

    # ---- device-resident timing -----------------------------------------------------------------------
    # Warm-up runs eagerly; then every (input set, accumulator block) pair is captured into a CUDA graph - kernels AND
    # the NCCL collectives - and the timed region replays them: one cudaGraphLaunch per step.  --no-graph (or a failed
    # capture) times eager calls instead.
    n_warm = warmup + (warmup % 2)                            # even: graph i then sees input set i and block i % 2
    for i in range(n_warm):
        step(dev_sets[i % nset][0], t_dev, dev_sets[i % nset][1])
    step.global_confmat()                                     # warm-up of the pass-end collective
    torch.cuda.synchronize()
    graphs, graph_err = None, None
    if world > 1 and (step.comm is None or os.environ.get("LC2IS_DP_GRAPH") == "0"):
        # torch.distributed's NCCL collectives captured into a CUDA graph hung ProcessGroupNCCL's watchdog on this stack
        # (torch 2.11 / NCCL 2.28): without the direct ncclAllReduce route the data-parallel runs time eager launches
        graph_err = "not attempted (collectives through torch.distributed are not captured)"
    elif not a.no_graph:
        state = (step._cur, step._pending)
        try:
            graphs = [step.capture(dev_sets[i][0], t_dev, dev_sets[i][1]) for i in range(nset)]
            torch.cuda.synchronize()
            assert (step._cur, step._pending) == state
        except Exception as e:  # noqa: BLE001
            graphs, graph_err = None, repr(e)[:300]
            step._cur, step._pending = state
            torch.cuda.synchronize()
        if world > 1:                                         # all ranks replay graphs, or none does
            ok = torch.tensor([1 if graphs is not None else 0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok) == 0 and graphs is not None:
                graphs, graph_err = None, "capture failed on another rank"
                step._cur, step._pending = state
        if graphs is not None:
            for i in range(nset):                             # one untimed replay of every graph
                graphs[i]()
            torch.cuda.synchronize()

    def one_step(i):
        if graphs is not None:
            graphs[i % nset]()
        else:
            step(dev_sets[i % nset][0], t_dev, dev_sets[i % nset][1])

    sampler = ClockSampler(physical_gpu_index(local_rank))
    barrier()
    torch.cuda.synchronize()
    launches0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    step.reset_metrics()
    sampler.start()
    t_host0 = time.perf_counter()
    ev0.record()
    for i in range(steps):
        one_step(i)
    step.flush()                                             # the last step's gradient-bucket all-reduce (N > 1)
    cm_total = step.global_confmat()                         # ONE int64 all-reduce for the whole pass (N > 1)
    ev1.record()
    host_enqueue_ms = (time.perf_counter() - t_host0) * 1e3 / steps     # host time to enqueue one step
    torch.cuda.synchronize()
    sampler.stop_flag = True
    if a.dump_outputs and rank == 0:
        # before the eager passes below overwrite the step's buffers; grad_v is not computed without the backward
        outs = {"loss": step.loss, "n_valid": step.n_valid, "logits": step.logits, "confmat": cm_total}
        if backward:
            outs.update(grad_v=step.grad_v, grad_t=step.grad_t)
        write_outputs(outs, a.dump_outputs)
    barrier()
    launches = _lib.launch_count() - launches0
    ms_total = ev0.elapsed_time(ev1)
    tm = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    ms_total = float(tm)
    ms_per_step = ms_total / steps
    value = world * B * steps / (ms_total * 1e-3)
    loss_val = float(step.loss)
    n_valid_val = int(step.n_valid)
    cm_sum = int(cm_total.sum())
    miou = None
    try:
        from lc2is_b200 import metrics
        miou = float(metrics.miou_from_confmat(cm_total, 0))
    except Exception:  # noqa: BLE001
        pass
    sampler.join(timeout=1)
    clocks = sampler.result()

    # ---- the dominant kernel, timed in situ: an eager pass over the same steps right after the timed region, CUDA
    # events around the launch inside every step (events cannot be read back from inside a replayed graph)
    k_steps = min(steps, 50)
    k2_pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k_steps)]
    for i in range(k_steps):
        step.k2_events = k2_pairs[i]
        step(dev_sets[i % nset][0], t_dev, dev_sets[i % nset][1])
    step.k2_events = None
    step.flush()
    torch.cuda.synchronize()
    k2_ms = statistics.mean(s.elapsed_time(e) for s, e in k2_pairs)
    launches_per_step_eager = None
    if graphs is not None:                                   # a replayed graph launches the same kernels as an eager step
        l0 = _lib.launch_count()
        step(dev_sets[0][0], t_dev, dev_sets[0][1])
        step.flush()
        launches_per_step_eager = _lib.launch_count() - l0
        launches = launches_per_step_eager * steps

    section_us = None
    if a.kernel_times:
        step.timers = {}
        for i in range(20):
            step(dev_sets[i % nset][0], t_dev, dev_sets[i % nset][1])
        step.flush()
        torch.cuda.synchronize()
        section_us = {k: round(statistics.mean(s.elapsed_time(e) for s, e in v) * 1e3, 1) for k, v in step.timers.items()}
        step.timers = None

    # ---- data-parallel parity, visible to the driver (the 2-GPU pytest is skipped on a 1-GPU box) ------------
    dp_check = None
    if world > 1:
        try:
            vd, ld = dev_sets[0]
            step.reset_metrics()
            step(vd, t_dev, ld)
            step.flush()
            cm_dp = step.global_confmat().clone()
            nv_dp, loss_dp, gt_dp = int(step.n_valid), float(step.loss), step.grad_t.clone()
            v_all = [torch.empty_like(vd) for _ in range(world)]
            l_all = [torch.empty_like(ld) for _ in range(world)]
            dist.all_gather(v_all, vd)
            dist.all_gather(l_all, ld)
            dp_check = {"confmat_total_timed_pass": cm_sum, "expected_total": world * B * steps * H * W,
                        "confmat_total_ok": cm_sum == world * B * steps * H * W}
            if rank == 0:
                ref = HeadStep(world * B, h, w, H, W, C, D, ignore_index=0, backward=backward, device=dev, distributed=False)
                ref(torch.cat(v_all), t_dev, torch.cat(l_all))
                torch.cuda.synchronize()
                dp_check.update({
                    "one_step_vs_single_gpu_on_concatenated_batch": {
                        "confmat_equal": bool(torch.equal(cm_dp, ref.confmat)),
                        "n_valid": [nv_dp, int(ref.n_valid)],
                        "loss_rel_err": abs(loss_dp - float(ref.loss)) / abs(float(ref.loss)),
                        "grad_t_rel_err": float((gt_dp - ref.grad_t).abs().max() / ref.grad_t.abs().max()),
                    }})
                o = dp_check["one_step_vs_single_gpu_on_concatenated_batch"]
                dp_check["ok"] = bool(dp_check["confmat_total_ok"] and o["confmat_equal"] and o["n_valid"][0] == o["n_valid"][1]
                                      and o["loss_rel_err"] <= 1e-5 and o["grad_t_rel_err"] <= 5e-3)
                del ref
            del v_all, l_all
            torch.cuda.empty_cache()
        except Exception as e:  # noqa: BLE001
            dp_check = {"error": repr(e)[:300]}
        barrier()

    # ---- end to end: host (pinned) buffers through the C-ABI host entry, H2D/D2H inside the timed region
    e2e = None
    if not a.no_e2e:
        hstep = HostStep(B, h, w, H, W, C, D, ignore_index=0, backward=backward, device=dev, depth=2)
        cm_dev = torch.zeros(C, C, dtype=torch.int64, device=dev)
        e_steps = max(3, min(steps, 200))

        cm_host = torch.zeros(C, C, dtype=torch.int64)

        def finish(out):
            cm_host.add_(out[2])                            # the pass's confusion matrix accumulates on the host

        def reduce_confmat():
            if world > 1:                                   # DP: ONE int64 all-reduce for the whole pass
                cm_dev.copy_(cm_host)
                dist.all_reduce(cm_dev)
                torch.cuda.synchronize()

        def run(n, first):
            """n steps through submit / wait with two steps in flight: every step copies its own inputs from
            pinned host memory and reads its own results back; the copy of step i+1 overlaps the kernels of
            step i (a prefetching loader).  Returns the last results."""
            hv, hl = host_sets[first % nset]
            hstep.submit(hv, t_pin, hl)
            out = None
            for i in range(1, n):
                hv, hl = host_sets[(first + i) % nset]
                hstep.submit(hv, t_pin, hl)
                if i + 1 < n:                               # loader-style prefetch: the library's host threads pack the
                    hstep.prefetch(host_sets[(first + i + 1) % nset][1])   # next batch's labels while this thread waits
                out = hstep.wait()
                finish(out)
            out = hstep.wait()
            finish(out)
            reduce_confmat()
            return out

        def timed(fn):
            barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            barrier()
            ms = max(e0.elapsed_time(e1), wall * 1e3)        # the calls block the host: take the larger clock
            tm = torch.tensor([ms], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            return float(tm)

        run(4, 0)
        ms_pipe = timed(lambda: run(e_steps, 4))
        assert int(hstep.out_n_valid) > 0

        def blocking():
            for i in range(e_steps):
                hv, hl = host_sets[(4 + i) % nset]
                hstep(hv, t_pin, hl)
                finish((hstep.out_loss, hstep.out_n_valid, hstep.out_confmat))
            reduce_confmat()
        hstep(host_sets[0][0], t_pin, host_sets[0][1])
        ms_block = timed(blocking)
        e2e = {"value": world * B * e_steps / (ms_pipe * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": hstep.h2d_bytes, "d2h_bytes_per_step": hstep.d2h_bytes,
               "steps": e_steps, "ms_per_step": ms_pipe / e_steps,
               "h2d_gbs_per_gpu": hstep.h2d_bytes / (ms_pipe / e_steps * 1e-3) / 1e9,
               "h2d_gbs_node_aggregate": world * hstep.h2d_bytes / (ms_pipe / e_steps * 1e-3) / 1e9,
               "scope": "per-rank independent steps (each rank's own loss / n_valid / gradients; only the integer confusion "
                        "matrix is all-reduced, once per pass): the ranks share the host's cores, DRAM and PCIe root, so "
                        "this figure is platform-bound at N > 1",
               "api": "lc2is_head_step_host_submit / _wait, 2 steps in flight, labels of the next batch packed in the "
                      "background (lc2is_pack_labels_host_begin/_end); pinned host buffers in: bf16 V, fp32 T, int64 labels "
                      "narrowed to 1 byte (C <= 254) by the library's host threads and widened on the device; loss/n_valid/confmat out",
               "label_route": {"host_label_bytes": hstep.label_bytes, "n_raw_int64_images": hstep.n_raw if hstep.host_pack else B,
                               "calibration": hstep.calibration},
               "blocking_call": {"api": "lc2is_head_step_host", "ms_per_step": ms_block / e_steps,
                                 "value": world * B * e_steps / (ms_block * 1e-3)}}
        hstep.close()
        del hstep
        torch.cuda.empty_cache()

    # ---- secondary legs: the other BASELINE configurations / geometries, short and device-timed ----------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (burst copy)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    secondary = None
    if not a.no_secondary and a.geometry == "A":
        del dev_sets, host_sets
        torch.cuda.empty_cache()
        secondary = {}
        legs = [
            ("cfg3_eval", lambda: _cfg3_leg(world, rank, dev, dist, peak)),
            ("G-B", lambda: _step_leg("G-B main head (final.py:44)", "B", B, C, world, rank, dev, dist)),
            ("cfg4", lambda: _step_leg("cfg4 data-parallel training step, global batch 8 x N", "A", 8, C, world, rank, dev, dist,
                                       steps=20, extra_bucket_floats=656384,
                                       note="2.93 MB gradient bucket: d prototypes + loss (live) + 656,384 zero-filled fp32 slots "
                                            "standing in for the TextToPatch gradients (the projection backward is not part of "
                                            "this step), all-reduced behind the next step")),
            ("cfg5", lambda: _step_leg("cfg5 open-vocabulary stress", "5", 8, 847, world, rank, dev, dist, steps=5, warmup=2)),
        ]
        for name, fn in legs:
            if name not in a.legs.split(","):
                continue
            try:
                secondary[name] = fn()
            except Exception as e:  # noqa: BLE001
                secondary[name] = {"error": repr(e)[:300]}
                torch.cuda.empty_cache()
            barrier()

    if rank != 0:
        if world > 1:
            torch.cuda.synchronize()
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel ---------------------------------------------------------------------
    split, fused = step.split, getattr(step, "fused", False)
    # Dominant launch: on the x16 geometry K2 (bilinear upsample + softmax-CE fwd/bwd) and K3 (argmax + confusion matrix)
    # are ONE kernel.  Algorithmic bytes of that launch (SURVEY 8d: K2 fused reads low + writes grad_low + the label map;
    # the labels reach this kernel packed to uint16 by k2_pack_labels_kernel): 2*B*C*h*w*4 + B*H*W*2 + 8.
    if fused:
        k2_bytes = 2 * B * C * h * w * 4 + B * H * W * 2 + 8
        k2_name = "k23_rc_kernel<16>"
        k2_desc = "lc2is_ce_argmax_fused_packed: bilinear upsample + softmax-CE fwd/bwd + argmax + confusion matrix"
    else:
        k2_bytes = 2 * B * C * h * w * 4 + B * H * W * (2 if split else 8) + 8
        k2_name = ("k2_strip_kernel<16, true>" if H // h == 16 else "k2_strip_kernel<8, true>") if split else \
            "k2_fast_kernel / k2_generic_kernel"
        k2_desc = "lc2is_upsample_ce_packed: fused bilinear upsample + softmax-CE fwd+bwd"
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath) and a.geometry == "A" and B == 16 and C == 150:
        traffic = json.load(open(tpath)).get(k2_name)                 # from one `ncu --set full` capture
    hbm_achieved = k2_bytes / (k2_ms * 1e-3) / 1e9
    # The kernel never materialises the upsampled [B,C,H,W] tensor, so HBM does not bind it (a few % of peak by
    # construction); what binds is the FP32 pipe: per upsampled element 2 lane-ops in pass A (add, mul), 2 in the
    # Horner sweep (two fma) and - fused kernel - 1 to evaluate the logit for the argmax.  Peak = 128 FP32 lanes per SM
    # and clock (a packed FFMA2 / FADD2 / FMUL2 issues at 2.0 warp-inst/clk/SM = the same 128 lane-ops; measured,
    # tools/micro).  The running maximum (FMNMX3) goes to the ALU pipe and is not counted.
    sm_hz = (clocks.get("sm_mhz") or 1965) * 1e6
    ops_per_elem = 5 if fused else 4
    lane_ops = float(B) * C * H * W * ops_per_elem
    fp32_peak = 148 * 128 * sm_hz / 1e12
    fp32_achieved = lane_ops / (k2_ms * 1e-3) / 1e12
    roofline = {"kernel": f"{k2_name} ({k2_desc})",
                "bound": "fp32_issue", "achieved": fp32_achieved, "peak": fp32_peak, "unit": "T fp32 lane-op/s",
                "frac": fp32_achieved / fp32_peak, "traffic": traffic,
                "peak_source": "148 SMs x 128 FP32 lanes x the SM clock sampled during the timed region",
                "algorithmic_lane_ops": lane_ops, "lane_ops_per_upsampled_element": ops_per_elem,
                "kernel_us": k2_ms * 1e3,
                "kernel_us_source": f"CUDA events around the launch in {k_steps} eager steps right after the timed region",
                "upsampled_elements_per_s": B * C * H * W / (k2_ms * 1e-3),
                "hbm": {"achieved": hbm_achieved, "peak": peak, "unit": "GB/s", "frac": hbm_achieved / peak,
                        "algorithmic_bytes": k2_bytes, "peak_source": peak_src,
                        "note": "secondary: HBM does not bind this kernel"}}

    cpu_baseline = None
    if not a.no_cpu_baseline and world == 1:
        cores = os.cpu_count() or 1
        dt, thr = cpu_reference_time(2, h, w, C, 2, 1, cores)
        cpu_baseline = {"value": 2 / dt, "unit": UNIT, "cores": thr, "kind": "port",
                        "sample": "2 images per step of the same workload, 2 timed steps after 1 warm-up "
                                  "(oracle.head_step: reference lines on torch CPU, fp32)"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": n_warm,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": workload_name(a, h, w), "global_batch": world * B, "parallelism": f"dp{world}",
                   "backward": backward},
        "timing": {"l2": f"inputs rotate over {nset} distinct sets ({nset * set_bytes / 2**20:.0f} MiB) > 126 MiB L2; no flush",
                   "launch": ("CUDA graph replay (one graph per input set" +
                              ("; three kernel-only graphs per step, the two ncclAllReduce launches eager in between)"
                               if world > 1 else ")")) if graphs is not None else "eager launches",
                   "graph_error": graph_err},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
        "cpu_baseline": cpu_baseline, "section_us": section_us, "host_enqueue_ms_per_step": host_enqueue_ms,
        "check": {"loss": loss_val, "mIoU": miou, "n_valid": n_valid_val, "confmat_total": cm_sum,
                  "confmat_total_expected": world * B * steps * H * W},
        "dp_check": dp_check, "secondary": secondary,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)


if __name__ == "__main__":
    main()
