"""TextToPatch.visual's projection GEMMs per element against float64 references built from their own bf16 operands:
lc2is_linear_fwd (k1_linear_2sm_kernel, the cta_group::2 CTA-pair form, or k1_logits_kernel<1>, the persistent 1-SM form)
and lc2is_linear_bwd (gx: transpose_bf16_kernel, then lc2is_linear_fwd on the transposed weight, either form; gw:
k1b_dt_kernel<true, 2, true> split-K slices summed by reduce_partials_kernel; gb: colsum_bf16_kernel + colsum_finish_kernel).

References, float64 on the device, each with its error scale A (the same sum over absolute values):
    y  = x w^T + b            A = |x| |w|^T + |b|
    gx = gy w                 A = |gy| |w|
    gw = base + gy^T x        A = |gy|^T |x|
    gb = base + sum_m gy      A = sum_m |gy|
Bound, per element: |got - ref| <= TAU A, plus BF16_OUT |ref| for a bf16 output and one fp32 rounding of base + ref for an
accumulated one; TAU = 2^-16 and BF16_OUT = 2^-8 as in tests/k1b_reference.py (test_gpu_k1b_exact.py says where they come
from).  check_bound asserts it per [128 rows x 64 channels] block, so a failure names the block.  The entries are called
directly with y and gx filled with NaN and the workspace with NaN bytes: an element no kernel writes, or a split-K slice no
CTA stores, fails.  Every call also asserts its route - the kernels torch.profiler records, in launch order, with their grid
sizes - against the plan the entries compute from the device's SM count (_fwd_plan, _gw_plan, _gb_blocks below), and each
case asserts that the plan takes the branch it is there for.

Inputs: x rows scaled over 4x, output channels of w (and of gy) scaled by powers of two from 2^-3 to 2^3 so that small
outputs sit next to large ones, every eighth row of gy zero (their gx rows must come out exactly 0), bias on and off.

Worst |got - ref| / A measured on one B200 (1000 W power limit), per route, over the fp32 outputs of every case here:
    y  k1_logits_kernel<1>      5.4e-7 (2^-20.8)   M 1000, K 4096, N 256 (64 k-blocks per tile)
    y  k1_linear_2sm_kernel     3.7e-7 (2^-21.4)   G-B
    gx k1_logits_kernel<1>      6.4e-7 (2^-20.6)   M 1000, K 320, N 512
    gx k1_linear_2sm_kernel     8.1e-7 (2^-20.2)   G-B
    gw split-K + reduction      7.9e-7 (2^-20.3)   M 4000, K 2560, N 4096 (one slice: 63 k-blocks in one accumulator)
                                2.2e-7             G-B (24 slices of about 170 k-blocks)
    gb column sums              1.1e-8 (2^-26.4)   M 3000, N 384 (accumulated); 1.4e-9 at G-B
i.e. at most 1/19 of TAU; the file runs in about 10 s.  A bf16 y or gx uses up to 0.99 of its bound: that is its own
rounding (at most 2^-8 |x|), not kernel error.  Dropping the last k-block of the 1-SM route (P.num_kb = K / 64 - 1 in
lc2is_linear_fwd) makes every 1-SM case tried fail - the G-A forward, the M = 129 channel tails and K = 4096, the last at
970x the bound - with the message naming the block.
"""
import json
import os
import tempfile

import pytest
import torch

from k1b_reference import check_bound
from lc2is_b200 import _lib, ops
from lc2is_b200._lib import F32, lib, ptr, stream_ptr

pytestmark = pytest.mark.gpu
DEV = "cuda"
ERR_ARG = -1
BF16 = torch.bfloat16
FP32 = torch.float32

TWO_SM, ONE_SM = "k1_linear_2sm_kernel", "k1_logits_kernel<1>"
GW_GEMM = "k1b_dt_kernel<true,2,true>"
KERNELS = (TWO_SM, ONE_SM, "transpose_bf16_kernel", GW_GEMM, "reduce_partials_kernel", "colsum_bf16_kernel",
           "colsum_finish_kernel")


def _sm() -> int:
    return torch.cuda.get_device_properties(0).multi_processor_count


def _cdiv(a: int, b: int) -> int:
    return -(-a // b)


def _fwd_plan(M, N, K):
    """lc2is_linear_fwd's route (k1_logits.cu): the 2-SM form when 256 x 256 pair tiles cover the output exactly and
    there are at least two per CTA pair, the 1-SM form with tiles of 128 rows x NB channels otherwise.
    -> dict(kernel, grid, tiles, NB)."""
    pairs = _sm() // 2
    pair_tiles = (M // 256) * (N // 256)
    if M % 256 == 0 and N % 256 == 0 and pair_tiles >= 2 * pairs:
        return dict(kernel=TWO_SM, grid=2 * pairs, tiles=pair_tiles, NB=256)
    nb = _cdiv(_cdiv(N, _cdiv(N, 256)), 16) * 16
    tiles = _cdiv(M, 128) * _cdiv(N, nb)
    return dict(kernel=ONE_SM, grid=min(_sm(), tiles), tiles=tiles, NB=nb)


def _gw_plan(M, N, K):
    """The weight-gradient GEMM of lc2is_linear_bwd (k1b_bwd.cu): NB channels and 256 features per CTA, the 64-row blocks
    split in ksplit slices = SM count / tiles, clamped to [1, number of blocks] and to 32.
    -> dict(NB, tiles, kb, ksplit)."""
    nb = 256 if N % 256 == 0 else 128 if N % 128 == 0 else 64
    tiles = _cdiv(K, 256) * (N // nb)
    kb = _cdiv(M, 64)
    return dict(NB=nb, tiles=tiles, kb=kb, ksplit=min(max(_sm() // tiles, 1), kb, 32))


def _gb_blocks(M):
    """CTAs of colsum_bf16_kernel: one per 256 rows, at most two per SM and 1024."""
    return min(_cdiv(M, 256), 2 * _sm(), 1024)


def _bwd_launches(M, N, K, need_gx, need_gw, need_gb):
    out = []
    if need_gx:
        p = _fwd_plan(M, K, N)
        out += [("transpose_bf16_kernel", _cdiv(K, 32)), (p["kernel"], p["grid"])]
    if need_gw:
        p = _gw_plan(M, N, K)
        out += [(GW_GEMM, p["tiles"] * p["ksplit"]),
                ("reduce_partials_kernel", min(_cdiv(N * K // 4, 256), 8 * _sm()))]
    if need_gb:
        out += [("colsum_bf16_kernel", _gb_blocks(M)), ("colsum_finish_kernel", _cdiv(N, 32))]
    return out


def _launches(fn):
    """fn()'s return value and [(kernel, grid.x)] of the CUDA kernels it launched, in launch order, from torch.profiler's
    trace; demangled names lose their spaces and are shortened to the entry of KERNELS they contain."""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        rc = fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    kernels = sorted((e for e in events if e.get("cat") == "kernel"), key=lambda e: e["ts"])

    def short(name):
        name = name.replace(" ", "")
        return next((k for k in KERNELS if k in name), name)
    return rc, [(short(e["name"]), e["args"]["grid"][0]) for e in kernels]


def _operands(M, N, K, seed, bias=True):
    """bf16 x [M, K], bf16 w [N, K], fp32 bias [N] (or None) and bf16 gy [M, N] (see the module docstring)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(M, K, generator=g, device=DEV) * (0.5 + 1.5 * torch.rand(M, 1, generator=g, device=DEV))
    ch = 2.0 ** torch.randint(-3, 4, (N, 1), generator=g, device=DEV)
    w = torch.randn(N, K, generator=g, device=DEV) * K ** -0.5 * ch
    b = torch.randn(N, generator=g, device=DEV) * ch[:, 0] if bias else None
    gy = torch.randn(M, N, generator=g, device=DEV) * 2.0 ** torch.randint(-3, 4, (1, N), generator=g, device=DEV)
    gy[7::8] = 0
    return x.to(BF16), w.to(BF16), b, gy.to(BF16)


def _report(route, case, r, bf16_out):
    print(f"linear-exact {route} [{case}]: |d|/A {r[0]:.3g}{' (bf16 out)' if bf16_out else ''}  bound use {r[1]:.3g}")


def _route(kernel):
    return "2-SM" if kernel == TWO_SM else "1-SM"


def _fwd(x, w, b, y):
    return lib.lc2is_linear_fwd(ptr(x), ptr(w), ptr(b), x.shape[0], w.shape[0], x.shape[1], ptr(y), ops._dt(y),
                                stream_ptr())


def _bwd(gy, x, w, gx, gw, gb, ws):
    (M, N), K = gy.shape, x.shape[1]
    return lib.lc2is_linear_bwd(ptr(gy), ptr(x), ptr(w), M, N, K, ptr(gx), F32 if gx is None else ops._dt(gx), ptr(gw),
                                ptr(gb), ptr(ws), stream_ptr())


def _workspace(N, K):
    return torch.full((int(lib.lc2is_linear_bwd_workspace(N, K)),), 0xFF, dtype=torch.uint8, device=DEV)


def run_fwd(x, w, b, out_dtype, case):
    """One lc2is_linear_fwd call: route asserted, y checked per element."""
    M, K = x.shape
    N = w.shape[0]
    y = torch.full((M, N), float("nan"), dtype=out_dtype, device=DEV)
    rc, launches = _launches(lambda: _fwd(x, w, b, y))
    assert rc == 0, _lib.last_error()
    plan = _fwd_plan(M, N, K)
    assert launches == [(plan["kernel"], plan["grid"])], (case, launches)
    x64, w64 = x.double(), w.double()
    ref, A = x64 @ w64.t(), x64.abs() @ w64.abs().t()
    if b is not None:
        ref += b.double()
        A += b.double().abs()
    bf = out_dtype == BF16
    _report(f"fwd {_route(plan['kernel'])}", case, check_bound(f"{case} y", y, ref, A, bf16_out=bf), bf)


def run_bwd(x, w, gy, gx_dtype, case, need=(True, True, True), gw0=None, gb0=None):
    """One lc2is_linear_bwd call for the requested outputs (gw / gb accumulated into gw0 / gb0, zeros by default): route
    asserted, every output checked per element."""
    M, K = x.shape
    N = w.shape[0]
    gx = torch.full((M, K), float("nan"), dtype=gx_dtype, device=DEV) if need[0] else None
    gw = (torch.zeros(N, K, device=DEV) if gw0 is None else gw0.clone()) if need[1] else None
    gb = (torch.zeros(N, device=DEV) if gb0 is None else gb0.clone()) if need[2] else None
    ws = _workspace(N, K)
    rc, launches = _launches(lambda: _bwd(gy, x, w, gx, gw, gb, ws))
    assert rc == 0, _lib.last_error()
    assert launches == _bwd_launches(M, N, K, *need), (case, launches)
    gy64 = gy.double()
    if gx is not None:
        w64 = w.double()
        bf = gx_dtype == BF16
        r = check_bound(f"{case} gx", gx, gy64 @ w64, gy64.abs() @ w64.abs(), bf16_out=bf)
        _report(f"gx {_route(_fwd_plan(M, K, N)['kernel'])}", case, r, bf)
    if gw is not None:
        x64 = x.double()
        r = check_bound(f"{case} gw", gw, gy64.t() @ x64, gy64.abs().t() @ x64.abs(), base=gw0)
        _report("gw", case, r, False)
    if gb is not None:
        r = check_bound(f"{case} gb", gb.view(1, N), gy64.sum(0, keepdim=True), gy64.abs().sum(0, keepdim=True),
                        base=None if gb0 is None else gb0.view(1, N))
        _report("gb", case, r, False)


# ---- the training shapes ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,K,N,out_dtype", [
    pytest.param(16384, 768, 512, BF16, id="G-A-bf16"),
    pytest.param(16384, 768, 512, FP32, id="G-A-f32"),
    pytest.param(262144, 768, 512, BF16, id="G-B-bf16"),
    pytest.param(262144, 768, 512, FP32, id="G-B-f32"),
])
def test_training_projection(M, K, N, out_dtype):
    """TextToPatch.visual at the benchmark's two geometries (16 images of 32^2 / 128^2 patches, 768 -> 512), forward and
    the whole backward."""
    fwd, gx, gw = _fwd_plan(M, N, K), _fwd_plan(M, K, N), _gw_plan(M, N, K)
    if M == 16384:
        # below the 2-SM threshold: persistent 1-SM CTAs with more than one tile each (TMEM buffer reuse, the stage ring
        # wrapping across tiles); the gx product (N = 768) is above it
        assert fwd["kernel"] == ONE_SM and fwd["tiles"] > fwd["grid"], fwd
        assert gx["kernel"] == TWO_SM, gx
    else:
        # about 28 tiles per CTA pair: the double-buffered accumulator and the cross-CTA drained barrier go through
        # many phases
        assert fwd["kernel"] == gx["kernel"] == TWO_SM and fwd["tiles"] >= 20 * (fwd["grid"] // 2), fwd
    assert gw["ksplit"] == _sm() // gw["tiles"] and gw["kb"] >= 256, gw
    x, w, b, gy = _operands(M, N, K, seed=M)
    case = f"M{M} K{K} N{N} {'bf16' if out_dtype == BF16 else 'f32'}"
    run_fwd(x, w, b, out_dtype, case)
    run_bwd(x, w, gy, out_dtype, case)


# ---- lc2is_linear_fwd: the 2-SM threshold and the 1-SM kernel's channel tails ----------------------------------------
@pytest.mark.parametrize("below", [False, True], ids=["at", "below"])
@pytest.mark.parametrize("K", [64, 128])
def test_two_sm_threshold(K, below):
    """N = 256 (one N tile per pair) and K = 64 / 128 (one or two k-blocks, fewer than the six stages): exactly
    2 (sm / 2) pair tiles take the 2-SM kernel, one pair tile fewer the 1-SM kernel (then with 256-channel tiles)."""
    P = 2 * (_sm() // 2) - int(below)
    M, N = 256 * P, 256
    assert _fwd_plan(M, N, K)["kernel"] == (ONE_SM if below else TWO_SM)
    x, w, b, _ = _operands(M, N, K, seed=K + below, bias=K == 128)
    run_fwd(x, w, b, FP32 if K == 64 else BF16, f"M{M} K{K} N{N}")


@pytest.mark.parametrize("out_dtype", [BF16, FP32], ids=["bf16", "f32"])
@pytest.mark.parametrize("N", [16, 48, 272, 400])
@pytest.mark.parametrize("M", [1, 129, 4001])
def test_one_sm_channel_tails(M, N, out_dtype):
    """N = 16 / 48: one 128-byte column group, which the second epilogue warp of a lane quarter takes alone, ending in
    the 16-column tail; N = 272 / 400: two N tiles of NB = 144 / 208 channels, the last one narrower; M = 1 / 129 / 4001:
    a last row tile with fewer than 32 valid rows per warp."""
    K = 192
    plan = _fwd_plan(M, N, K)
    assert plan["kernel"] == ONE_SM and (N <= 48 or N % plan["NB"] != 0), plan
    x, w, b, _ = _operands(M, N, K, seed=M * 1000 + N, bias=M != 129)
    run_fwd(x, w, b, out_dtype, f"M{M} K{K} N{N} {'bf16' if out_dtype == BF16 else 'f32'}")


def test_deep_k():
    """K = 4096: 64 k-blocks per tile, the longest accumulation chain of the forward, checked at fp32 resolution; and the
    backward of the same shape."""
    M, K, N = 1000, 4096, 256
    x, w, b, gy = _operands(M, N, K, seed=4096)
    run_fwd(x, w, b, FP32, f"M{M} K{K} N{N}")
    run_bwd(x, w, gy, FP32, f"M{M} K{K} N{N}")


# ---- lc2is_linear_bwd: the weight- and bias-gradient branches --------------------------------------------------------
@pytest.mark.parametrize("K", [64, 320])
@pytest.mark.parametrize("N", [64, 192, 384, 512])
def test_weight_gradient_tiles(N, K):
    """NB = 64 / 64 / 128 / 256 channels per gw tile, and K = 64 / 320 - a CTA owns 256 features (MT = 2 accumulators of
    128), so K = 64 masks three quarters of its tile and K = 320 most of the second tile's; M = 1000 ends in a partial
    64-row block."""
    M = 1000
    assert _gw_plan(M, N, K)["NB"] == {64: 64, 192: 64, 384: 128, 512: 256}[N]
    x, w, _, gy = _operands(M, N, K, seed=N + K)
    run_bwd(x, w, gy, BF16 if N == 192 else FP32, f"M{M} K{K} N{N}")


@pytest.mark.parametrize("M,K,N,clamp", [
    pytest.param(4000, 2560, 4096, "one", id="ksplit-1"),
    pytest.param(100, 256, 256, "blocks", id="ksplit-blocks"),
    pytest.param(20000, 256, 256, "max", id="ksplit-32"),
])
def test_weight_gradient_split(M, K, N, clamp):
    """The three clamps of gw's split count: more tiles than SMs (one slice), fewer 64-row blocks than SMs (one slice per
    block) and the 32 slices the workspace holds."""
    p = _gw_plan(M, N, K)
    assert p["ksplit"] == {"one": 1, "blocks": p["kb"], "max": 32}[clamp], p
    assert clamp != "one" or p["tiles"] > _sm()
    assert clamp != "blocks" or p["kb"] < _sm() // p["tiles"]
    assert clamp != "max" or min(_sm() // p["tiles"], p["kb"]) > 32
    x, w, _, gy = _operands(M, N, K, seed=M + N)
    run_bwd(x, w, gy, BF16, f"M{M} K{K} N{N}")


@pytest.mark.parametrize("N", [768, 9216])
@pytest.mark.parametrize("M", [1, 3000])
def test_bias_gradient_column_sums(M, N):
    """gb alone.  N = 768: 96 column groups of 8, so 1024 threads hold 10 row groups and 64 idle threads; N = 9216: 1152
    groups, two column passes of which the second is mostly idle.  M = 1: only the tail of the row loop runs."""
    K = 64
    nvec = N // 8
    assert (nvec < 1024 and 1024 % nvec != 0) or nvec > 1024
    x, w, _, gy = _operands(M, N, K, seed=M + N + 1)
    run_bwd(x, w, gy, FP32, f"M{M} N{N} gb only", need=(False, False, True))


def test_accumulation_and_partial_requests():
    """gw and gb accumulate into non-zero values (a second micro-batch): base + ref, one more fp32 rounding; and every
    subset of the outputs launches only its own kernels."""
    M, K, N = 3000, 320, 384
    x, w, _, gy = _operands(M, N, K, seed=77)
    g = torch.Generator(device=DEV).manual_seed(78)
    gw0 = torch.randn(N, K, generator=g, device=DEV) * 40.0
    gb0 = torch.randn(N, generator=g, device=DEV) * 40.0
    run_bwd(x, w, gy, BF16, "gw and gb accumulated", need=(False, True, True), gw0=gw0, gb0=gb0)
    run_bwd(x, w, gy, BF16, "gx only", need=(True, False, False))
    run_bwd(x, w, gy, FP32, "gw only", need=(False, True, False), gw0=gw0)
    run_bwd(x, w, gy, FP32, "gb only", need=(False, False, True), gb0=gb0)


# ---- pointer alignment -------------------------------------------------------------------------------------------------
def _offset(t):
    """A copy of t that starts 4 bytes past a 16-byte boundary (a view into a larger buffer)."""
    skip = 4 // t.element_size()
    v = torch.empty(t.numel() + skip, dtype=t.dtype, device=t.device)[skip:].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 16 == 4
    return v


def test_unaligned_pointers_are_rejected_before_any_launch():
    """Every pointer the kernels read or write with 16-byte vectors or TMA: LC2IS_ERR_ARG, nothing launched, the outputs
    as they were (y and gx NaN, gw and gb their starting values)."""
    M, K, N = 300, 128, 256
    x, w, b, gy = _operands(M, N, K, seed=5)
    y = torch.full((M, N), float("nan"), dtype=BF16, device=DEV)
    gx = torch.full((M, K), float("nan"), dtype=BF16, device=DEV)
    gw0, gb0 = torch.randn(N, K, device=DEV), torch.randn(N, device=DEV)
    gw, gb = gw0.clone(), gb0.clone()
    ws = _workspace(N, K)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    fwd_args = dict(x=x, w=w, b=b, y=y)
    for name in fwd_args:
        a = dict(fwd_args, **{name: _offset(fwd_args[name])})
        assert _fwd(a["x"], a["w"], a["b"], a["y"]) == ERR_ARG, name
        assert "aligned" in _lib.last_error(), name
    bwd_args = dict(gy=gy, x=x, gx=gx, gw=gw, ws=ws)
    for name in bwd_args:
        a = dict(bwd_args, **{name: _offset(bwd_args[name])})
        assert _bwd(a["gy"], a["x"], w, a["gx"], a["gw"], gb, a["ws"]) == ERR_ARG, name
        assert "aligned" in _lib.last_error(), name
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0
    assert bool(y.isnan().all()) and bool(gx.isnan().all())
    assert torch.equal(gw, gw0) and torch.equal(gb, gb0)
    # gb is read and written per element: an unaligned gb is accepted
    gb_off = _offset(gb0)
    assert _bwd(gy, x, w, None, None, gb_off, ws) == 0, _lib.last_error()
    torch.cuda.synchronize()
    check_bound("unaligned gb", gb_off.view(1, N), gy.double().sum(0, keepdim=True), gy.double().abs().sum(0, keepdim=True),
                base=gb0.view(1, N))


def test_unaligned_views_through_ops_and_text_to_patch():
    """ops.linear_fwd / ops.linear_bwd accept views that start anywhere (copied to aligned memory; a caller's gw accumulated
    through an aligned copy and written back), bit for bit the aligned call; and TextToPatch with its bias a view into a
    flat buffer and an unaligned upstream gradient."""
    from lc2is_b200.model.text_patch import TextToPatch
    M, K, N = 300, 128, 256
    x, w, b, gy = _operands(M, N, K, seed=6)
    assert torch.equal(ops.linear_fwd(_offset(x), _offset(w), _offset(b)), ops.linear_fwd(x, w, b))
    g = torch.Generator(device=DEV).manual_seed(7)
    gw0, gb0 = torch.randn(N, K, generator=g, device=DEV), torch.randn(N, generator=g, device=DEV)
    ref = ops.linear_bwd(gy, x, w, gw=gw0.clone(), gb=gb0.clone())
    gw_off, gb_off = _offset(gw0), _offset(gb0)
    gw_t = gw0.t().contiguous().t()                                   # a transposed view: not contiguous
    for gw_in in (gw_off, gw_t):
        got = ops.linear_bwd(_offset(gy), _offset(x), _offset(w), gw=gw_in, gb=gb_off if gw_in is gw_off else None,
                             need_gb=gw_in is gw_off)
        assert got[1] is gw_in                                        # accumulated into the caller's tensor
        assert torch.equal(got[0], ref[0]) and torch.equal(gw_in, ref[1])
    assert torch.equal(gb_off, ref[2])

    torch.manual_seed(8)
    m = TextToPatch(K, 64, N, tensor_cores=True).to(DEV)
    m_off = TextToPatch(K, 64, N, tensor_cores=True).to(DEV)
    m_off.load_state_dict(m.state_dict())
    m_off.visual.bias = torch.nn.Parameter(_offset(m.visual.bias.detach()))
    img = x.view(2, M // 2, K)
    outs = []
    for mod, grad in ((m, gy), (m_off, _offset(gy))):
        im = img.clone().requires_grad_(True)
        _, v = mod(im, torch.randn(5, 64, device=DEV))
        v.backward(grad.view(2, M // 2, N))
        outs.append((v.detach(), im.grad, mod.visual.weight.grad, mod.visual.bias.grad))
    assert m_off.visual.bias.data_ptr() % 16 == 4
    for a, c in zip(*outs):
        assert torch.equal(a, c)
