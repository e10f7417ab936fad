"""Every GPTQ kernel variant, entry point and dispatch boundary vs the fp64 oracle (``oracle.gptq.dequant_matmul``).

``tests/test_gpu_gptq.py`` covers the default configuration of each kernel.  The cases below reach the branches it
does not, on purpose (the case ids name the branch):
  1. routes: which kernel the automatic dispatch of ``gptq4_matmul`` and ``gptq4_linear_f16`` launches at the M
     thresholds (32, 768) and for misaligned pointers, K % 8 != 0 and N % 4 != 0 -- checked with torch.profiler
     kernel records and the library's launch counter, next to the numbers;
  2. the tcgen05 per-group kernel with the wide TMEM drain and the mbarrier wait back-off: bit-identical outputs;
  3. the persistent tensor-memory-operand kernel with 2-3 tiles per CTA (stage and chunk counters carried across
     tiles), every chunk size, with and without the activation low plane, integer and fractional zero points, and
     its fp16 entry;
  4. all 16 variants of the decode kernel, the CTAs-per-SM nibble up to the K-slice caps S = 8 / 4 / 2, and the fp16
     single-launch path, whose reduction is in slice order (bit-identical across variants that share S);
  5. the batched decode entry point (1-4 problems, mixed group sizes and K, the LLaMA-7B q/k/v and gate/up shapes)
     and the error contract of the batched and the per-call entry points;
  6. every token-tile instantiation of the SIMT 4-bit and the 2 / 3-bit kernels, their shared-memory K-slice caps and
     qweight with more rows than K needs;
  7. a NaN, an inf and an all-zero token next to ordinary ones on every route: the per-token scales and row sums and
     the CTA- or kernel-wide hi / lo decision must not let one token change another token's output.
Weights are drawn as uniform integers (any K, ragged last group) or as uniform packed words (the large shapes, which
are compared on a fixed sample of columns).  Shapes that depend on the SM count are computed inside the tests."""
import collections
import ctypes
import functools
import time

import numpy as np
import pytest
import torch

from gpu_util import dev, t
from oracle import gptq as ogptq
from sparsebit_b200 import _lib, launch_count, ops

pytestmark = pytest.mark.gpu
F32 = np.float32
TOL = dict(rtol=1e-5, atol=1e-5)  # the reference's bar, test_cuda_kernel.py:47
TS, TC, DECODE, SIMT, LOWBIT = "gptq4_ts_kernel", "gptq4_tc_kernel", "gptq4_decode_kernel", "gptq4_simt_kernel", "gptq_lowbit_kernel"
KERNELS = (TS, TC, DECODE, SIMT, LOWBIT)
NO_CUPTI = "CUPTI gave the profiler no kernel record for this call: the numbers were checked, the route was not asserted"


@pytest.fixture(autouse=True)
def lib():
    """The kernel switches are process-wide: every test leaves the library defaults behind, also when it fails."""
    lib = _lib.load()
    yield lib
    _lib.check(lib.sb200_gptq4_set_impl(0))
    _lib.check(lib.sb200_gptq4_set_decode(6))
    _lib.check(lib.sb200_gptq4_set_tc_drain(1))
    _lib.check(lib.sb200_gptq4_set_wait_backoff(0))


# ----------------------------------------------------------------------------- data, oracle, helpers
Case = collections.namedtuple("Case", "m k n gs seed bit frac fp16", defaults=(4, False, False))


@functools.lru_cache(maxsize=16)
def _case(c):
    """x [m, k], qweight, bias [n], scales / zeros [n, G] of a seeded problem; integer weights and integer zero points
    (``frac``: zero points with a fractional part), fp32 activations (``fp16``: fp16-representable ones).
    Callers must not modify the returned arrays (they are cached)."""
    rng = np.random.default_rng(c.seed)
    g = 1 if c.gs == 0 else -(-c.k // c.gs)
    q = rng.integers(0, 2**c.bit, (c.k, c.n))
    scales = (rng.uniform(0.5, 1.5, (c.n, g)) / (2**c.bit * np.sqrt(c.k))).astype(F32)
    zint = rng.integers(0, 2**c.bit, (c.n, g)).astype(F32)
    if c.frac:
        zint = zint + rng.uniform(0.1, 0.9, (c.n, g)).astype(F32)
    zeros = (scales * zint).astype(F32)
    x = rng.standard_normal((c.m, c.k)).astype(F32)
    if c.fp16:
        x = x.astype(np.float16).astype(F32)
    bias = (rng.standard_normal(c.n) * 0.1).astype(F32)
    return x, ogptq.pack_values(q, c.bit), bias, scales, zeros


@functools.lru_cache(maxsize=4)
def _words(k, n, bit, seed):
    """Large layers: uniformly random packed words (every nibble / bit field uniform, including the padding beyond K),
    one group, integer zero points.  Returns qweight, bias, scales, zeros."""
    rng = np.random.default_rng(seed)
    qw = rng.integers(0, 2**32, (ogptq.packed_rows(k, bit), n), dtype=np.uint32).view(np.int32)
    scales = (rng.uniform(0.5, 1.5, (n, 1)) / (2**bit * np.sqrt(k))).astype(F32)
    zeros = (scales * rng.integers(0, 2**bit, (n, 1))).astype(F32)
    bias = (rng.standard_normal(n) * 0.1).astype(F32)
    return qw, bias, scales, zeros


def _ref(x, qw, init, scales, zeros, gs, bit=4, cols=None):
    """fp64 oracle on the columns ``cols`` (default: all), 2048 columns at a time."""
    cols = np.arange(qw.shape[1]) if cols is None else np.asarray(cols)
    init = np.broadcast_to(init, (x.shape[0], qw.shape[1]))
    y = np.empty((x.shape[0], cols.size))
    for c0 in range(0, cols.size, 2048):
        c = cols[c0:c0 + 2048]
        y[:, c0:c0 + c.size] = ogptq.dequant_matmul(x, qw[:, c], init[:, c], scales[c], zeros[c], gs, bit=bit)
    return y


@functools.lru_cache(maxsize=8)
def _expected(c):
    x, qw, bias, scales, zeros = _case(c)
    return _ref(x, qw, bias, scales, zeros, c.gs, c.bit)


def _sample_cols(n, seed=0):
    """First and last 128-column blocks and 256 columns in between."""
    rng = np.random.default_rng(seed)
    return np.unique(np.concatenate([np.arange(128), np.arange(n - 128, n), rng.integers(128, n - 128, 256)]))


def _dev(a, offset=0, dtype=None):
    """Device copy of ``a`` that starts ``offset`` elements into its allocation."""
    a = np.ascontiguousarray(a)
    buf = torch.empty(a.size + offset, dtype=dtype or torch.from_numpy(a[:0]).dtype, device=dev())
    v = buf[offset:].view(a.shape)
    v.copy_(torch.from_numpy(a))
    return v


def _out(bias, m, offset=0):
    return _dev(np.tile(bias, (m, 1)), offset)


def _assert_f16(y16, exp, what=""):
    """fp16 result within 0.51 fp16 ulp of the fp64 oracle (+ 1e-5 relative for the fp32 accumulation)."""
    y = np.asarray(y16).astype(np.float64)
    ulp = np.abs(exp).astype(np.float16).astype(F32) * 2.0**-10 + 2.0**-24
    bad = ~(np.abs(y - exp) <= 0.51 * ulp + 1e-5 * (1 + np.abs(exp)))
    assert not bad.any(), f"{what}: {int(bad.sum())} fp16 outputs off by more than 0.51 ulp, first at {np.argwhere(bad)[0]}"


def _traced(fn):
    """Run ``fn`` once under torch.profiler.  Returns (result, kernel names or None if CUPTI recorded no kernel,
    library launches)."""
    torch.cuda.synchronize()
    before = launch_count()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        # a lone kernel of a few microseconds right at an edge of the trace window can be dropped from the trace:
        # keep the window a few milliseconds wider than the work on both sides
        time.sleep(0.005)
        res = fn()
        torch.cuda.synchronize()
        time.sleep(0.005)
    launches = launch_count() - before
    cuda = torch.autograd.DeviceType.CUDA
    # the raw device records: kernels launched through the C-ABI have no torch operator around them, and the
    # operator-level event list does not always keep them
    names = [e.name() for e in prof.profiler.kineto_results.events() if e.device_type() == cuda]
    names += [e.name for e in prof.events() if e.device_type == cuda]
    kernels = [nm for nm in names if "Memset" not in nm and "Memcpy" not in nm]
    return res, (kernels or None), launches


def _gptq_kernels(names):
    return {k for k in KERNELS if any(k in nm for nm in names)}


def _check_route(names, want, what):
    """Assert the GPTQ kernels launched are exactly ``want``; False when CUPTI gave no records (the caller skips after
    its numeric checks)."""
    if names is None:
        return False
    got = _gptq_kernels(names)
    print(f"route {what}: expected {sorted(want)}, launched {sorted(got)}")
    assert got == set(want), f"{what}: expected {sorted(want)}, launched {sorted(got)} ({names})"
    return True


def _decode_split(sm, per_sm, colblocks, nblk, m):
    """K blocks per slice of the decode kernel, as gptq4_decode_batch computes it: (S, S before the cap, cap)."""
    want = max(1, min(-(-sm * per_sm // colblocks), nblk))
    s = -(-nblk // want)
    cap = 8 if m <= 8 else (4 if m <= 16 else 2)
    return min(s, cap), s, cap


# ----------------------------------------------------------------------------- 1. routes
# (id, m, k, n, gs, x offset, qweight offset, out offset (4-byte elements), expected kernel)
ROUTES = [
    ("M31_below_tc_threshold-decode", 31, 512, 264, 128, 0, 0, 0, DECODE),
    ("M32_tc_threshold-tc", 32, 512, 264, 128, 0, 0, 0, TC),
    ("M767_below_ts_threshold-tc", 767, 512, 264, 128, 0, 0, 0, TC),
    ("M768_ts_threshold-ts", 768, 512, 264, 128, 0, 0, 0, TS),
    ("M300_x_misaligned-decode", 300, 512, 264, 128, 1, 0, 0, DECODE),
    ("M1000_x_misaligned-decode_multipass", 1000, 512, 264, 128, 1, 0, 0, DECODE),
    ("M40_qweight_misaligned-simt", 40, 512, 264, 128, 0, 1, 0, SIMT),
    ("M40_N_not_mult4-simt", 40, 512, 262, 128, 0, 0, 0, SIMT),
    ("M40_K_not_mult8-decode", 40, 500, 264, 0, 0, 0, 0, DECODE),
    ("M100_out_misaligned-tc_scalar_epilogue", 100, 512, 264, 128, 0, 0, 1, TC),
]


@pytest.mark.parametrize("m,k,n,gs,x_off,qw_off,out_off,want", [r[1:] for r in ROUTES], ids=[r[0] for r in ROUTES])
def test_auto_dispatch_route(m, k, n, gs, x_off, qw_off, out_off, want, request):
    c = Case(m, k, n, gs, seed=m + k + n)
    x, qw, bias, scales, zeros = _case(c)
    xd, qd, out = _dev(x, x_off), _dev(qw, qw_off), _out(bias, m, out_off)
    _, names, launches = _traced(lambda: ops.gptq4_matmul(xd, qd, out, t(scales), t(zeros), gs))
    np.testing.assert_allclose(out.cpu().numpy(), _expected(c), **TOL)
    assert launches >= 1
    if not _check_route(names, {want}, request.node.callspec.id):
        pytest.skip(NO_CUPTI)


F16_M = [1, 32, 33, 300, 767, 768, 1000]
F16_LAYOUTS = {  # k, n, gs, x offset (2-byte elements)
    "aligned": (1024, 264, 128, 0),
    "x_2byte_offset": (1024, 264, 128, 1),
    "K_not_mult8": (1020, 264, 0, 0),
    "N_not_mult4": (1024, 262, 128, 0),
}


def _f16_route(m, layout):
    """(kernel, path) sb200_gptq4_linear_f16_ex takes; path: 'single' (one launch), 'fp16_ts' (fp16 in / out, no
    staging), 'staged' (cast, bias, fp32 kernel, cast)."""
    if layout == "N_not_mult4":
        return SIMT, "staged"
    if m <= 32:
        return DECODE, "single"
    if layout == "aligned" and m >= 768:
        return TS, "fp16_ts"
    if layout == "K_not_mult8":
        return DECODE, "staged"
    return (TS if m >= 768 else TC), "staged"


@pytest.mark.parametrize("layout", list(F16_LAYOUTS))
@pytest.mark.parametrize("m", F16_M)
def test_linear_f16_route(m, layout, request):
    k, n, gs, x_off = F16_LAYOUTS[layout]
    want, path = _f16_route(m, layout)
    c = Case(m, k, n, gs, seed=3 * m + k + n, fp16=True)
    x, qw, bias, scales, zeros = _case(c)
    xd = _dev(x.astype(np.float16), x_off)
    y, names, launches = _traced(lambda: ops.gptq4_linear_f16(xd, t(qw), t(scales), t(zeros), t(bias), gs))
    y = y.cpu().numpy()
    assert y.dtype == np.float16 and y.shape == (m, n)
    _assert_f16(y, _expected(c), request.node.callspec.id)
    if path == "single":
        assert launches == 1
    elif path == "fp16_ts":
        assert launches == 3  # weight prepare, fp16 permute, persistent kernel
    else:
        assert launches >= 4  # cast, bias, kernel(s), cast
    if not _check_route(names, {want}, request.node.callspec.id):
        pytest.skip(NO_CUPTI)
    assert any("f16_to_f32_kernel" in nm for nm in names) == (path == "staged")
    assert any("gptq_permute_f16_kernel" in nm for nm in names) == (path == "fp16_ts")


# ----------------------------------------------------------------------------- 2. tcgen05 per-group kernel variants
TC_CASES = [  # test_gpu_gptq.TC_CASES
    ((1,), 128, 128, 128), ((128,), 256, 128, 128), ((130,), 512, 264, 128), ((29,), 8192, 1024, 128),
    ((4,), 6144, 768, 384), ((300,), 1024, 512, 256), ((2, 130), 512, 260, 128), ((257,), 192 * 2, 132, 128),
    ((256,), 4096, 4096, 128), ((64,), 11008, 512, 128),
]
TC_VARIANTS = [(drain, backoff) for drain in (1, 0) for backoff in (0, 64, 2000)]  # (1, 0) = the default, first


@pytest.mark.parametrize("bshape,k,n,gs", TC_CASES, ids=[f"M{int(np.prod(b))}_K{k}_N{n}_gs{g}" for b, k, n, g in TC_CASES])
def test_tc_drain_and_backoff_variants_bit_identical(bshape, k, n, gs, lib):
    """Each output element is owned by one CTA and summed in the same order whatever the TMEM drain width (.x16 or
    pairs of .x8) and the mbarrier poll back-off: the variants must agree bit for bit, and the default meets the oracle."""
    m = int(np.prod(bshape))
    x, qw, bias, scales, zeros = _case(Case(m, k, n, gs, seed=7 * k + n))
    x = x.copy()
    x[0, :5] = [3e4, -7e4, 1e-6, 0.0, 123.0]  # per-row power-of-two scaling
    if m > 2:
        x[2] *= 1e-4
    exp = _ref(x, qw, bias, scales, zeros, gs)
    xd, qd, sd, zd = t(x), t(qw), t(scales), t(zeros)
    base = None
    for drain, backoff in TC_VARIANTS:
        _lib.check(lib.sb200_gptq4_set_tc_drain(drain))
        _lib.check(lib.sb200_gptq4_set_wait_backoff(backoff))
        out = _out(bias, m)
        ops.gptq4_matmul(xd, qd, out, sd, zd, gs, impl=2)
        y = out.cpu().numpy()
        if base is None:
            base = y
            plain = [r for r in range(m) if r not in (0, 2)]
            if plain:
                np.testing.assert_allclose(y[plain], exp[plain], **TOL)
            for r in (0, 2):  # outlier rows: bounded by the row magnitude
                if r < m:
                    np.testing.assert_array_less(np.abs(y[r] - exp[r]), 1e-5 + 1e-5 * max(np.abs(exp[r]).max(), 1.0))
        else:
            np.testing.assert_array_equal(y, base, err_msg=f"drain {'.x8 pairs' if drain else '.x16'}, back-off {backoff} ns")


# ----------------------------------------------------------------------------- 3. TS persistent kernel across tiles
TS_K = [(640, 128), (704, 256)]  # 10 and 11 stages of 64 K (num_kb % 3 = 1, 2); 704 = 2 x 256 + 192: ragged last group
TS_K_IDS = ["numkb10_mod3_1-gs128", "numkb11_mod3_2-gs256_ragged"]


def _ts_shape(sm, m):
    """Feature count with a ragged last 128-feature tile such that every CTA of the persistent grid runs 2-3 tiles."""
    tiles_m = -(-m // 256)
    tiles_n = -(-5 * sm // (2 * tiles_m))  # ~2.5 tiles per SM
    n = tiles_n * 128 - 60
    tiles = tiles_m * tiles_n
    assert 2 * sm < tiles <= 3 * sm, (sm, m, tiles)
    return n


@pytest.mark.parametrize("zero_kind", ["int_zero", "frac_zero"])
@pytest.mark.parametrize("acts", ["need_lo", "fp16_exact_no_lo"])
@pytest.mark.parametrize("k,gs", TS_K, ids=TS_K_IDS)
def test_ts_persistent_multi_tile(k, gs, acts, zero_kind, lib):
    """M = 728: three token tiles, the last one ragged (728 % 256 and 728 % 16 != 0); every chunk size from one stage
    (odd chunk counts) to the default 8; all outputs against the oracle."""
    m = 728
    n = _ts_shape(lib.sb200_sm_count(), m)
    c = Case(m, k, n, gs, seed=k + n, frac=zero_kind == "frac_zero", fp16=acts == "fp16_exact_no_lo")
    x, qw, bias, scales, zeros = _case(c)
    exp = _expected(c)
    xd, qd, sd, zd = t(x), t(qw), t(scales), t(zeros)
    for chunk_k in (0, 64, 128, 192):
        out = _out(bias, m)
        ops.gptq4_matmul(xd, qd, out, sd, zd, gs, impl=3, chunk_k=chunk_k)
        np.testing.assert_allclose(out.cpu().numpy(), exp, err_msg=f"chunk_k {chunk_k}", **TOL)


@pytest.mark.parametrize("zero_kind", ["int_zero", "frac_zero"])
@pytest.mark.parametrize("k,gs", TS_K, ids=TS_K_IDS)
def test_ts_persistent_multi_tile_fp16_entry(k, gs, zero_kind, lib):
    """sb200_gptq4_linear_f16 at M = 984 (>= 768: fp16 in, fp16 bias + x @ W out from the persistent kernel), four
    token tiles, the last one ragged."""
    m = 984
    n = _ts_shape(lib.sb200_sm_count(), m)
    c = Case(m, k, n, gs, seed=2 * k + n, frac=zero_kind == "frac_zero", fp16=True)
    x, qw, bias, scales, zeros = _case(c)
    before = launch_count()
    y = ops.gptq4_linear_f16(t(x.astype(np.float16)), t(qw), t(scales), t(zeros), t(bias), gs).cpu().numpy()
    assert launch_count() - before == 3  # weight prepare, fp16 permute, persistent kernel: no fp32 staging
    _assert_f16(y, _expected(c), "fp16 TS")


# ----------------------------------------------------------------------------- 4. decode kernel modes
DEC_SHAPES = [(1000, 260, 0), (4000, 4100, 128)]  # K % 128 != 0, N % 128 != 0; the second: 2 K blocks per slice
DEC_SHAPE_IDS = ["K1000_N260_gs0", "K4000_N4100_gs128_ragged"]
DEC_M = [1, 8, 9, 16, 17, 32]  # NB = 1, 1, 2, 2, 4, 4; slab x_rows < 8 NB for 1, 9, 17
MODE_NAMES = {1: "slab", 2: "pdl", 4: "prefetch", 8: "static"}


def _mode_id(mode):
    return "mode%02d_" % mode + ("+".join(v for b, v in MODE_NAMES.items() if mode & b) or "plain")


@pytest.mark.parametrize("mode", range(16), ids=[_mode_id(md) for md in range(16)])
@pytest.mark.parametrize("m", DEC_M, ids=[f"M{m}" for m in DEC_M])
@pytest.mark.parametrize("k,n,gs", DEC_SHAPES, ids=DEC_SHAPE_IDS)
def test_decode_modes(k, n, gs, m, mode, lib):
    c = Case(m, k, n, gs, seed=13 * k + n + m)
    x, qw, bias, scales, zeros = _case(c)
    _lib.check(lib.sb200_gptq4_set_decode(mode))
    out = _out(bias, m)
    ops.gptq4_matmul(t(x), t(qw), out, t(scales), t(zeros), gs, impl=1)
    np.testing.assert_allclose(out.cpu().numpy(), _expected(c), **TOL)


@pytest.mark.parametrize("m", DEC_M, ids=[f"M{m}" for m in DEC_M])
@pytest.mark.parametrize("k,n,gs", DEC_SHAPES, ids=DEC_SHAPE_IDS)
def test_decode_modes_f16_single_launch(k, n, gs, m, lib):
    """fp16 single-launch path under all 16 variants at the default CTAs per SM: they share S, the slices' partial
    sums are added in slice order, so every variant gives the same fp16 bits."""
    c = Case(m, k, n, gs, seed=17 * k + n + m, fp16=True)
    x, qw, bias, scales, zeros = _case(c)
    args = (t(x.astype(np.float16)), t(qw), t(scales), t(zeros), t(bias), gs)
    exp = _expected(c)
    base = None
    for mode in range(16):
        _lib.check(lib.sb200_gptq4_set_decode(mode))
        before = launch_count()
        y = ops.gptq4_linear_f16(*args).cpu().numpy()
        assert launch_count() - before == 1
        if base is None:
            _assert_f16(y, exp, _mode_id(mode))
            base = y
        else:
            np.testing.assert_array_equal(y.view(np.uint16), base.view(np.uint16), err_msg=_mode_id(mode))


CAP_M = [(8, "M8_cap8"), (16, "M16_cap4"), (32, "M32_cap2")]


@pytest.mark.parametrize("m", [c[0] for c in CAP_M], ids=[c[1] for c in CAP_M])
@pytest.mark.parametrize("nibble", [1, 2, 15], ids=["1_cta_per_sm", "2_ctas_per_sm", "15_ctas_per_sm"])
def test_decode_slice_cap(nibble, m, lib):
    """The CTAs-per-SM nibble with one 128-feature block per SM and 8 * nibble + 1 K blocks: the K split wants 9 blocks
    per slice and is capped at S = 8 / 4 / 2 (8 / 16 / 32 tokens).  Register-staged and slab variants (with S = 8 every
    thread issues a slab row and all 8 block barriers are used), fp32 and fp16 single-launch; the two fp16 variants
    share S and must agree bit for bit."""
    sm = lib.sb200_sm_count()
    n = sm * 128 - 28  # one (ragged) feature block per SM
    nblk = 8 * nibble + 1
    k = nblk * 128 - 40
    s, s_uncapped, cap = _decode_split(sm, nibble, -(-n // 128), nblk, m)
    assert s == cap and s_uncapped > cap, (s, s_uncapped, cap)
    qw, bias, scales, zeros = _words(k, n, 4, nibble)
    rng = np.random.default_rng(nibble * 100 + m)
    x = rng.standard_normal((m, k)).astype(np.float16).astype(F32)  # fp16-exact: the same data for both entry points
    cols = _sample_cols(n)
    exp = _ref(x, qw, bias, scales, zeros, 0, cols=cols)
    xd, xh, qd, sd, zd, bd = t(x), t(x.astype(np.float16)), t(qw), t(scales), t(zeros), t(bias)
    y16 = {}
    for low in (6, 7):  # register-staged + pdl + prefetch; slab + pdl + prefetch
        mode = (nibble << 4) | low
        _lib.check(lib.sb200_gptq4_set_decode(mode))
        out = _out(bias, m)
        ops.gptq4_matmul(xd, qd, out, sd, zd, 0, impl=1)
        np.testing.assert_allclose(out.cpu().numpy()[:, cols], exp, err_msg=f"mode 0x{mode:02x}", **TOL)
        y16[low] = ops.gptq4_linear_f16(xh, qd, sd, zd, bd, 0).cpu().numpy()
        _assert_f16(y16[low][:, cols], exp, f"fp16 mode 0x{mode:02x}")
    np.testing.assert_array_equal(y16[6].view(np.uint16), y16[7].view(np.uint16))


# ----------------------------------------------------------------------------- 5. batched decode entry point
BATCH_PROBS = [(1536, 516, 384), (512, 132, 128), (1000, 260, 0), (1400, 388, 128)]  # K, N, gs: shorter K second


def _problem_array(problems):
    """problems: [(x, qweight, out, scales, zeros, k, n, gs)] device tensors."""
    arr = (ops._Gptq4Problem * max(1, len(problems)))()
    for i, (x, qw, out, sc, zr, k, n, gs) in enumerate(problems):
        arr[i] = ops._Gptq4Problem(x.data_ptr(), qw.data_ptr(), out.data_ptr(), sc.data_ptr(), zr.data_ptr(), k, n,
                                   qw.shape[0], gs)
    return arr


def _batch(lib, problems, m, flags, count=None):
    count = len(problems) if count is None else count
    return lib.sb200_gptq4_matmul_batch_ex(_problem_array(problems), count, m, flags, torch.cuda.current_stream().cuda_stream)


BATCH_CASES = [(cnt, m, static, mode) for cnt in (1, 2, 3, 4) for m in (1, 9, 32) for static in (0, 1) for mode in (6, 7)]


@pytest.mark.parametrize("count,m,static,mode", BATCH_CASES,
                         ids=[f"{c}probs-M{m}-{'static' if s else 'plain'}-{'slab' if md & 1 else 'regs'}" for c, m, s, md in BATCH_CASES])
def test_batch_entry_point(count, m, static, mode, lib, request):
    """1-4 problems with different K (ragged, one shorter: its CTAs beyond its K return early), group sizes 384 / 128 /
    0 (one group) per problem, one launch, every out accumulated in place."""
    _lib.check(lib.sb200_gptq4_set_decode(mode))
    probs, exps, outs = [], [], []
    for i, (k, n, gs) in enumerate(BATCH_PROBS[:count]):
        c = Case(m, k, n, gs, seed=31 * i + m)
        x, qw, bias, scales, zeros = _case(c)
        out = _out(bias, m)
        probs.append((t(x), t(qw), out, t(scales), t(zeros), k, n, gs))
        outs.append(out)
        exps.append(_expected(c))
    rc, names, launches = _traced(lambda: _batch(lib, probs, m, static))
    _lib.check(rc)
    assert launches == 1
    for i, (o, e) in enumerate(zip(outs, exps)):
        np.testing.assert_allclose(o.cpu().numpy(), e, err_msg=f"problem {i}", **TOL)
    if not _check_route(names, {DECODE}, request.node.callspec.id):
        pytest.skip(NO_CUPTI)


LLAMA = {"qkv": [(4096, 4096)] * 3, "gate_up": [(4096, 11008)] * 2}


@pytest.mark.parametrize("m", [1, 32], ids=["M1", "M32"])
@pytest.mark.parametrize("layer", list(LLAMA))
def test_batch_llama7b_shapes(layer, m, lib, request):
    """The batched launches the benchmark times: q / k / v (3 x 4096 x 4096) and gate / up (2 x 4096 x 11008), int4
    g128, static weights."""
    rng = np.random.default_rng(m)
    x = rng.standard_normal((m, 4096)).astype(F32)
    xd = t(x)
    probs, exps, outs = [], [], []
    for i, (k, n) in enumerate(LLAMA[layer]):
        qw, bias, scales, zeros = _words(k, n, 4, 1000 + i)
        g = k // 128
        scales = np.repeat(scales, g, axis=1) * rng.uniform(0.8, 1.2, (n, g)).astype(F32)
        zeros = (scales * rng.integers(0, 16, (n, g))).astype(F32)
        out = _out(bias, m)
        probs.append((xd, t(qw), out, t(scales), t(zeros), k, n, 128))
        outs.append(out)
        exps.append(_ref(x, qw, bias, scales, zeros, 128))
    rc, names, launches = _traced(lambda: _batch(lib, probs, m, ops.GPTQ4_STATIC_WEIGHTS))
    _lib.check(rc)
    assert launches == 1
    for i, (o, e) in enumerate(zip(outs, exps)):
        np.testing.assert_allclose(o.cpu().numpy(), e, err_msg=f"problem {i}", **TOL)
    if not _check_route(names, {DECODE}, request.node.callspec.id):
        pytest.skip(NO_CUPTI)


def _err_problems(m=4, n=132, qw_off=0):
    x, qw, bias, scales, zeros = _case(Case(m, 256, 132, 128, seed=5))
    qd = _dev(qw, qw_off)
    if n != 132:
        qd = torch.zeros(qw.shape[0], n, dtype=torch.int32, device=dev())
    out = _out(np.zeros(n, F32), m)
    return [(t(x), qd, out, t(scales), t(zeros), 256, n, 128)], out


BATCH_ERRORS = {  # id: (problems kwargs, count, m, flags, message)
    "count0": ({}, 0, 4, 0, "1 .. 4 problems"),
    "count5": ({}, 5, 4, 0, "1 .. 4 problems"),
    "m0": ({}, None, 0, 0, "decode-sized M only"),
    "m33": ({}, None, 33, 0, "decode-sized M only"),
    "N_not_mult4": ({"n": 130}, None, 4, 0, "N % 4 == 0"),
    "qweight_misaligned": ({"qw_off": 1}, None, 4, 0, "16-byte aligned qweight"),
    "unknown_flag": ({}, None, 4, 2, "unknown flags"),
}


@pytest.mark.parametrize("case", list(BATCH_ERRORS))
def test_batch_error_contract(case, lib):
    kw, count, m, flags, msg = BATCH_ERRORS[case]
    probs, out = _err_problems(**kw)
    if count == 5:
        probs = probs * 5
    before = out.clone()
    rc = _batch(lib, probs, m, flags, count)
    assert rc != 0
    assert msg in lib.sb200_last_error().decode()
    torch.cuda.synchronize()
    assert torch.equal(out, before)  # nothing launched


MATMUL_EX_ERRORS = {  # id: (options (impl, chunk_k, flags, reserved[0]), x offset, message)
    "impl5": ((5, 0, 0, 0), 0, "impl must be 0"),
    "chunk_k_not_mult64": ((3, 96, 0, 0), 0, "chunk_k must be a multiple of 64"),
    "reserved_nonzero": ((0, 0, 0, 1), 0, "reserved option fields must be zero"),
    "unknown_flag": ((0, 0, 4, 0), 0, "unknown flags"),
    "impl2_forced_x_misaligned": ((2, 0, 0, 0), 1, "tcgen05 path forced but shape/workspace unsupported"),
    "impl3_forced_x_misaligned": ((3, 0, 0, 0), 1, "tcgen05 path forced but shape/workspace unsupported"),
}


@pytest.mark.parametrize("case", list(MATMUL_EX_ERRORS))
def test_matmul_ex_error_contract(case, lib):
    (impl, chunk_k, flags, res0), x_off, msg = MATMUL_EX_ERRORS[case]
    m, k, n, gs = 64, 512, 264, 128
    x, qw, bias, scales, zeros = _case(Case(m, k, n, gs, seed=9))
    xd, qd, sd, zd, out = _dev(x, x_off), t(qw), t(scales), t(zeros), _out(bias, m)
    before = out.clone()
    ws_bytes = int(lib.sb200_gptq4_workspace_bytes(m, k, n, gs))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev())
    opts = ops._Gptq4Options(impl, chunk_k, flags)
    opts.reserved[0] = res0
    rc = lib.sb200_gptq4_matmul_ex(xd.data_ptr(), qd.data_ptr(), out.data_ptr(), sd.data_ptr(), zd.data_ptr(), m, k, n,
                                   qw.shape[0], gs, ctypes.byref(opts), ws.data_ptr(), ws_bytes,
                                   torch.cuda.current_stream().cuda_stream)
    assert rc != 0
    assert msg in lib.sb200_last_error().decode()
    torch.cuda.synchronize()
    assert torch.equal(out, before)


# ----------------------------------------------------------------------------- 6. SIMT 4-bit and low-bit tiles
TILE_M = [1, 2, 3, 4, 5, 6, 7, 8, 9, 15, 16, 17, 33]  # MT = 1, 2, 4, 4, 8 ...: partial 8-token tiles and several passes


def _run_scalar(bit, x, qw, bias, scales, zeros, gs):
    out = _out(bias, x.shape[0])
    if bit == 4:
        ops.gptq4_matmul(t(x), t(qw), out, t(scales), t(zeros), gs, impl=4)
    else:
        ops.gptq_matmul(t(x), t(qw), out, t(scales), t(zeros), bit, gs)
    return out.cpu().numpy()


@pytest.mark.parametrize("m", TILE_M, ids=[f"M{m}" for m in TILE_M])
@pytest.mark.parametrize("bit", [4, 2, 3], ids=["simt4", "lowbit2", "lowbit3"])
def test_scalar_kernel_token_tiles(bit, m):
    c = Case(m, 1000, 300, 128, seed=bit * 100 + m, bit=bit)  # ragged K block, group and feature block
    x, qw, bias, scales, zeros = _case(c)
    np.testing.assert_allclose(_run_scalar(bit, x, qw, bias, scales, zeros, 128), _expected(c), **TOL)


@pytest.mark.parametrize("bit", [4, 2, 3], ids=["simt4", "lowbit2", "lowbit3"])
def test_scalar_kernel_extra_qweight_rows(bit):
    """qweight with more rows than K needs (random words): the rows beyond K contribute nothing."""
    m = 9
    c = Case(m, 1000, 300, 128, seed=bit * 100 + m, bit=bit)
    x, qw, bias, scales, zeros = _case(c)
    extra = np.random.default_rng(bit).integers(0, 2**32, (6, qw.shape[1]), dtype=np.uint32).view(np.int32)
    y = _run_scalar(bit, x, np.concatenate([qw, extra]), bias, scales, zeros, 128)
    np.testing.assert_allclose(y, _expected(c), **TOL)


@pytest.mark.parametrize("bit", [4, 2, 3], ids=["simt4_cap8", "lowbit2_cap16", "lowbit3_cap8"])
def test_scalar_kernel_slice_cap(bit, lib):
    """8 x SMs feature blocks: the K split wants one slice per column block and the shared-memory cap on the K blocks
    per slice applies (8 for the 4-bit kernel, 1024 / block K for 2 / 3-bit).  Compared on a column sample."""
    sm = lib.sb200_sm_count()
    n, k, m = 8 * sm * 128, 1208, 9
    block_k = {4: 128, 2: 64, 3: 128}[bit]
    cap = 8 if bit == 4 else 1024 // block_k
    nblk = -(-k // block_k)
    want = max(1, min(-(-sm * 8 // (n // 128)), nblk))
    assert want == 1 and -(-nblk // want) > cap
    qw, bias, scales, zeros = _words(k, n, bit, 7)
    x = np.random.default_rng(bit).standard_normal((m, k)).astype(F32)
    cols = _sample_cols(n)
    y = _run_scalar(bit, x, qw, bias, scales, zeros, 0)
    np.testing.assert_allclose(y[:, cols], _ref(x, qw, bias, scales, zeros, 0, bit=bit, cols=cols), **TOL)


# ----------------------------------------------------------------------------- 7. non-finite token isolation
NONFINITE_ROUTES = {  # id: (m, k, n, gs, bit, runner)
    "ts": (40, 512, 264, 128, 4, "impl3"),
    "tc": (40, 512, 264, 128, 4, "impl2"),
    "decode_regs": (12, 1000, 260, 0, 4, "decode6"),
    "decode_slab": (12, 1000, 260, 0, 4, "decode7"),
    "simt": (12, 1000, 300, 128, 4, "impl4"),
    "lowbit2": (12, 1000, 300, 128, 2, "lowbit"),
    "lowbit3": (12, 1000, 300, 128, 3, "lowbit"),
    "f16_single_launch": (12, 1000, 260, 0, 4, "f16"),
    "f16_ts": (800, 512, 264, 128, 4, "f16"),
}


@pytest.mark.parametrize("route", list(NONFINITE_ROUTES))
def test_nonfinite_token_isolation(route, lib):
    """Token 0 holds a NaN, token 1 a +inf, token 2 is all zeros: tokens 0 and 1 give non-finite outputs everywhere,
    token 2 gives exactly its initial out (the bias), every other token is untouched by its neighbours."""
    m, k, n, gs, bit, runner = NONFINITE_ROUTES[route]
    f16 = runner == "f16"
    c = Case(m, k, n, gs, seed=m + k + bit, bit=bit, fp16=f16)
    x, qw, bias, scales, zeros = _case(c)
    x = x.copy()
    x[0, 5] = np.nan
    x[1, 7] = np.inf
    x[2] = 0.0
    if f16:
        want = {"f16_single_launch": DECODE, "f16_ts": TS}[route]
        _lib.check(lib.sb200_gptq4_set_decode(6))
        y, names, _ = _traced(lambda: ops.gptq4_linear_f16(t(x.astype(np.float16)), t(qw), t(scales), t(zeros), t(bias), gs))
        y = y.cpu().numpy()
        assert not np.isfinite(y[:2]).any()
        np.testing.assert_array_equal(y[2].view(np.uint16), bias.astype(np.float16).view(np.uint16))
        _assert_f16(y[3:], _ref(x[3:], qw, bias, scales, zeros, gs), route)
    else:
        out = _out(bias, m)
        xd, qd, sd, zd = t(x), t(qw), t(scales), t(zeros)
        if runner == "lowbit":
            want = LOWBIT
            fn = lambda: ops.gptq_matmul(xd, qd, out, sd, zd, bit, gs)  # noqa: E731
        elif runner.startswith("decode"):
            want = DECODE
            _lib.check(lib.sb200_gptq4_set_decode(int(runner[-1])))
            fn = lambda: ops.gptq4_matmul(xd, qd, out, sd, zd, gs, impl=1)  # noqa: E731
        else:
            impl = int(runner[-1])
            want = {2: TC, 3: TS, 4: SIMT}[impl]
            fn = lambda: ops.gptq4_matmul(xd, qd, out, sd, zd, gs, impl=impl)  # noqa: E731
        _, names, _ = _traced(fn)
        y = out.cpu().numpy()
        assert not np.isfinite(y[:2]).any(), f"{np.isfinite(y[:2]).sum()} finite outputs in the NaN / inf tokens"
        np.testing.assert_array_equal(y[2], bias)
        np.testing.assert_allclose(y[3:], _ref(x[3:], qw, bias, scales, zeros, gs, bit=bit), **TOL)
    if not _check_route(names, {want}, route):
        pytest.skip(NO_CUPTI)
