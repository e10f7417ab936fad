"""Every dispatch branch of the fake-quant forward, the STE backward and the PACT clamp backward vs the numpy oracle.

Each streaming entry point picks a kernel or template instantiation from pointer alignment, channel count, row length,
rounding mode and size.  The tests below reach each branch on purpose (the case ids name it) and compare bit for bit:
  * forward: per-tensor LDG / TMA with and without fused statistics, per-channel with the shared-memory parameter table
    (C <= 2048) and without it, the channel-last column kernel, the mask-fused per-channel kernel and QdqMulti;
  * backward: the per-tensor head / scalar paths, row tiles (warp and CTA tiles, several tiles per row) and the
    channel-last kernel with many row blocks.
The forward inputs are near-tie data (``near_tie_values``): quotients x / s within a few ulp of a rounding midpoint,
where a reciprocal multiply or a broken exact fallback rounds to a different integer, and odd quotients in
[2^22, 2^24), which the 1.5 * 2^23 rounding trick moves to an even neighbour.  With qmin / qmax = -+2^24 clamping
cannot hide a wrong rounding."""
import numpy as np
import pytest
import torch

from gpu_util import bits_equal, dev, t
from oracle import qdq as oqdq
from sparsebit_b200 import _lib, ops

F32 = np.float32
GATE = F32(2.0**-60)  # smallest |scale| the fp32 fast path of quant_round accepts (common.cuh QP::set)
SPECIALS = np.array([3e38, -3e38, 1e-40, -1e-40, 1e-45, -1e-45, 0.0, -0.0, np.inf, -np.inf, np.nan], F32)


def near_tie_scales(rng, n_random=40):
    """Random scales in [1e-4, 10], 0.1, 1/3, and 2^-60 with its fp32 neighbours on both sides of the fast-path gate."""
    fixed = [F32(0.1), F32(1) / F32(3), GATE, np.nextafter(GATE, F32(0)), np.nextafter(GATE, F32(1))]
    return np.concatenate([rng.uniform(1e-4, 10, n_random).astype(F32), np.array(fixed, F32)])


def near_tie_values(s, rng):
    """Inputs for the per-element scales ``s``; returns (x, kind), both shaped like s.
    kind 0: RN32((k + 1/2) s) +- 0..4 ulp, |k| log-uniform up to 2^21 + 2;  kind 1: the same around k = 2^22;
    kind 2: RN32(k s) for odd k in [2^22, 2^24);  kind 3: quotient overflow, denormals, +-0, +-inf, NaN."""
    s = np.asarray(s, F32)
    shape, s = s.shape, s.reshape(-1)
    n = s.size
    kind = rng.choice(4, size=n, p=[0.70, 0.10, 0.15, 0.05])
    sign = np.where(rng.random(n) < 0.5, -1.0, 1.0)
    k = np.floor(np.exp2(rng.uniform(-1.0, np.log2(2.0**21 + 3), n)))
    k = np.where(kind == 1, 2.0**22 + rng.integers(-8, 9, n), k)
    s64 = s.astype(np.float64)
    x = (sign * (k + 0.5) * s64).astype(F32)  # (k + 1/2) * s is exact in fp64: one rounding to fp32
    x = (x.view(np.int32) + rng.integers(-4, 5, n).astype(np.int32)).view(F32)  # +- ulps (x is never near 0 or inf)
    odd = (2 * rng.integers(2**21, 2**23, n) + 1).astype(np.float64)
    x = np.where(kind == 2, (sign * odd * s64).astype(F32), x)
    x = np.where(kind == 3, rng.choice(SPECIALS, n), x).astype(F32)
    return x.reshape(shape), kind.reshape(shape)


TIE_SCALES = near_tie_scales(np.random.default_rng(2024))
WIDE = 1 << 24


def _ranges(c, rng):
    """(qmin, qmax, zero_point[c]): int8 symmetric, uint8 with half-integer zero points (rounded by the kernel), and the
    wide range in which nothing clamps."""
    z_u8 = (rng.integers(0, 256, c) + rng.choice([0.0, 0.5], c)).astype(F32)
    return [(-128, 127, np.zeros(c, F32)), (0, 255, z_u8), (-WIDE, WIDE, rng.integers(-50, 51, c).astype(F32))]


def _dev(a, offset=0, dtype=torch.float32):
    """Device copy of ``a`` that starts ``offset`` elements into its allocation (offset 1: 4-byte aligned floats)."""
    a = np.ascontiguousarray(a)
    buf = torch.empty(a.size + offset, dtype=dtype, device=dev())
    v = buf[offset:].view(a.shape)
    v.copy_(torch.from_numpy(a))
    return v


def _empty(shape, offset=0):
    return torch.empty(int(np.prod(shape)) + offset, dtype=torch.float32, device=dev())[offset:].view(shape)


def _chan_scales(shape, ch_axis):
    c = shape[ch_axis]
    s = TIE_SCALES[np.arange(c) % TIE_SCALES.size]
    b = [1] * len(shape)
    b[ch_axis] = c
    return s, np.broadcast_to(s.reshape(b), shape)


# ------------------------------------------------------------------------------------------------ generator self-check
def test_near_tie_inputs_have_teeth():
    """The data must separate a correct quotient from the shortcuts the fast path avoids."""
    rng = np.random.default_rng(1)
    s = np.repeat(TIE_SCALES, 4000)
    x, kind = near_tie_values(s, rng)
    with np.errstate(all="ignore"):
        exact = np.rint(x / s)
        recip = np.rint(x * (F32(1) / s))
        trick = (x / s + F32(12582912)) - F32(12582912)  # rint by the 1.5 * 2^23 trick, fp32
    tie = kind <= 1
    assert np.mean(exact[tie] != recip[tie]) >= 0.01  # reciprocal multiply rounds >= 1 % of them differently
    q = x[tie].astype(np.float64) / s[tie].astype(np.float64)
    assert np.mean(0.5 - np.abs(q - np.rint(q)) <= np.abs(q) * 2.0**-22) >= 0.3  # quant_round's exact-fallback window
    big = kind == 2
    assert np.all(np.abs(exact[big]) >= 2**22) and np.mean(trick[big] != exact[big]) >= 0.3
    assert np.isin(SPECIALS.view(np.int32), x.view(np.int32)).all()
    assert (TIE_SCALES < GATE).sum() == 1 and (TIE_SCALES == GATE).sum() == 1 and (TIE_SCALES > GATE).sum() > 1


# ------------------------------------------------------------------------------------------------ forward
@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("variant", [1, 2])
def test_pertensor_near_ties_ldg_tma_and_fused_stats(variant, offset):
    """sb200_set_variant 1 = LDG register pipeline, 2 = TMA ring (16-byte aligned only; offset 1 takes the scalar LDG
    instantiation), each with and without the fused MinMax; n % 4 == 3 exercises the scalar tail."""
    lib = _lib.load()
    rng = np.random.default_rng(10 * variant + offset)
    n = 4 * 4096 * 2 + 7  # TMA serves n >= 4 tiles of 4096
    assert lib.sb200_set_variant(variant) == 0
    try:
        for s in TIE_SCALES:
            x, _ = near_tie_values(np.full(n, s, F32), rng)
            xt = _dev(x, offset)
            for qmin, qmax, z in _ranges(1, rng):
                exp = oqdq.qdq(x, np.float32([s]), z, qmin, qmax)
                y = ops.qdq_pertensor(xt, t(np.float32([s])), t(z), qmin, qmax, out=_empty(n, offset))
                assert bits_equal(y.cpu().numpy(), exp), (s, qmin)
                st = ops.minmax_new(1, dev())
                y2 = ops.qdq_stats_pertensor(xt, t(np.float32([s])), t(z), qmin, qmax, st, out=_empty(n, offset))
                assert bits_equal(y2.cpu().numpy(), exp), (s, qmin)
                mn, mx = ops.minmax_read(st)
                assert bits_equal(mn.cpu().numpy(), [np.min(x)]) and bits_equal(mx.cpu().numpy(), [np.max(x)])
    finally:
        lib.sb200_set_variant(0)


PERCHANNEL_ROUTES = [
    pytest.param((4, 1000, 49), 1, id="table-inner49"),
    pytest.param((2, 2048, 301), 1, id="table-C2048"),
    pytest.param((3072, 768), 0, id="notable-deit-fc1"),
    pytest.param((3, 2049, 5), 1, id="notable-C2049-tail3"),
    pytest.param((50, 3072, 3), 1, id="notable-C3072-inner3"),
    pytest.param((30, 4096, 2), 1, id="notable-C4096-inner2"),
    pytest.param((300, 768), 1, id="cols-C768"),
    pytest.param((301, 50), 1, id="cols-C50"),
]
_inputs = {}


def _perchannel_inputs(shape, ch_axis):
    """Near-tie data for channel c's scale TIE_SCALES[c % len]; cached per shape (the oracle side is the slow part)."""
    key = (shape, ch_axis)
    if key not in _inputs:
        s, se = _chan_scales(shape, ch_axis)
        _inputs[key] = (s, near_tie_values(se, np.random.default_rng(sum(shape)))[0])
    return _inputs[key]


@pytest.mark.gpu
@pytest.mark.parametrize("rounding", [0, 1, 2])
@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("shape,ch_axis", PERCHANNEL_ROUTES)
def test_perchannel_forward_routes(shape, ch_axis, offset, rounding):
    """Sizes span several grid strides with outer * C * inner not a multiple of the stride, so the channel cursor wraps;
    C > 2048 has no shared-memory table and reloads the parameters whenever the channel changes."""
    s, x = _perchannel_inputs(shape, ch_axis)
    rng = np.random.default_rng(rounding)
    xt = _dev(x, offset)
    for qmin, qmax, z in _ranges(s.size, rng):
        y = ops.qdq_perchannel(xt, t(s), t(z), qmin, qmax, ch_axis, rounding, out=_empty(shape, offset))
        assert bits_equal(y.cpu().numpy(), oqdq.qdq(x, s, z, qmin, qmax, ch_axis, rounding)), qmin


@pytest.mark.gpu
@pytest.mark.parametrize("rounding", [0, 1, 2])
@pytest.mark.parametrize("x_off,m_off", [(0, 0), (0, 1), (1, 3)])
@pytest.mark.parametrize("shape,ch_axis", [((3, 2049, 5), 1), ((16, 1000, 9), 1), ((40, 768), 1), ((7, 1, 5), 1)])
def test_mask_apply_qdq_perchannel_offset_mask(shape, ch_axis, x_off, m_off, rounding):
    """Sparser mask-apply fused into the per-channel QDQ: an unaligned mask (or x) takes the scalar instantiation,
    inner == 1 stays on the channel-row kernel, C == 1 on the per-tensor one."""
    s, x = _perchannel_inputs(shape, ch_axis)
    rng = np.random.default_rng(x_off + 3 * m_off)
    m = rng.random(shape) < 0.7
    xt, mt = _dev(x, x_off), _dev(m, m_off, torch.bool)
    with np.errstate(all="ignore"):
        xm = (x * m.astype(F32)).astype(F32)
    for qmin, qmax, z in _ranges(s.size, rng):
        y = ops.mask_apply_qdq_perchannel(xt, mt, t(s), t(z), qmin, qmax, ch_axis, rounding, out=_empty(shape, x_off))
        assert bits_equal(y.cpu().numpy(), oqdq.qdq(xm, s, z, qmin, qmax, ch_axis, rounding)), qmin


@pytest.mark.gpu
def test_qdq_multi_hundreds_of_descriptors():
    """300 tensors in one plan: ch_axis 0 / 1 / -1, rows of 1 - 3 elements next to 16-byte aligned rows of 768, tensors
    packed back to back in one buffer (most rows unaligned), half of them masked, 8-bit and wide ranges."""
    rng = np.random.default_rng(7)
    shapes = [((int(rng.integers(1, 40)), 1), 0), ((int(rng.integers(1, 40)), 2), 0), ((int(rng.integers(1, 40)), 3), 0),
              ((2, int(rng.integers(1, 30)), 3), 1), ((3, int(rng.integers(1, 30))), -1), ((int(rng.integers(1, 9)), 768), 0),
              ((2, int(rng.integers(1, 9)), 5, 5), 1)]
    specs = [shapes[i % len(shapes)] for i in range(300)]
    total = sum(int(np.prod(sh)) + 4 for sh, _ in specs)
    buf = torch.empty(total, dtype=torch.float32, device=dev())
    items, expected, off = [], [], 0
    for i, (shape, ch_axis) in enumerate(specs):
        if shape[-1] == 768:
            off = (off + 3) // 4 * 4  # keep the long rows 16-byte aligned (vector path)
        c = shape[ch_axis]
        s = TIE_SCALES[rng.integers(0, TIE_SCALES.size, c)]
        b = [1] * len(shape)
        b[ch_axis] = c
        x, _ = near_tie_values(np.broadcast_to(s.reshape(b), shape), rng)
        qmin, qmax, z = _ranges(c, rng)[i % 3]
        xv = buf[off:off + x.size].view(shape)
        xv.copy_(torch.from_numpy(x))
        off += x.size
        item = dict(x=xv, scale=t(s), zero_point=t(z), qmin=qmin, qmax=qmax, ch_axis=ch_axis)
        xm = x
        if i % 2:
            m = rng.random(shape) < 0.6
            item["mask"] = t(m)
            with np.errstate(all="ignore"):
                xm = (x * m.astype(F32)).astype(F32)
        items.append(item)
        expected.append(oqdq.qdq(xm, s, z, qmin, qmax, ch_axis % len(shape)))
    plan = ops.QdqMulti(items)
    for _ in range(2):  # run() re-reads the tensors: same result twice
        outs = plan.run()
        for i, (y, e) in enumerate(zip(outs, expected)):
            assert bits_equal(y.cpu().numpy(), e), (i, specs[i])


# ------------------------------------------------------------------------------------------------ STE backward
BWD_CASES = [
    pytest.param((100_003,), None, id="pertensor"),
    pytest.param((3, 4, 128, 100), 1, id="rows-2tiles"),
    pytest.param((2, 8, 1023), 1, id="rows-warp-tile-1023"),
    pytest.param((2, 8, 1024), 1, id="rows-cta-tile-1024"),
    pytest.param((8, 197, 768), 2, id="cols-768-64thr"),
    pytest.param((8, 197, 512), 2, id="cols-512-128thr"),
    pytest.param((2000, 50), 1, id="cols-50-scalar"),
]


def _bwd_inputs(shape, ch_axis, qmin, qmax, rng):
    c = 1 if ch_axis is None else shape[ch_axis]
    s = rng.uniform(0.005, 0.05, c).astype(F32)
    z = rng.integers(-3, 4, c).astype(F32)
    b = [1] * len(shape)
    if ch_axis is not None:
        b[ch_axis] = c
    se, ze = np.broadcast_to(s.reshape(b), shape), np.broadcast_to(z.reshape(b), shape)
    x, _ = near_tie_values(se, rng)
    # a fifth of the elements exactly on vq == qmin / vq == qmax (the inside / clipped boundary of both gzp rules)
    edge = rng.random(shape)
    x = np.where(edge < 0.1, ((qmin - ze) * se).astype(F32), x)
    x = np.where(edge > 0.9, ((qmax - ze) * se).astype(F32), x).astype(F32)
    gy = rng.standard_normal(shape).astype(F32)
    return x, gy, s, z


def _assert_sum(got, terms, axes, what):
    ref = terms.sum(axis=axes).reshape(-1)
    l1 = np.abs(terms).sum(axis=axes).reshape(-1)
    err = np.abs(got.cpu().numpy().astype(np.float64).reshape(-1) - ref)
    assert np.all(err <= 1e-5 * l1 + 1e-30), (what, float(np.max(err / (l1 + 1e-30))))


@pytest.mark.gpu
@pytest.mark.parametrize("offsets", [(0, 0, 0), (1, 1, 1), (1, 0, 2)], ids=["aligned", "head", "mismatched"])
@pytest.mark.parametrize("rounding", [0, 1, 2])
@pytest.mark.parametrize("shape,ch_axis", BWD_CASES)
def test_ste_backward_routes(shape, ch_axis, rounding, offsets):
    """gx bit-exact, gs / gzp within 1e-5 of the L1 norm of their fp64 terms, identical bits on a second run, and
    need_gs / need_gzp alone give the same values.  Offsets (x, gy, gx) in floats: all shifted alike take the
    vector path after a scalar head, mismatched ones the scalar path."""
    qmin, qmax = (-16, 15) if rounding else (-128, 127)
    rng = np.random.default_rng(sum(shape) + rounding)
    x, gy, s, z = _bwd_inputs(shape, ch_axis, qmin, qmax, rng)
    xt, gyt = _dev(x, offsets[0]), _dev(gy, offsets[1])
    rules = [False] if ch_axis is None else [False, True]
    axes = None if ch_axis is None else tuple(a for a in range(len(shape)) if a != ch_axis)
    for closed in rules:
        egx, gs_e, gz_e = oqdq.ste_backward_terms(x, s, z, gy, qmin, qmax, ch_axis or 0, rounding,
                                                  gzp_open_top=ch_axis is not None and not closed)

        def run(need_gs=True, need_gzp=True):
            return ops.qdq_backward(xt, t(s), t(z), gyt, qmin, qmax, ch_axis, rounding, need_gs, need_gzp, closed,
                                    out=_empty(shape, offsets[2]))

        gx, gs, gzp = run()
        assert bits_equal(gx.cpu().numpy(), egx), closed
        _assert_sum(gs, gs_e, axes, "gs")
        _assert_sum(gzp, gz_e, axes, "gzp")
        gx2, gs2, gzp2 = run()
        assert torch.equal(gx, gx2) and torch.equal(gs, gs2) and torch.equal(gzp, gzp2)
        _, gs3, gzp3 = run(need_gzp=False)
        assert torch.equal(gs3, gs) and not gzp3.any()
        _, gs4, gzp4 = run(need_gs=False)
        assert torch.equal(gzp4, gzp) and not gs4.any()
    assert 0 < np.count_nonzero(egx) < egx.size  # both inside and clipped elements


# ------------------------------------------------------------------------------------------------ PACT clamp backward
@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("n", [1, 3, 4097, 5_000_003])
def test_clamp_backward_vector_scalar_and_bounds(n, offset):
    """x exactly on lo and hi passes its gradient to x (closed interval), never to the bounds."""
    rng = np.random.default_rng(n + offset)
    lo, hi = F32(-1.25), F32(0.75)
    x = (rng.standard_normal(n) * 1.2).astype(F32)
    x[0] = hi
    x[1::7] = lo
    x[2::5] = hi
    gy = rng.standard_normal(n).astype(F32)
    gx, g_hi, g_lo = ops.clamp_backward(_dev(x, offset), _dev(gy, offset), t(np.float32([lo])), t(np.float32([hi])))
    egx, e_hi, e_lo = oqdq.clamp_backward(x, gy, lo, hi)
    assert bits_equal(gx.cpu().numpy(), egx)
    g64 = np.abs(gy.astype(np.float64))
    assert abs(float(g_hi) - e_hi) <= 1e-6 * g64[x > hi].sum()
    assert abs(float(g_lo) - e_lo) <= 1e-6 * g64[x < lo].sum()
