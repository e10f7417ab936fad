"""Every dispatch branch of the observer reductions vs the numpy oracle: MinMax qparams of many quantizers in one
launch, the per-channel MinMax regimes, radix select / percentile (segment sizes, many rows, several tensors, keys that
share their high bits), the MSE sweep and row moments over rows of many tiles, and the histogram's scalar path.
Order statistics, min / max and histogram counts are exact; float sums are compared at a stated relative bound."""
import numpy as np
import pytest
import torch

from gpu_util import bits_equal, dev, t
from oracle import observers as oobs
from oracle import qdq as oqdq
from sparsebit_b200 import _lib, ops
from sparsebit_b200._lib import SparsebitB200Error

F32 = np.float32


def _dev(a, offset=0):
    """Device copy of ``a`` that starts ``offset`` floats into its allocation (offset 1: 4-byte aligned)."""
    a = np.ascontiguousarray(a, F32)
    buf = torch.empty(a.size + offset, dtype=torch.float32, device=dev())
    v = buf[offset:].view(a.shape)
    v.copy_(torch.from_numpy(a))
    return v


# ------------------------------------------------------------------------------------------------ MinMax qparams
def _channel_rows(c, rng):
    """[c, 5] rows cycling through: mixed sign, all positive, all negative, all zero, one NaN, -inf and +inf."""
    x = (rng.standard_normal((c, 5)) * rng.uniform(1e-3, 50, (c, 1))).astype(F32)
    flavour = np.arange(c) % 6
    x[flavour == 1] = np.abs(x[flavour == 1]) + F32(0.01)
    x[flavour == 2] = -np.abs(x[flavour == 2]) - F32(0.01)
    x[flavour == 3] = 0.0
    x[flavour == 4, 2] = np.nan
    x[flavour == 5, 0] = -np.inf
    x[flavour == 5, 4] = np.inf
    return x


@pytest.mark.gpu
def test_minmax_qparams_multi_vs_oracle():
    """300 quantizers in one launch; channel counts 1, 127, 128, 129 and 5000 cover the 128-thread loop."""
    rng = np.random.default_rng(3)
    chans = [1, 127, 128, 129, 5000] + [int(v) for v in rng.integers(1, 60, 295)]
    ranges = [(-128, 127), (0, 255), (-8, 7), (0, 15)]
    requests, expected = [], []
    for i, c in enumerate(chans):
        x = _channel_rows(c, rng)
        if c == 1:
            x[0] = [-3.0, 1.0, 0.5, 2.0, -0.25]
        st = ops.minmax_new(c, dev())
        ops.minmax_update(t(x), st, ch_axis=0)
        qmin, qmax = ranges[i % 4]
        sym = (i // 4) % 2 == 0
        requests.append((st, qmin, qmax, sym))
        mn, mx = oobs.minmax([x], per_channel=True, ch_axis=0)
        s, z = oobs.calc_qparams_with_minmax(mn, mx, qmin, qmax, sym)
        expected.append((mn, mx, s, z))
    outs = ops.minmax_qparams_multi(requests)
    for i, (got, exp) in enumerate(zip(outs, expected)):
        for name, g, e in zip(("min", "max", "scale", "zero_point"), got, exp):
            assert bits_equal(g.cpu().numpy(), e), (i, chans[i], name)
    assert np.isnan(expected[1][2]).any() and (expected[1][2] == F32(1e-6)).any()  # NaN channel, 1e-6 scale floor


# ------------------------------------------------------------------------------------------------ per-channel MinMax
MINMAX_CASES = [pytest.param((3, 37, inner), 1, id=f"inner{inner}") for inner in (2, 3, 4, 63, 64, 65, 4095, 4096, 8193)]
MINMAX_CASES += [pytest.param((300, c), 1, id=f"cols-C{c}") for c in (4, 5, 768)]


@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("shape,ch_axis", MINMAX_CASES)
def test_minmax_perchannel_regimes_and_alignment(shape, ch_axis, offset):
    """inner <= 64: rows staged in shared memory; 64 < inner < 4096: a warp per 4 rows (vector loads only when inner % 4
    == 0 and x is aligned); inner >= 4096: CTA tiles; inner == 1: the channel-last kernel.  One NaN poisons its channel
    and no other."""
    rng = np.random.default_rng(sum(shape) + offset)
    x = (rng.standard_normal(shape) * 3).astype(F32)
    idx = list(np.array(shape) // 2)
    x[tuple(idx)] = np.nan
    st = ops.minmax_new(shape[ch_axis], dev())
    ops.minmax_update(_dev(x, offset), st, ch_axis)
    mn, mx = ops.minmax_read(st)
    emn, emx = oobs.minmax([x], per_channel=True, ch_axis=ch_axis)
    assert bits_equal(mn.cpu().numpy(), emn) and bits_equal(mx.cpu().numpy(), emx)
    assert np.isnan(mn.cpu().numpy()).sum() == 1 and np.isnan(mx.cpu().numpy()).sum() == 1


# ------------------------------------------------------------------------------------------------ radix select
def _select(rows, ranks, tensors, ntpr=1):
    rs = ops.RadixSelect(rows, ntpr, dev())
    rs.set_ranks(torch.tensor(ranks, dtype=torch.int64, device=dev()))
    for p in range(3):
        for x2 in tensors:
            rs.hist_pass(p, x2)
        rs.scan(p)
    return rs.values().cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0, 1])
def test_radix_select_one_row_of_65536_element_segments(offset):
    """A row of >= 6 x SMs x 65536 elements keeps the largest segment; offset 1 makes every segment start with a
    three-element scalar head."""
    n = 6 * _lib.load().sb200_sm_count() * 65536 + 12345
    g = torch.Generator(device="cuda").manual_seed(5)
    buf = torch.randn(n + 1, generator=g, device=dev())
    x = buf[offset:offset + n]
    ks = [0, n // 2, n - 1]
    got = _select(1, [ks[0]], [x.reshape(1, -1)])
    got = [float(got[0])] + [float(ops.kth_value(x, k)) for k in ks[1:]]
    exp = np.partition(x.cpu().numpy(), ks)[ks]
    assert got == [float(v) for v in exp]


@pytest.mark.gpu
def test_percentile_ranks_257_rows_two_targets():
    """The percentile observer's device flow for 257 rows x 2 targets vs oracle.observers.percentile(per_channel)."""
    rng = np.random.default_rng(9)
    rows, n, alpha = 257, 20_001, 1e-3
    x = (rng.standard_normal((rows, n)) * rng.uniform(0.1, 10, (rows, 1))).astype(F32)
    x[3] = np.abs(x[3])  # no negatives: min stays 0
    x[4] = -np.abs(x[4]) - 1  # no non-negatives: max stays 0
    x[5] = np.round(x[5])  # heavy duplicates
    xt = t(x)
    rs = ops.RadixSelect(rows, 2, dev())
    rs.hist_pass(0, xt, with_counts=True)
    rs.percentile_ranks(torch.full((rows,), n, dtype=torch.int64, device=dev()), alpha)
    rs.scan(0)
    for p in (1, 2):
        rs.hist_pass(p, xt)
        rs.scan(p)
    vals, counts = rs.values().reshape(rows, 2), rs.counts.reshape(rows, 2)
    zero = torch.zeros(rows, device=dev())
    mn = torch.where(counts[:, 0] > 0, vals[:, 0], zero).cpu().numpy()
    mx = torch.where(counts[:, 1] > 0, vals[:, 1], zero).cpu().numpy()
    emn, emx = oobs.percentile([x], alpha, per_channel=True, ch_axis=0)
    assert bits_equal(mn, emn) and bits_equal(mx, emx)


@pytest.mark.gpu
def test_radix_select_accumulates_three_tensors():
    rng = np.random.default_rng(4)
    parts = [rng.standard_normal(1_000_003).astype(F32), (rng.standard_normal(77) * 5).astype(F32),
             (rng.standard_normal(300_000) + 1).astype(F32)]
    allx = np.concatenate(parts)
    ks = [12_345, allx.size - 40]
    got = _select(1, ks, [_dev(p, i % 2).reshape(1, -1) for i, p in enumerate(parts)], ntpr=2)
    assert np.array_equal(got, np.partition(allx, ks)[ks])


@pytest.mark.gpu
@pytest.mark.parametrize("span", [2**11 + 1, 2**10], ids=["top11-shared", "top22-shared"])
def test_radix_select_keys_sharing_high_bits(span):
    """Values 1 + j * 2^-23, j < span: with span 2^11 + 1 (data in [1, 1 + 2^-12]) pass 0 sees one bucket, with 2^10
    passes 0 and 1 do and pass 2 alone decides."""
    rng = np.random.default_rng(span)
    x = (F32(1) + rng.integers(0, span, 700_001).astype(F32) * F32(2.0**-23)).astype(F32)
    ks = [0, 1, 350_000, 700_000]
    got = [float(ops.kth_value(_dev(x, 1), k)) for k in ks]
    assert got == [float(v) for v in np.partition(x, ks)[ks]]


@pytest.mark.gpu
def test_radix_select_heavy_duplicates_and_signed_zeros():
    rng = np.random.default_rng(8)
    x = rng.choice(np.array([-1.5, -0.0, 0.0, 1e-45, 2.0], F32), 100_003, p=[0.2, 0.25, 0.25, 0.1, 0.2]).astype(F32)
    xs = np.sort(x)
    for k in [0, 20_000, 20_001, 45_000, 70_000, 80_000, 100_002]:
        assert float(ops.kth_value(_dev(x), k)) == float(xs[k]), k


def test_kth_value_rejects_out_of_range_rank():
    x = torch.zeros(5)
    for k in (5, 6, -1):
        with pytest.raises(SparsebitB200Error, match="kth_value"):
            ops.kth_value(x, k)


# ------------------------------------------------------------------------------------------------ MSE sweep and moments
@pytest.mark.gpu
@pytest.mark.parametrize("rows,row_len", [(1, 8192 * 64 + 5), (1, 20_000_000), (3, 1_000_000)])
def test_mse_sweep_and_moments_long_rows(rows, row_len):
    """Rows of many tiles: the fixed-order finish sums many slices of partials per output."""
    g = torch.Generator(device="cuda").manual_seed(row_len)
    x = torch.randn(rows, row_len, generator=g, device=dev()) * 1.5
    xc = x.cpu().numpy()
    ncand = 8 if x.numel() > 10_000_000 else 20
    f = np.array([1.0 - 0.03 * i for i in range(ncand)]).astype(F32)
    cs, cz = oobs.calc_qparams_with_minmax(xc.min(axis=1)[:, None] * f, xc.max(axis=1)[:, None] * f, 0, 15, False)
    sse = torch.zeros(rows, ncand, dtype=torch.float64, device=dev())
    ops.mse_sweep(x, t(cs), t(cz), 0, 15, sse)
    x64 = xc.astype(np.float64)
    exp = np.array([[((x64[r] - oqdq.qdq(xc[r], cs[r, i:i + 1], cz[r, i:i + 1], 0, 15)) ** 2).sum() for i in range(ncand)]
                    for r in range(rows)])
    got = sse.cpu().numpy()
    np.testing.assert_allclose(got, exp, rtol=1e-5)
    assert np.array_equal(got.argmin(axis=1), exp.argmin(axis=1))

    mean = x64.mean(axis=1)
    for centre in (None, mean):
        out = ops.moments_update(x, ops.moments_new(rows, dev()), None if centre is None else t(centre))
        c = np.zeros((rows, 1)) if centre is None else centre[:, None]
        d = x64 - c
        exp_m = np.stack([x64.sum(1), (x64 * x64).sum(1), np.abs(x64).sum(1), np.abs(d).sum(1), (d * d).sum(1)], axis=1)
        scale = np.stack([np.abs(x64).sum(1), (x64 * x64).sum(1), np.abs(x64).sum(1), np.abs(d).sum(1), (d * d).sum(1)], axis=1)
        assert np.all(np.abs(out.cpu().numpy() - exp_m) <= 1e-12 * scale), centre is None


# ------------------------------------------------------------------------------------------------ histogram
@pytest.mark.gpu
@pytest.mark.parametrize("bins,lo,hi", [(10, -2.0, 3.0), (7, -1.0, 1.3)])
def test_hist_unaligned_tiny_inputs_on_bin_edges(bins, lo, hi):
    """One and three unaligned elements per call (the scalar path), on every bin edge, its neighbours, lo and hi."""
    lo, hi = F32(lo), F32(hi)
    edges = (lo + np.arange(bins + 1, dtype=F32) * ((hi - lo) / F32(bins))).astype(F32)
    vals = np.concatenate([edges, np.nextafter(edges, F32(-np.inf)), np.nextafter(edges, F32(np.inf)),
                           np.array([lo, hi, np.nan, -np.inf, np.inf, hi * 2], F32)]).astype(F32)
    counts = torch.zeros(bins, dtype=torch.int64, device=dev())
    rng_t = t(np.array([lo, hi], F32))
    exp = np.zeros(bins, np.int64)
    chunks = [vals[i:i + 1] for i in range(vals.size)] + [vals[i:i + 3] for i in range(0, vals.size - 2, 3)]
    for ch in chunks:
        ops.hist_update(_dev(ch, 1), rng_t, counts)
        exp += oobs.histc(ch, bins, lo, hi)
    big = np.random.default_rng(bins).choice(vals, 1001).astype(F32)
    ops.hist_update(_dev(big, 1), rng_t, counts)
    exp += oobs.histc(big, bins, lo, hi)
    assert np.array_equal(counts.cpu().numpy(), exp)
