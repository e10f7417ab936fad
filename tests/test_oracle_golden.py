"""CPU: pin the numpy oracle against golden vectors produced by the unmodified reference
(tests/golden/make_golden.py).  Integer / mask paths bit-exact, float rescale bit-exact too
(same IEEE op sequence), MSE argmin identical, KL threshold identical."""
import numpy as np
import pytest

from oracle import gptq as ogptq
from oracle import observers as oobs
from oracle import qdq as oqdq
from oracle import sparse as osparse


def _eq_bits(a, b):
    a = np.asarray(a, dtype=np.float32)
    b = np.asarray(b, dtype=np.float32)
    # treat +0 / -0 as equal (SURVEY Q17), NaN == NaN
    return np.array_equal(np.where(a == 0, 0.0, a), np.where(b == 0, 0.0, b), equal_nan=True)


def test_qdq_matches_reference(golden):
    g = golden("qdq")
    for name in g["cases"]:
        qmin, qmax, ch_axis, _ = g[name + "_meta"]
        y = oqdq.qdq(g[name + "_x"], g[name + "_scale"], g[name + "_zp"], int(qmin), int(qmax), int(ch_axis))
        assert _eq_bits(y, g[name + "_y"]), name
        if name + "_ytrt" in g.files:  # symmetric: TensorRT-style branch equals zp == 0
            y0 = oqdq.qdq(g[name + "_x"], g[name + "_scale"], np.zeros_like(g[name + "_zp"]), int(qmin), int(qmax), int(ch_axis))
            assert _eq_bits(y0, g[name + "_ytrt"]), name


def _batches(g, name):
    return [g[f"{name}_x{i}"] for i in range(int(g[name + "_nb"]))]


@pytest.mark.parametrize("kind", ["minmax", "pct", "kl", "mse"])
def test_observers_match_reference(golden, kind):
    g = golden("observers")
    seen = 0
    for name in g["cases"]:
        if not name.startswith(kind):
            continue
        seen += 1
        qmin, qmax, ch_axis, perch, sym, bit = (int(v) for v in g[name + "_meta"])
        xs = _batches(g, name)
        if kind == "minmax":
            mn, mx = oobs.minmax(xs, bool(perch), ch_axis)
        elif kind == "pct":
            mn, mx = oobs.percentile(xs, float(g[name + "_alpha"]), bool(perch), ch_axis)
        elif kind == "kl":
            mn, mx = oobs.kl_histogram(xs, bit)
        if kind == "mse":
            s, z, _ = oobs.mse(xs, qmin, qmax, bool(sym), bool(perch), ch_axis)
        else:
            assert _eq_bits(np.reshape(mn, -1), g[name + "_min"]), name
            assert _eq_bits(np.reshape(mx, -1), g[name + "_max"]), name
            s, z = oobs.calc_qparams_with_minmax(mn, mx, qmin, qmax, bool(sym))
        assert _eq_bits(np.reshape(s, -1), g[name + "_scale"]), name
        assert _eq_bits(np.reshape(z, -1), g[name + "_zp"]), name
    assert seen > 0


def test_histc_matches_aten(golden):
    g = golden("observers")
    am = float(g["histc_absmax"])
    h = oobs.histc(g["histc_x"], 2048, -am, am)
    assert np.array_equal(h, g["histc_counts"].astype(np.int64))


def test_sparse_matches_reference(golden):
    g = golden("sparse")
    for name in g["cases"]:
        w, ratio = g[name + "_w"], float(g[name + "_ratio"])
        m = osparse.l1_unstructured_mask(w, ratio)
        assert np.array_equal(np.asarray(m).astype(np.float32), g[name + "_mask"].astype(np.float32)), name
        assert _eq_bits(osparse.mask_apply(w, m), g[name + "_masked"]), name


def test_gptq_matches_reference(golden):
    g = golden("gptq")
    for name in g["cases"]:
        gs = int(g[name + "_gs"])
        x, qw = g[name + "_x"], g[name + "_qweight"]
        n = qw.shape[1]
        k = x.shape[-1]
        # packed integers decode back to the dequantised weights the reference's ground truth uses
        s, z = g[name + "_scales"], g[name + "_zeros"]
        q = ogptq.unpack_int4(qw, k).astype(np.float32)
        gsz = k if gs == -1 else gs
        gi = np.arange(k) // gsz
        w = (s.T[gi] * q - z.T[gi]).T  # [N, K]
        np.testing.assert_allclose(w, g[name + "_wdq"], rtol=0, atol=2e-7)
        # packing the decoded integers again gives the reference's words bit for bit (any K, no group structure)
        assert np.array_equal(ogptq.pack_values(ogptq.unpack_int4(qw, k), 4), qw), name
        bias = np.broadcast_to(g[name + "_bias"], x.shape[:-1] + (n,))
        y = ogptq.dequant_matmul(x, qw, bias, s, z, 0 if gs == -1 else gs)
        # reference pin: test_cuda_kernel.py:47  rtol = atol = 1e-5 against Linear(dequantised W)
        np.testing.assert_allclose(y, g[name + "_gt"], rtol=1e-5, atol=1e-5)
        # the oracle's own find_params / pack reproduce the reference's packed tensors
        s2, z2 = ogptq.find_params_int4(g[name + "_wdq"], gs)
        qw2, sc2, zr2 = ogptq.pack_int4(g[name + "_wdq"], s2, z2)
        # (dequantised weights re-quantise onto the same grid)
        np.testing.assert_allclose(sc2, s, rtol=1e-6, atol=0)


def test_torch_port_matches_reference(golden):
    """oracle/torch_port.py (the CPU baseline bench.py times) == the reference's outputs."""
    import torch

    from oracle import torch_port

    g = golden("qdq")
    for name in g["cases"]:
        qmin, qmax, ch_axis, perch = (int(v) for v in g[name + "_meta"])
        x = torch.from_numpy(g[name + "_x"])
        shape = [1] * x.dim()
        if perch:
            shape[ch_axis] = -1
        s = torch.from_numpy(g[name + "_scale"]).reshape(shape)
        z = torch.from_numpy(g[name + "_zp"]).reshape(shape)
        y = torch_port.ort_fake_quant_cpu(x, s, z, qmin, qmax)
        assert _eq_bits(y.numpy(), g[name + "_y"]), name


def test_torch_port_observers_and_sparser_match_reference(golden):
    """The observer / sparser CPU op chains bench.py times as ``cpu_baselines`` (oracle/torch_port.py) reproduce the
    reference's per-tensor results: same min/max, same MSE candidate, same k-th values, same KL threshold, same mask."""
    import torch

    from oracle import torch_port

    g = golden("observers")
    for name in g["cases"]:
        qmin, qmax, ch_axis, perch, sym, bit = (int(v) for v in g[name + "_meta"])
        if perch:
            continue
        xs = [torch.from_numpy(g[f"{name}_x{i}"]) for i in range(int(g[name + "_nb"]))]
        if name.startswith("minmax"):
            mn, mx = torch_port.minmax_observer_cpu(xs)
            assert float(mn) == float(g[name + "_min"].reshape(-1)[0]) and float(mx) == float(g[name + "_max"].reshape(-1)[0])
            s, z = torch_port.calc_qparams_with_minmax_cpu(mn, mx, qmin, qmax, bool(sym))
        elif name.startswith("mse"):
            s, z = torch_port.mse_observer_cpu(xs, qmin, qmax, bool(sym))
        elif name.startswith("pct"):
            mn, mx = torch_port.percentile_observer_cpu(xs, float(g[name + "_alpha"]))
            assert float(mn) == float(g[name + "_min"].reshape(-1)[0]) and float(mx) == float(g[name + "_max"].reshape(-1)[0])
            s, z = torch_port.calc_qparams_with_minmax_cpu(mn, mx, qmin, qmax, bool(sym))
        else:
            mn, mx = torch_port.kl_observer_cpu(xs, bit)
            np.testing.assert_allclose([mn, mx], [g[name + "_min"].reshape(-1)[0], g[name + "_max"].reshape(-1)[0]], rtol=1e-6)
            continue
        assert _eq_bits(np.float32(s).reshape(-1), g[name + "_scale"].reshape(-1)), name
        assert _eq_bits(np.float32(z).reshape(-1), g[name + "_zp"].reshape(-1)), name
    g = golden("sparse")
    for name in g["cases"]:
        ratio = float(g[name + "_ratio"])
        if ratio == 0.0:
            continue
        m = torch_port.l1_unstructured_mask_cpu(torch.from_numpy(g[name + "_w"]), ratio)
        assert np.array_equal(m.numpy(), g[name + "_mask"].astype(bool)), name


def test_c_restatement_matches_reference(golden):
    """oracle/c/libsb_oracle.so (plain C, -ffp-contract=off) == the reference's outputs."""
    import ctypes
    import os

    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "c", "libsb_oracle.so")
    if not os.path.exists(path):
        pytest.skip("oracle/c not built (run __graft_entry__.build())")
    lib = ctypes.CDLL(path)
    vp = ctypes.c_void_p
    g = golden("qdq")
    for name in g["cases"]:
        qmin, qmax, ch_axis, perch = (int(v) for v in g[name + "_meta"])
        x = np.ascontiguousarray(g[name + "_x"])
        s, z = np.ascontiguousarray(g[name + "_scale"]), np.ascontiguousarray(g[name + "_zp"])
        out = np.empty_like(x)
        if perch:
            outer = int(np.prod(x.shape[:ch_axis], dtype=np.int64))
            c, inner = x.shape[ch_axis], int(np.prod(x.shape[ch_axis + 1 :], dtype=np.int64))
        else:
            outer, c, inner = 1, 1, x.size
        lib.sbo_qdq(x.ctypes.data_as(vp), s.ctypes.data_as(vp), z.ctypes.data_as(vp), out.ctypes.data_as(vp),
                    ctypes.c_int64(outer), ctypes.c_int64(c), ctypes.c_int64(inner), qmin, qmax)
        assert _eq_bits(out, g[name + "_y"]), name
    gg = golden("gptq")
    name = "group128_b29"
    x, qw = np.ascontiguousarray(gg[name + "_x"]), np.ascontiguousarray(gg[name + "_qweight"])
    n, k = qw.shape[1], x.shape[-1]
    out = np.ascontiguousarray(np.broadcast_to(gg[name + "_bias"], (x.shape[0], n))).copy()
    sc, zr = np.ascontiguousarray(gg[name + "_scales"]), np.ascontiguousarray(gg[name + "_zeros"])
    lib.sbo_gptq4(x.ctypes.data_as(vp), qw.ctypes.data_as(vp), out.ctypes.data_as(vp), sc.ctypes.data_as(vp),
                  zr.ctypes.data_as(vp), ctypes.c_int64(x.shape[0]), ctypes.c_int64(k), ctypes.c_int64(n), 128)
    np.testing.assert_allclose(out, gg[name + "_gt"], rtol=1e-5, atol=1e-5)


def test_adaround_restatement_matches_reference(golden):
    """oracle/qdq.py adaround_* vs the unmodified reference quantizer (adaround.py) incl. autograd's dL/dv."""
    g = golden("next_rows")
    for name in g["ada_cases"]:
        qmin, qmax, ch_axis, perch, _, _ = (int(v) for v in g[name + "_meta"])
        w, v0, v1, s, zp = (g[name + k] for k in ("_w", "_v0", "_v1", "_scale", "_zp"))
        # hard rounding is integer work: bit-exact
        assert _eq_bits(oqdq.adaround_forward(w, v1, s, zp, qmin, qmax, ch_axis, soft=False), g[name + "_yhard"]), name
        # exp / log differ by an ulp between libms: float tolerance of the north star (1e-5 relative)
        np.testing.assert_allclose(oqdq.adaround_init(w, s, ch_axis), v0, rtol=1e-5, atol=1e-6, err_msg=name)
        np.testing.assert_allclose(oqdq.adaround_forward(w, v1, s, zp, qmin, qmax, ch_axis, soft=True), g[name + "_ysoft"],
                                   rtol=1e-5, atol=1e-7, err_msg=name)
        np.testing.assert_allclose(oqdq.adaround_grad_v(w, v1, s, zp, g[name + "_gy"], qmin, qmax, ch_axis), g[name + "_gv"],
                                   rtol=1e-5, atol=1e-8, err_msg=name)


def test_clamp_backward_restatement_matches_aten_autograd():
    """oracle.qdq.clamp_backward against autograd through torch.clamp with tensor bounds (what pact.py:43-46 runs), incl.
    values exactly on the bounds."""
    import torch

    g = torch.Generator().manual_seed(3)
    x = torch.randn(5, 7, 11, generator=g) * 2
    x.view(-1)[:4] = torch.tensor([1.5, -1.5, 1.5000001, -1.5000001])
    gy = torch.randn(x.shape, generator=g)
    for symmetric in (True, False):
        alpha = torch.tensor([1.5], requires_grad=True)
        xr = x.clone().requires_grad_(True)
        lower = -alpha if symmetric else torch.zeros(1)
        torch.clamp(xr, lower, alpha).backward(gy)
        gx, g_hi, g_lo = oqdq.clamp_backward(x.numpy(), gy.numpy(), float(lower.detach()), 1.5)
        assert np.array_equal(gx, xr.grad.numpy())
        expect = g_hi - g_lo if symmetric else g_hi
        np.testing.assert_allclose(float(alpha.grad), expect, rtol=1e-5)


def test_dorefa_restatement_matches_reference(golden):
    """oracle.qdq.dorefa_forward against the reference's DoReFa quantizer output (dorefa.py:15-20); numpy's tanh may
    differ from ATen's by an ulp, which can move a value across a rounding boundary: a few grid flips are allowed."""
    g = golden("next_rows")
    x = g["dorefa_w4_x0"]
    qmin, qmax = (int(v) for v in g["dorefa_w4_meta"][:2])
    y = oqdq.dorefa_forward(x, g["dorefa_w4_scale"], g["dorefa_w4_zp"], qmin, qmax)
    assert np.mean(y != g["dorefa_w4_y"]) < 5e-3
    step = float(g["dorefa_w4_scale"][0])
    assert np.abs(y - g["dorefa_w4_y"]).max() <= step * 1.0001  # a flip moves a value by exactly one grid step
    xn, t, m = oqdq.dorefa_normalise(x)
    assert np.abs(xn).max() == 1.0 and m == np.abs(np.tanh(x.astype(np.float32))).max()
    # gradient restatement: finite-difference-free sanity -- zero where the STE masks, else gy / m * (1 - t^2)
    gy = np.ones_like(x)
    gx = oqdq.dorefa_grad_x(x, g["dorefa_w4_scale"], g["dorefa_w4_zp"], gy, qmin, qmax)
    assert gx.shape == x.shape and np.all(gx >= 0) and np.all(gx <= 1.0 / m + 1e-6)


def test_gptq_lowbit_matches_reference(golden):
    """3-bit / 2-bit packing + matmul restatement vs the reference's QuantLinear.pack and its
    Linear(dequantised W) ground truth (test_cuda_kernel.py bit=2,3 cases, scaled down)."""
    g = golden("gptq_lowbit")
    for name in g["cases"]:
        bit, gs = (int(v) for v in g[name + "_meta"])
        x, qw = g[name + "_x"], g[name + "_qweight"]
        n, k = qw.shape[1], x.shape[-1]
        s, z, zi = g[name + "_scales"], g[name + "_zeros"], g[name + "_zero_int"]
        assert qw.shape[0] == ogptq.packed_rows(k, bit), name
        q = ogptq.unpack_bits(qw, k, bit)
        assert q.max() <= 2**bit - 1
        assert np.array_equal(ogptq.pack_values(q, bit), qw), name
        gi = np.arange(k) // (k if gs == -1 else gs)
        w = (s.T[gi] * q.astype(np.float32) - z.T[gi]).T
        np.testing.assert_allclose(w, g[name + "_wdq"], rtol=0, atol=4e-7, err_msg=name)
        # re-packing the dequantised weights gives the reference's words bit for bit
        qw2, s2, z2 = ogptq.pack_bits(g[name + "_wdq"], s, zi, bit)
        assert np.array_equal(qw2, qw), name
        assert np.array_equal(z2, z), name
        bias = np.broadcast_to(g[name + "_bias"], x.shape[:-1] + (n,))
        y = ogptq.dequant_matmul(x, qw, bias, s, z, 0 if gs == -1 else gs, bit=bit)
        np.testing.assert_allclose(y, g[name + "_gt"], rtol=1e-5, atol=1e-5, err_msg=name)
        # parameter search restatement (scale is (max - min) / (2^bit - 1) of the float weights; the
        # dequantised weights span the same range up to rounding at the ends)
        s3, _ = ogptq.find_params(g[name + "_wdq"], bit, gs)
        assert s3.shape == s.shape


def test_c_restatement_widened_rows(golden):
    """oracle/c: 3 / 2-bit GPTQ unpack + matmul and the AdaRound evaluation branch vs the reference's outputs."""
    import ctypes
    import os

    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "c", "libsb_oracle.so")
    if not os.path.exists(path):
        pytest.skip("oracle/c not built (run __graft_entry__.build())")
    lib = ctypes.CDLL(path)
    if not hasattr(lib, "sbo_gptq_bits"):
        pytest.skip("oracle/c is stale (run __graft_entry__.build())")
    vp, i64 = ctypes.c_void_p, ctypes.c_int64
    g = golden("gptq_lowbit")
    for name in ("b3_irregular", "b3_group128_b29", "b2_irregular", "b2_group64_b29", "b2_group192_b4"):
        bit, gs = (int(v) for v in g[name + "_meta"])
        x = np.ascontiguousarray(g[name + "_x"].reshape(-1, g[name + "_x"].shape[-1]))
        qw = np.ascontiguousarray(g[name + "_qweight"])
        n, k = qw.shape[1], x.shape[1]
        out = np.ascontiguousarray(np.broadcast_to(g[name + "_bias"], (x.shape[0], n))).copy()
        sc, zr = np.ascontiguousarray(g[name + "_scales"]), np.ascontiguousarray(g[name + "_zeros"])
        lib.sbo_gptq_bits(x.ctypes.data_as(vp), qw.ctypes.data_as(vp), out.ctypes.data_as(vp), sc.ctypes.data_as(vp),
                          zr.ctypes.data_as(vp), i64(x.shape[0]), i64(k), i64(n), 0 if gs == -1 else gs, bit)
        np.testing.assert_allclose(out, g[name + "_gt"].reshape(-1, n), rtol=1e-5, atol=1e-5, err_msg=name)
    g = golden("next_rows")
    for name in g["ada_cases"]:
        qmin, qmax, ch_axis, perch, _, _ = (int(v) for v in g[name + "_meta"])
        w, v1 = np.ascontiguousarray(g[name + "_w"]), np.ascontiguousarray(g[name + "_v1"])
        s, zp = np.ascontiguousarray(g[name + "_scale"]), np.ascontiguousarray(g[name + "_zp"])
        outer, c, inner = (1, w.shape[0], w[0].size) if perch else (1, 1, w.size)
        out = np.empty_like(w)
        lib.sbo_adaround_hard(w.ctypes.data_as(vp), v1.ctypes.data_as(vp), s.ctypes.data_as(vp), zp.ctypes.data_as(vp),
                              out.ctypes.data_as(vp), i64(outer), i64(c), i64(inner), qmin, qmax)
        assert _eq_bits(out, g[name + "_yhard"]), name


def test_exact_division_schemes_on_cpu():
    """oracle/c/validate_div.c: the kernels' two replacements for div.rn.f32 (fp64-reciprocal product; fp32
    Markstein quotient + magic rounding with its acceptance guard) re-enacted with IEEE CPU arithmetic."""
    import json
    import os
    import shutil
    import subprocess

    cdir = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "c")
    if shutil.which("gcc") is None and shutil.which("cc") is None:
        pytest.skip("no C compiler")
    subprocess.run(["make", "-C", cdir, "validate_div"], check=True, capture_output=True)
    res = subprocess.run([os.path.join(cdir, "validate_div"), "2000000", "7"], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr
    out = json.loads(res.stdout)
    assert out["exact_trick_mismatches"] == 0 and out["fast_path_mismatches"] == 0
    assert out["cases"] > 5_000_000 and out["fast_path_accepted"] > 1_000_000


def test_ste_backward_oracle_pinned_to_reference_myste(golden):
    """oracle.qdq.ste_backward against outputs of the reference's MySTE.backward (quant_tensor.py:46-71,
    generated by tests/golden/make_golden.py:gen_bwd): gx bit-exact; the scale / zero-point gradients equal the
    fp64 sums of the reference's elementwise terms."""
    from oracle import qdq as oqdq

    g = golden("bwd")
    for name in g["cases"]:
        qmin, qmax, ch_axis, perch = (int(v) for v in g[name + "_meta"])
        x, gy = g[name + "_x"], g[name + "_gy"]
        gx, gs, gzp = oqdq.ste_backward(x, g[name + "_scale"], g[name + "_zp"], gy, qmin, qmax, ch_axis)
        assert np.array_equal(gx, g[name + "_gx"]), name
        axes = tuple(a for a in range(x.ndim) if a != ch_axis) if perch else None
        ref_gs = g[name + "_gs_elem"].astype(np.float64).sum(axis=axes).reshape(-1)
        ref_gz = g[name + "_gz_elem"].astype(np.float64).sum(axis=axes).reshape(-1)
        l1s = np.abs(g[name + "_gs_elem"]).astype(np.float64).sum(axis=axes).reshape(-1) + 1e-30
        l1z = np.abs(g[name + "_gz_elem"]).astype(np.float64).sum(axis=axes).reshape(-1) + 1e-30
        assert np.all(np.abs(gs - ref_gs) <= 1e-6 * l1s), name
        assert np.all(np.abs(gzp - ref_gz) <= 1e-6 * l1z), name
        # the open-top rule only ever moves elements with vq == qmax into the clipped set
        _, _, gzp_open = oqdq.ste_backward(x, g[name + "_scale"], g[name + "_zp"], gy, qmin, qmax, ch_axis, gzp_open_top=True)
        assert gzp_open.shape == gzp.shape
