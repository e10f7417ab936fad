"""GPU parity against the REFERENCE'S OWN CUDA extensions, built unmodified by ``oracle/build_ref.py``:

  fake_quant_ref  torch_extensions/export.cc + fake_quant_tensor.cu -- the four entry points of export.cc:3-8
  gptq_ref        cuda/cuda_kernel*.cu                               -- vecquant{2,3,4}matmul (+ group variants)

What those kernels returned on the inputs below was recorded on a B200 by ``tests/golden/make_ref_ext.py`` into
``tests/golden/ref_ext.npz``, so the comparison needs neither the reference checkout nor its binaries.  Every
case stores a SHA-256 of its inputs (the inputs are regenerated from seeds and must be the recorded ones).

Forward outputs and gx are compared bit for bit: the golden file holds a SHA-256 of the whole reference output
(zeros and NaNs canonicalised, as ``bits_equal`` does) and its values at a fixed sample of positions.  The float
reductions gs / gzp are stored whole and compared at 1e-5 (relative to the L1 norm of the summed terms: the
reference accumulates with fp32 atomics in launch order); the GPTQ outputs at a fixed sample of positions, at
the reference's own tolerance.  Shapes keep every thread of the reference kernels inside its data: its backward
kernels call __syncthreads() under divergent control flow (fake_quant_tensor.cu:123,128,260,265), which is only
well defined when no thread leaves the loop early."""
import hashlib

import numpy as np
import pytest
import torch

from gpu_util import bits_equal, dev, t
from oracle import qdq as oqdq
from sparsebit_b200 import fake_quant
from sparsebit_b200.gptq import cuda_kernel

pytestmark = pytest.mark.gpu

PERTENSOR_CASES = [(512 * 40, -128, 127, 0.0), (2560 * 512, 0, 255, 37.0), (2 * 2560 * 512, -8, 7, 0.0)]
PERCHANNEL_CASES = [((8, 16, 32, 32), 1, -128, 127), ((64, 512), 0, -8, 7), ((4, 6, 7, 512), 1, 0, 15), ((16, 3, 1024), 1, 0, 255)]
GATE_CASES = [(False, False), (True, False), (False, True)]
GPTQ_CASES = [(4, 1, 4096, 4096, 128), (4, 16, 4096, 11008, 128), (4, 5, 1024, 768, -1), (3, 3, 4096, 512, 128),
              (2, 7, 2048, 256, 64), (4, 256, 2048, 1024, 128)]
BITS_SAMPLE = 256  # stored values per bit-exact output (the digest covers all of it)
GPTQ_SAMPLE = 4096  # stored values per GPTQ output


def digest(*arrays):
    """SHA-256 of arrays as ``bits_equal`` sees them: float32, -0 -> +0, every NaN the same NaN."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.asarray(a)
        if a.dtype.kind == "f":
            a = np.asarray(a, np.float32)
            a = np.where(a == 0, np.float32(0), np.where(np.isnan(a), np.float32(np.nan), a))
        h.update(str((a.dtype.str, a.shape)).encode())
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def sample_index(size, count):
    """Fixed positions (seeded, sorted) at which a flattened output of `size` elements is stored."""
    if size <= count:
        return np.arange(size)
    return np.sort(np.random.default_rng(0).choice(size, count, replace=False))


def pertensor_key(n, qmin, qmax, zp):
    return f"pt_{n}_{qmin}_{qmax}_{zp:g}"


def pertensor_inputs(n, qmin, qmax, zp):
    rng = np.random.default_rng(n + qmax)
    x = (rng.standard_normal(n) * 1.5).astype(np.float32)
    gy = rng.standard_normal(n).astype(np.float32)
    s = np.float32([np.abs(x).max() / (qmax - qmin) * 1.2])  # clips ~ 10 % of a symmetric range
    z = np.float32([zp])
    return x, gy, s, z


def perchannel_key(shape, ch_axis, qmin, qmax):
    return f"pc_{'x'.join(map(str, shape))}_{ch_axis}_{qmin}_{qmax}"


def perchannel_inputs(shape, ch_axis, qmin, qmax):
    rng = np.random.default_rng(sum(shape) + qmax)
    x = (rng.standard_normal(shape) * 1.5).astype(np.float32)
    gy = rng.standard_normal(shape).astype(np.float32)
    c = shape[ch_axis]
    s = (rng.uniform(0.6, 1.4, c) * 4.0 / (qmax - qmin)).astype(np.float32)
    z = np.rint(rng.uniform(-2, 2, c) + (0 if qmin < 0 else (qmax + 1) // 2)).astype(np.float32)
    return x, gy, s, z


def gate_inputs():
    rng = np.random.default_rng(4096)
    return (rng.standard_normal(512 * 8).astype(np.float32), rng.standard_normal(512 * 8).astype(np.float32),
            np.float32([0.05]), np.float32([3.0]))


def gptq_key(bit, m, k, n, gs):
    return f"gptq_{bit}_{m}_{k}_{n}_{gs}"


def gptq_name(bit, gs):
    return f"vec{'group' if gs != -1 else ''}quant{bit}matmul"


def gptq_inputs(bit, m, k, n, gs):
    """The same packed checkpoint and activations for both implementations: (x, qweight, scales, zeros, bias)."""
    from sparsebit_b200.gptq import find_params, pack_intweight

    torch.manual_seed(bit * 1000 + m)
    w = torch.randn(n, k) / k**0.5
    scale, zero = find_params(w, bit, gs)
    g = scale.reshape(n, -1).shape[1]
    q = torch.clamp(torch.round(w.view(n, g, -1) / scale.view(n, g, 1)) + zero.view(n, g, 1), 0, 2**bit - 1)
    qw = pack_intweight(q.view(n, k).to(torch.int64).t().contiguous(), bit).to(dev())
    scales = scale.reshape(n, g).contiguous().to(dev())
    zeros = (zero * scale).reshape(n, g).contiguous().to(dev())
    x = torch.randn(m, k, device=dev())
    bias = torch.randn(n, device=dev()) * 0.1
    return x, qw, scales, zeros, bias


def _np(*ts):
    return [v.detach().cpu().numpy() for v in ts]


def _close(a, b, l1, tol=1e-5):
    return np.all(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)) <= tol * (np.asarray(l1, np.float64) + 1e-30))


def _assert_bits_equal_reference(ours, g, key):
    ours = np.asarray(ours, np.float32).reshape(-1)
    idx = sample_index(ours.size, BITS_SAMPLE)
    assert bits_equal(ours[idx], g[key + "_sample"]), key
    assert digest(ours) == str(g[key + "_sha256"]), key


@pytest.fixture(scope="module")
def ref(golden):
    return golden("ref_ext")


@pytest.mark.parametrize("n,qmin,qmax,zp", PERTENSOR_CASES)
def test_pertensor_forward_backward_equal_reference_kernels(ref, n, qmin, qmax, zp):
    key = pertensor_key(n, qmin, qmax, zp)
    x, gy, s, z = pertensor_inputs(n, qmin, qmax, zp)
    assert digest(x, gy, s, z) == str(ref[key + "_inputs_sha256"])
    xt, gt = t(x), t(gy)
    st, zt = t(s).requires_grad_(True), t(z).requires_grad_(True)
    y = fake_quant.quant_pertensor_forward(xt, st, zt, qmin, qmax, 0)
    _assert_bits_equal_reference(y.cpu().numpy(), ref, key + "_y")
    gx, gs, gz = _np(*fake_quant.quant_pertensor_backward(xt, st, zt, gt, qmin, qmax, 0))
    _assert_bits_equal_reference(gx, ref, key + "_gx")
    _, egs, egz = oqdq.ste_backward(x, s, z, gy, qmin, qmax)
    l1g = np.abs(gy).astype(np.float64).sum()
    l1s, l1z = l1g * max(abs(qmin - zp), abs(qmax - zp), 1.0), l1g * s[0]  # L1 norms of the summed terms
    assert _close(gs, egs, l1s, 1e-6) and _close(gz, egz, l1z, 1e-6)  # ours vs fp64
    assert _close(gs, ref[key + "_gs"], l1s) and _close(gz, ref[key + "_gz"], l1z)


@pytest.mark.parametrize("shape,ch_axis,qmin,qmax", PERCHANNEL_CASES)
def test_perchannel_forward_backward_equal_reference_kernels(ref, shape, ch_axis, qmin, qmax):
    key = perchannel_key(shape, ch_axis, qmin, qmax)
    x, gy, s, z = perchannel_inputs(shape, ch_axis, qmin, qmax)
    assert digest(x, gy, s, z) == str(ref[key + "_inputs_sha256"])
    xt, gt = t(x), t(gy)
    st, zt = t(s).requires_grad_(True), t(z).requires_grad_(True)
    y = fake_quant.quant_perchannel_forward(xt, st, zt, qmin, qmax, ch_axis, 0)
    _assert_bits_equal_reference(y.cpu().numpy(), ref, key + "_y")
    gx, gs, gz = _np(*fake_quant.quant_perchannel_backward(xt, st, zt, gt, qmin, qmax, ch_axis, 0))
    _assert_bits_equal_reference(gx, ref, key + "_gx")
    gs_r, gz_r = ref[key + "_gs"], ref[key + "_gz"]
    axes = tuple(a for a in range(len(shape)) if a != ch_axis)
    l1g = np.abs(gy).astype(np.float64).sum(axis=axes)
    l1s, l1z = l1g * np.maximum(np.abs(qmin - z), np.abs(qmax - z)), l1g * s
    assert _close(gs, gs_r, l1s)
    # zero-point gradient: the reference kernel's open-top rule (fake_quant_tensor.cu:264) is what ships by default
    assert _close(gz, gz_r, l1z)
    _, _, egz_open = oqdq.ste_backward(x, s, z, gy, qmin, qmax, ch_axis, gzp_open_top=True)
    _, _, egz_closed = oqdq.ste_backward(x, s, z, gy, qmin, qmax, ch_axis)
    assert _close(gz_r, egz_open, l1z) and not _close(gz_r, egz_closed, l1z)


def test_requires_grad_gates_match_reference(ref):
    x, gy, s, z = gate_inputs()
    assert digest(x, gy, s, z) == str(ref["gate_inputs_sha256"])
    x, gy, s, z = t(x), t(gy), t(s), t(z)
    for i, (rs, rz) in enumerate(GATE_CASES):
        st, zt = s.clone().requires_grad_(rs), z.clone().requires_grad_(rz)
        _, gs, gz = fake_quant.quant_pertensor_backward(x, st, zt, gy, -8, 7, 0)
        assert (ref["gate_gs"][i] == 0) == (float(gs) == 0) and (ref["gate_gz"][i] == 0) == (float(gz) == 0)


@pytest.mark.parametrize("bit,m,k,n,gs", GPTQ_CASES)
def test_gptq_kernels_equal_reference_kernels(ref, bit, m, k, n, gs):
    """Same packed checkpoint, same activations: ours vs the reference's VecQuant{2,3,4}MatMulKernel
    (cuda_kernel_{2,3,4}bit.cu) at the reference's own tolerance rtol = atol = 1e-5 (test_cuda_kernel.py:47)."""
    key = gptq_key(bit, m, k, n, gs)
    x, qw, scales, zeros, bias = gptq_inputs(bit, m, k, n, gs)
    assert digest(*_np(x, qw, scales, zeros, bias)) == str(ref[key + "_inputs_sha256"])
    y = bias.expand(m, n).contiguous()
    if gs == -1:
        getattr(cuda_kernel, gptq_name(bit, gs))(x, qw, y, scales, zeros)
    else:
        getattr(cuda_kernel, gptq_name(bit, gs))(x, qw, y, scales, zeros, gs)
    idx = sample_index(m * n, GPTQ_SAMPLE)
    torch.testing.assert_close(torch.from_numpy(y.cpu().numpy().reshape(-1)[idx]), torch.from_numpy(ref[key + "_y_sample"]),
                               rtol=1e-5, atol=1e-5)
