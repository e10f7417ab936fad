"""Oracle: quantize -> dequantize and its STE backward (numpy, IEEE fp32 op by op).

numpy float32 ufuncs (divide, rint, add, clip-by-comparison, subtract, multiply) are correctly
rounded IEEE operations, i.e. bit-identical to the ATen CPU ops the reference chains.
"""
import numpy as np

F32 = np.float32


def _round(v, rounding=0):
    """rounding 0: half-to-even (torch.round); 1: floor(v + .5); 2: ceil(v - .5)
    (sparsebit/quantization/torch_extensions/common.cuh:62-76)."""
    if rounding == 0:
        return np.rint(v)
    if rounding == 1:
        return np.floor(v + F32(0.5))
    if rounding == 2:
        return np.ceil(v - F32(0.5))
    raise ValueError(rounding)


def _clamp_keep_nan(v, lo, hi):
    """torch.clamp semantics: NaN stays NaN."""
    v = np.where(v < F32(lo), F32(lo), v)
    v = np.where(v > F32(hi), F32(hi), v)
    return v.astype(F32)


def _bcast(param, x, ch_axis):
    param = np.asarray(param, dtype=F32).reshape(-1)
    if param.size == 1:
        return param.reshape([1] * x.ndim)
    shape = [1] * x.ndim
    shape[ch_axis] = -1
    return param.reshape(shape)


def qdq(x, scale, zero_point, qmin, qmax, ch_axis=0, rounding=0):
    """ort_fake_quant CPU branch, sparsebit/quantization/quantizers/quant_tensor.py:181-184:
        zp = zero_point.round(); x_q = clamp((x / scale).round() + zp, qmin, qmax)
        x_dq = (x_q - zp) * scale
    ``scale`` / ``zero_point`` hold 1 value (per-tensor) or C values along ``ch_axis``
    (per-channel, fake_quant_tensor.cu:183 ``c = (i / inner) % C``)."""
    x = np.asarray(x, dtype=F32)
    s = _bcast(scale, x, ch_axis)
    zp = np.rint(_bcast(zero_point, x, ch_axis))
    with np.errstate(all="ignore"):
        q = _round((x / s).astype(F32), rounding)
        xq = _clamp_keep_nan((q + zp).astype(F32), qmin, qmax)
        return ((xq - zp).astype(F32) * s).astype(F32)


def quantize_int(x, scale, zero_point, qmin, qmax, ch_axis=0, rounding=0):
    """The integer grid point x_q (the 'integer clamp path' that must be bit-exact)."""
    x = np.asarray(x, dtype=F32)
    s = _bcast(scale, x, ch_axis)
    zp = np.rint(_bcast(zero_point, x, ch_axis))
    with np.errstate(all="ignore"):
        q = _round((x / s).astype(F32), rounding)
        return _clamp_keep_nan((q + zp).astype(F32), qmin, qmax)


def ste_backward(x, scale, zero_point, grad_y, qmin, qmax, ch_axis=0, rounding=0, gzp_open_top=False):
    """STE backward.  The production path has no CPU implementation (quant_tensor.py:113-116); restated
    from MySTE.backward (quant_tensor.py:46-71) and the CUDA kernels
    (torch_extensions/fake_quant_tensor.cu:111-131, 243-268), reductions in fp64:
        vq  = round(x/s) + zp
        gx  = gy * [qmin <= vq <= qmax]
        gs  = sum gy * (round(x/s) - x/s | qmin - zp | qmax - zp)
        gzp = sum -s * gy * [vq outside [qmin, qmax]]
    ``gzp_open_top``: the reference's PER-CHANNEL kernel tests ``vq >= qmin && vq < qmax``
    (fake_quant_tensor.cu:264), i.e. vq == qmax counts as clipped for the zero-point gradient only (SURVEY Q4).
    Pinned to MySTE.backward outputs (tests/golden/bwd.npz) and, on the GPU box, to the reference's own
    kernels (tests/test_gpu_reference_ext.py).  Returns gx (fp32), gs, gzp (fp64, shape [C] or [1])."""
    gx, gs_e, gz_e = ste_backward_terms(x, scale, zero_point, grad_y, qmin, qmax, ch_axis, rounding, gzp_open_top)
    nch = np.asarray(scale).size
    if nch == 1:
        return gx, np.array([gs_e.sum()]), np.array([gz_e.sum()])
    axes = tuple(a for a in range(gx.ndim) if a != ch_axis)
    return gx, gs_e.sum(axis=axes), gz_e.sum(axis=axes)


def ste_backward_terms(x, scale, zero_point, grad_y, qmin, qmax, ch_axis=0, rounding=0, gzp_open_top=False):
    """``ste_backward`` before the reductions: gx (fp32) and the per-element fp64 terms of gs and gzp, shaped like x
    (a tolerance for the sums can be stated against the L1 norm of their terms)."""
    x = np.asarray(x, dtype=F32)
    gy = np.asarray(grad_y, dtype=F32)
    s = _bcast(scale, x, ch_axis)
    zp = np.rint(_bcast(zero_point, x, ch_axis))
    with np.errstate(all="ignore"):
        q = (x / s).astype(F32)
        r = _round(q, rounding)
        vq = (r + zp).astype(F32)
    below = vq < F32(qmin)
    inside = (vq >= F32(qmin)) & (vq <= F32(qmax))
    gx = np.where(inside, gy, F32(0)).astype(F32)
    term = np.where(inside, (r - q).astype(F32), np.where(below, (F32(qmin) - zp).astype(F32), (F32(qmax) - zp).astype(F32)))
    gs_e = term.astype(np.float64) * gy.astype(np.float64)
    inside_z = inside & (vq < F32(qmax)) if gzp_open_top else inside
    gz_e = np.where(inside_z, 0.0, (-s).astype(np.float64) * gy.astype(np.float64))
    return gx, gs_e, gz_e


# --------------------------------------------------------------------------------------------
# PACT (sparsebit/quantization/quantizers/pact.py:43-46): torch.clamp(x, lower, alpha) in front of the STE.
def clamp_backward(x, grad_y, lo, hi):
    """Gradients of ``torch.clamp(x, lo, hi)`` with tensor bounds (ATen's convention: the closed interval passes the
    gradient to x, values above ``hi`` send it to ``hi``, values below ``lo`` to ``lo``); sums in fp64.
    Returns gx (fp32), g_hi, g_lo (fp64 scalars).  For the symmetric range PACT uses lower = -alpha, so
    d/d alpha = g_hi - g_lo; for the unsigned range lower is a constant zero and d/d alpha = g_hi."""
    x = np.asarray(x, dtype=F32)
    gy = np.asarray(grad_y, dtype=F32)
    lo, hi = F32(lo), F32(hi)
    inside = (x >= lo) & (x <= hi)
    gx = np.where(inside, gy, F32(0)).astype(F32)
    g_hi = gy.astype(np.float64)[x > hi].sum()
    g_lo = gy.astype(np.float64)[x < lo].sum()
    return gx, g_hi, g_lo


# --------------------------------------------------------------------------------------------
# DoReFa (sparsebit/quantization/quantizers/dorefa.py:15-26): tanh squash + abs-max normalise in front of the STE.
def dorefa_normalise(x):
    """dorefa.py:16-17 / :24-25: ``t = x.tanh(); t / t.abs().max()`` in fp32 (numpy's tanh may differ from ATen's by an
    ulp: compare downstream results with a small allowance for rounding flips)."""
    with np.errstate(all="ignore"):
        t = np.tanh(np.asarray(x, dtype=F32)).astype(F32)
        m = np.abs(t).max().astype(F32)
        return (t / m).astype(F32), t, m


def dorefa_forward(x, scale, zero_point, qmin, qmax, ch_axis=0):
    """dorefa.py:15-20: fake-quant of the normalised tensor."""
    xn, _, _ = dorefa_normalise(x)
    return qdq(xn, scale, zero_point, qmin, qmax, ch_axis)


def dorefa_grad_x(x, scale, zero_point, grad_y, qmin, qmax, ch_axis=0):
    """Autograd of the same chain with scale / zero_point as buffers: STE mask (quant_tensor.py:59-64) -> ``/ max`` ->
    tanh' = 1 - t^2, op by op in fp32 like ATen's div / tanh backward."""
    xn, t, m = dorefa_normalise(x)
    gx_ste, _, _ = ste_backward(xn, scale, zero_point, grad_y, qmin, qmax, ch_axis)
    with np.errstate(all="ignore"):
        return ((gx_ste / m).astype(F32) * (F32(1) - (t * t).astype(F32)).astype(F32)).astype(F32)


# --------------------------------------------------------------------------------------------
# AdaRound (sparsebit/quantization/quantizers/adaround.py) -- the quantizer that bypasses STE.
_STRETCH = F32(1.1 - (-0.1))  # zeta - gamma in Python doubles, narrowed to the tensor dtype by ATen
_GAMMA = F32(-0.1)


def _sigmoid(v):
    with np.errstate(all="ignore"):
        return (F32(1) / (F32(1) + np.exp(-np.asarray(v, F32)).astype(F32))).astype(F32)


def adaround_soft_values(v):
    """_get_soft_round_values, adaround.py:40-43: clamp(sigmoid(v) * (zeta - gamma) + gamma, 0, 1)."""
    raw = ((_sigmoid(v) * _STRETCH).astype(F32) + _GAMMA).astype(F32)
    return _clamp_keep_nan(raw, 0, 1), raw


def adaround_forward(x, v, scale, zero_point, qmin, qmax, ch_axis=0, soft=False):
    """_forward, adaround.py:46-54: x_floor = floor(x / scale); + soft values (training) or (v >= 0)
    (eval); clamp(. + zp, qmin, qmax); (. - zp) * scale.  zero_point is NOT rounded here."""
    x = np.asarray(x, F32)
    s, zp = _bcast(scale, x, ch_axis), _bcast(zero_point, x, ch_axis)
    with np.errstate(all="ignore"):
        fl = np.floor((x / s).astype(F32))
        r = adaround_soft_values(v)[0] if soft else (np.asarray(v, F32) >= 0).astype(F32)
        xq = _clamp_keep_nan(((fl + r).astype(F32) + zp).astype(F32), qmin, qmax)
        return ((xq - zp).astype(F32) * s).astype(F32)


def adaround_grad_v(x, v, scale, zero_point, grad_y, qmin, qmax, ch_axis=0):
    """What autograd derives for d(sum(out * grad_y)) / dv in the training branch (fp64 restatement:
    clamp passes gradients on the closed interval, sigmoid' = y (1 - y))."""
    x = np.asarray(x, F32)
    s, zp = _bcast(scale, x, ch_axis), _bcast(zero_point, x, ch_axis)
    with np.errstate(all="ignore"):
        fl = np.floor((x / s).astype(F32))
        soft, raw = adaround_soft_values(v)
        q = ((fl + soft).astype(F32) + zp).astype(F32)
        live = (q >= F32(qmin)) & (q <= F32(qmax)) & (raw >= 0) & (raw <= 1)
        y = _sigmoid(v).astype(np.float64)
        g = np.asarray(grad_y, np.float64) * s.astype(np.float64) * float(_STRETCH) * y * (1 - y)
        return np.where(live, g, 0.0)


def adaround_init(x, scale, ch_axis=0):
    """init_variables, adaround.py:26-32: v = -log((zeta - gamma) / (rest - gamma) - 1) with
    rest = x/scale - floor(x/scale); ATen computes scalar / tensor as reciprocal(tensor) * scalar."""
    x = np.asarray(x, F32)
    s = _bcast(scale, x, ch_axis)
    with np.errstate(all="ignore"):
        qv = (x / s).astype(F32)
        rest = (qv - np.floor(qv)).astype(F32)
        ratio = ((F32(1) / (rest - _GAMMA).astype(F32)).astype(F32) * _STRETCH).astype(F32)
        return (-np.log((ratio - F32(1)).astype(F32))).astype(F32)
