"""Tensor-level wrappers over the C-ABI: torch is used for device memory and streams only.

Every function takes CUDA fp32 tensors, launches on ``torch.cuda.current_stream()`` of the
tensor's device and never synchronises the host.  Non-fp32 / empty / CPU inputs raise
``RuntimeError`` like the reference's pybind modules do (torch_extensions/common.cuh:45-55).
"""
import ctypes

import torch

from . import _lib
from ._lib import SparsebitB200Error, check


def _stream(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def _req(t, name, dtype=torch.float32):
    if not isinstance(t, torch.Tensor):
        raise SparsebitB200Error(f"{name}: expected a torch.Tensor")
    if not t.is_cuda:
        raise SparsebitB200Error(f"{name}: expected a CUDA tensor (sparsebit_b200 has no CPU fallback)")
    if t.dtype != dtype:
        raise SparsebitB200Error(f"Kernel Failure, Invalid dtype of Input tensor: {name}(Expect to be {dtype})")
    if t.numel() == 0:
        raise SparsebitB200Error(f"Kernel Failure, Tensor is empty: {name}")
    if not t.is_contiguous():
        raise SparsebitB200Error(f"{name}: expected a contiguous tensor")
    return t


def channel_geometry(shape, ch_axis):
    """[outer, C, inner] view used by the per-channel kernels (fake_quant_tensor.cu:203-208)."""
    ch_axis = ch_axis % len(shape)
    outer = 1
    for d in shape[:ch_axis]:
        outer *= int(d)
    inner = 1
    for d in shape[ch_axis + 1 :]:
        inner *= int(d)
    return outer, int(shape[ch_axis]), inner


# ----------------------------------------------------------------------------- QDQ forward
def qdq_pertensor(x, scale, zero_point, qmin, qmax, rounding=0, out=None):
    lib = _lib.load()
    _req(x, "data"), _req(scale, "scale"), _req(zero_point, "zero_point")
    out = torch.empty_like(x) if out is None else out
    with torch.cuda.device(x.device):
        check(lib.sb200_qdq_pertensor_fwd(x.data_ptr(), scale.data_ptr(), zero_point.data_ptr(), out.data_ptr(),
                                          x.numel(), int(qmin), int(qmax), int(rounding), _stream(x)))
    return out


def qdq_perchannel(x, scale, zero_point, qmin, qmax, ch_axis, rounding=0, out=None):
    lib = _lib.load()
    _req(x, "data"), _req(scale, "scale"), _req(zero_point, "zero_point")
    outer, c, inner = channel_geometry(x.shape, ch_axis)
    if scale.numel() != c or zero_point.numel() != c:
        raise SparsebitB200Error(f"per-channel qparams need {c} elements (got {scale.numel()}, {zero_point.numel()})")
    out = torch.empty_like(x) if out is None else out
    with torch.cuda.device(x.device):
        check(lib.sb200_qdq_perchannel_fwd(x.data_ptr(), scale.data_ptr(), zero_point.data_ptr(), out.data_ptr(),
                                           outer, c, inner, int(qmin), int(qmax), int(rounding), _stream(x)))
    return out


def qdq_stats_pertensor(x, scale, zero_point, qmin, qmax, state, rounding=0, out=None):
    """Fused QDQ + running min/max of x.  ``state``: int32[2] tensor from ``minmax_new(1)``."""
    lib = _lib.load()
    _req(x, "data"), _req(scale, "scale"), _req(zero_point, "zero_point")
    out = torch.empty_like(x) if out is None else out
    with torch.cuda.device(x.device):
        check(lib.sb200_qdq_stats_pertensor_fwd(x.data_ptr(), scale.data_ptr(), zero_point.data_ptr(), out.data_ptr(),
                                                state.data_ptr(), x.numel(), int(qmin), int(qmax), int(rounding), _stream(x)))
    return out


# ----------------------------------------------------------------------------- STE backward
def clamp_backward(x, grad_y, lo, hi):
    """Backward of ``clamp(x, lo, hi)`` with tensor bounds: (gx, g_hi, g_lo) -- sb200_clamp_bwd (PACT)."""
    lib = _lib.load()
    _req(x, "data"), _req(grad_y, "grad"), _req(lo, "lower"), _req(hi, "alpha")
    if grad_y.shape != x.shape:
        raise SparsebitB200Error("grad_y must have the shape of data")
    gx = torch.empty_like(x)
    g_hi = torch.zeros(1, dtype=torch.float32, device=x.device)
    g_lo = torch.zeros(1, dtype=torch.float32, device=x.device)
    ws_bytes = int(lib.sb200_clamp_bwd_workspace_bytes(x.numel()))
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        check(lib.sb200_clamp_bwd(x.data_ptr(), grad_y.data_ptr(), lo.data_ptr(), hi.data_ptr(), gx.data_ptr(), g_hi.data_ptr(),
                                  g_lo.data_ptr(), x.numel(), ws.data_ptr(), ws_bytes, _stream(x)))
    return gx, g_hi, g_lo


BWD_GZP_CLOSED = 1  # include/sparsebit_b200.h SB200_BWD_GZP_CLOSED


def qdq_backward(x, scale, zero_point, grad_y, qmin, qmax, ch_axis=None, rounding=0, need_gs=True, need_gzp=True,
                 gzp_closed=False, out=None):
    """Returns (gx, gs, gzp); gs / gzp shaped like scale / zero_point (zeros when not requested,
    like the reference which returns zeros_like, fake_quant_tensor.cu:147-149).  Per-channel zero-point
    gradient: by default the reference kernel's rule (vq == qmax counts as clipped, fake_quant_tensor.cu:264);
    ``gzp_closed=True`` selects MySTE.backward's closed interval (quant_tensor.py:62-69).  ``out``: optional
    contiguous fp32 tensor shaped like x that receives gx."""
    lib = _lib.load()
    _req(x, "data"), _req(scale, "scale"), _req(zero_point, "zero_point"), _req(grad_y, "grad")
    if grad_y.shape != x.shape:
        raise SparsebitB200Error("grad_y must have the shape of data")
    gx = torch.empty_like(x) if out is None else _req(out, "grad_x")
    if gx.shape != x.shape:
        raise SparsebitB200Error("out must have the shape of data")
    gs = torch.zeros_like(scale)
    gzp = torch.zeros_like(zero_point)
    if ch_axis is None:
        outer, c, inner = 1, 1, x.numel()
    else:
        outer, c, inner = channel_geometry(x.shape, ch_axis)
        if scale.numel() != c or zero_point.numel() != c:
            raise SparsebitB200Error(f"per-channel qparams need {c} elements (got {scale.numel()}, {zero_point.numel()})")
    need = need_gs or need_gzp
    ws_bytes = int(lib.sb200_qdq_bwd_workspace_bytes(outer, c, inner)) if need else 0
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        if ch_axis is None:
            check(lib.sb200_qdq_pertensor_bwd(x.data_ptr(), scale.data_ptr(), zero_point.data_ptr(), grad_y.data_ptr(),
                                              gx.data_ptr(), gs.data_ptr() if need_gs else None,
                                              gzp.data_ptr() if need_gzp else None, x.numel(), int(qmin), int(qmax),
                                              int(rounding), ws.data_ptr(), ws_bytes, _stream(x)))
        else:
            check(lib.sb200_qdq_perchannel_bwd_ex(x.data_ptr(), scale.data_ptr(), zero_point.data_ptr(), grad_y.data_ptr(),
                                                  gx.data_ptr(), gs.data_ptr() if need_gs else None,
                                                  gzp.data_ptr() if need_gzp else None, outer, c, inner, int(qmin),
                                                  int(qmax), int(rounding), BWD_GZP_CLOSED if gzp_closed else 0,
                                                  ws.data_ptr(), ws_bytes, _stream(x)))
    return gx, gs, gzp


# ----------------------------------------------------------------------------- multi-tensor weight QDQ
class _QdqTensorDesc(ctypes.Structure):  # include/sparsebit_b200.h sb200_qdq_tensor_desc
    _fields_ = [("x", ctypes.c_void_p), ("mask", ctypes.c_void_p), ("scale", ctypes.c_void_p), ("zero_point", ctypes.c_void_p),
                ("out", ctypes.c_void_p), ("outer", ctypes.c_int64), ("channels", ctypes.c_int64), ("inner", ctypes.c_int64),
                ("qmin", ctypes.c_int), ("qmax", ctypes.c_int)]


class QdqMulti:
    """(mask-apply +) per-channel QDQ of many tensors in ONE launch (sb200_qdq_multi_plan / _run).

    ``items``: iterable of dicts ``x, scale, zero_point, qmin, qmax`` and optional ``mask`` (bool / uint8),
    ``out`` (default: a new tensor), ``ch_axis`` (default 0).  The plan keeps references to every tensor; ``run()``
    re-reads their CURRENT contents (the weights of a training step), one kernel launch per call."""

    def __init__(self, items):
        lib = _lib.load()
        self.items = []
        descs = []
        for it in items:
            x = _req(it["x"], "data")
            scale = _req(it["scale"].reshape(-1), "scale")
            zp = _req(it["zero_point"].reshape(-1), "zero_point")
            outer, c, inner = channel_geometry(x.shape, it.get("ch_axis", 0))
            if scale.numel() != c or zp.numel() != c:
                raise SparsebitB200Error(f"per-channel qparams need {c} elements (got {scale.numel()}, {zp.numel()})")
            mask = it.get("mask")
            if mask is not None:
                if mask.dtype not in (torch.bool, torch.uint8) or mask.shape != x.shape or not mask.is_contiguous():
                    raise SparsebitB200Error("mask must be a contiguous bool / uint8 tensor shaped like the data")
            out = it.get("out")
            out = torch.empty_like(x) if out is None else _req(out, "out")
            self.items.append((x, mask, scale, zp, out))
            descs.append(_QdqTensorDesc(x.data_ptr(), mask.data_ptr() if mask is not None else None, scale.data_ptr(),
                                        zp.data_ptr(), out.data_ptr(), outer, c, inner, int(it["qmin"]), int(it["qmax"])))
        if not descs:
            raise SparsebitB200Error("QdqMulti: no tensors")
        self.device = self.items[0][0].device
        self.count = len(descs)
        arr = (_QdqTensorDesc * self.count)(*descs)
        self.table = torch.empty(int(lib.sb200_qdq_multi_table_bytes(self.count)), dtype=torch.uint8, device=self.device)
        rows = ctypes.c_int64(0)
        with torch.cuda.device(self.device):
            check(lib.sb200_qdq_multi_plan(arr, self.count, self.table.data_ptr(), self.table.numel(), ctypes.byref(rows),
                                           torch.cuda.current_stream(self.device).cuda_stream))
        self.total_rows = rows.value
        self.outputs = [it[4] for it in self.items]

    def run(self):
        with torch.cuda.device(self.device):
            check(_lib.load().sb200_qdq_multi_run(self.table.data_ptr(), self.count, self.total_rows,
                                                  torch.cuda.current_stream(self.device).cuda_stream))
        return self.outputs


# ----------------------------------------------------------------------------- row moments
MOMENTS = 5  # sum x, sum x^2, sum |x|, sum |x - c|, sum (x - c)^2


def moments_new(rows, device):
    return torch.zeros(rows, MOMENTS, dtype=torch.float64, device=device)


def moments_update(x2d, out, centre=None):
    """Accumulate the fp64 row moments of x2d [rows, row_len] into ``out`` [rows, 5] (deterministic order)."""
    lib = _lib.load()
    _req(x2d, "data")
    if x2d.dim() != 2 or out.shape != (x2d.shape[0], MOMENTS) or out.dtype != torch.float64:
        raise SparsebitB200Error("moments_update: x2d must be [rows, row_len] and out float64 [rows, 5]")
    if centre is not None and (centre.dtype != torch.float64 or centre.numel() != x2d.shape[0]):
        raise SparsebitB200Error("moments_update: centre must hold one float64 per row")
    rows, row_len = x2d.shape
    ws_bytes = int(lib.sb200_moments_workspace_bytes(rows, row_len))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x2d.device)
    with torch.cuda.device(x2d.device):
        check(lib.sb200_observe_moments(x2d.data_ptr(), rows, row_len, centre.data_ptr() if centre is not None else None,
                                        out.data_ptr(), ws.data_ptr(), ws_bytes, _stream(x2d)))
    return out


# ----------------------------------------------------------------------------- DoReFa
def dorefa_absmax(x):
    """max |tanh(x)| as a one-element float tensor (dorefa.py:16-17), one 4 B/elem pass."""
    lib = _lib.load()
    _req(x, "data")
    m = torch.zeros(1, dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        check(lib.sb200_dorefa_absmax(x.data_ptr(), x.numel(), m.data_ptr(), _stream(x)))
    return m


def dorefa_forward(x, absmax, scale=None, zero_point=None, qmin=0, qmax=0, ch_axis=None):
    """tanh(x) / absmax, fake-quantised when qparams are given (dorefa.py:15-20); without them the normalised tensor
    the observer sees (dorefa.py:22-26)."""
    lib = _lib.load()
    _req(x, "data"), _req(absmax, "absmax")
    quantize = scale is not None
    if quantize:
        _req(scale, "scale"), _req(zero_point, "zero_point")
        outer, c, inner = _adaround_geometry(x, scale, ch_axis)
        if zero_point.numel() != c:
            raise SparsebitB200Error(f"dorefa: qparams need {c} elements (got {zero_point.numel()})")
    else:
        outer, c, inner = 1, 1, x.numel()
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        check(lib.sb200_dorefa_fwd(x.data_ptr(), absmax.data_ptr(), scale.data_ptr() if quantize else None,
                                   zero_point.data_ptr() if quantize else None, out.data_ptr(), outer, c, inner,
                                   int(qmin), int(qmax), int(quantize), _stream(x)))
    return out


def dorefa_backward(x, absmax, scale, zero_point, grad_y, qmin, qmax, ch_axis=None):
    """Gradient of dorefa_forward with respect to x (STE mask -> / absmax -> tanh'), one 12 B/elem pass."""
    lib = _lib.load()
    _req(x, "data"), _req(absmax, "absmax"), _req(scale, "scale"), _req(zero_point, "zero_point"), _req(grad_y, "grad")
    if grad_y.shape != x.shape:
        raise SparsebitB200Error("dorefa: grad_y must have the shape of data")
    outer, c, inner = _adaround_geometry(x, scale, ch_axis)
    if zero_point.numel() != c:
        raise SparsebitB200Error(f"dorefa: qparams need {c} elements (got {zero_point.numel()})")
    gx = torch.empty_like(x)
    with torch.cuda.device(x.device):
        check(lib.sb200_dorefa_bwd(x.data_ptr(), absmax.data_ptr(), scale.data_ptr(), zero_point.data_ptr(), grad_y.data_ptr(),
                                   gx.data_ptr(), outer, c, inner, int(qmin), int(qmax), _stream(x)))
    return gx


# ----------------------------------------------------------------------------- AdaRound
def _adaround_geometry(x, scale, ch_axis):
    if ch_axis is None:
        outer, c, inner = 1, 1, x.numel()
    else:
        outer, c, inner = channel_geometry(x.shape, ch_axis)
    if scale.numel() != c:
        raise SparsebitB200Error(f"adaround: qparams need {c} elements (got {scale.numel()})")
    return outer, c, inner


def adaround_forward(x, v, scale, zero_point, qmin, qmax, ch_axis=None, soft=False, out=None):
    """adaround.py:46-54; soft=True is the training branch, soft=False the (exact) eval branch."""
    lib = _lib.load()
    _req(x, "data"), _req(v, "v"), _req(scale, "scale"), _req(zero_point, "zero_point")
    if v.shape != x.shape:
        raise SparsebitB200Error("adaround: v must have the shape of data")
    outer, c, inner = _adaround_geometry(x, scale, ch_axis)
    out = torch.empty_like(x) if out is None else out
    with torch.cuda.device(x.device):
        check(lib.sb200_adaround_fwd(x.data_ptr(), v.data_ptr(), scale.data_ptr(), zero_point.data_ptr(), out.data_ptr(),
                                     outer, c, inner, int(qmin), int(qmax), int(bool(soft)), _stream(x)))
    return out


def adaround_backward(x, v, scale, zero_point, grad_y, qmin, qmax, ch_axis=None):
    lib = _lib.load()
    _req(x, "data"), _req(v, "v"), _req(scale, "scale"), _req(zero_point, "zero_point"), _req(grad_y, "grad")
    if v.shape != x.shape or grad_y.shape != x.shape:
        raise SparsebitB200Error("adaround: v and grad_y must have the shape of data")
    outer, c, inner = _adaround_geometry(x, scale, ch_axis)
    gv = torch.empty_like(x)
    with torch.cuda.device(x.device):
        check(lib.sb200_adaround_bwd(x.data_ptr(), v.data_ptr(), scale.data_ptr(), zero_point.data_ptr(),
                                     grad_y.data_ptr(), gv.data_ptr(), outer, c, inner, int(qmin), int(qmax), _stream(x)))
    return gv


def adaround_init(x, scale, ch_axis=None):
    """adaround.py:26-32."""
    lib = _lib.load()
    _req(x, "data"), _req(scale, "scale")
    outer, c, inner = _adaround_geometry(x, scale, ch_axis)
    v = torch.empty_like(x)
    with torch.cuda.device(x.device):
        check(lib.sb200_adaround_init(x.data_ptr(), scale.data_ptr(), v.data_ptr(), outer, c, inner, _stream(x)))
    return v


# ----------------------------------------------------------------------------- MinMax
def minmax_new(channels, device):
    """Fresh running min/max state: int32[2*C] (bit pattern of the uint32 ordered keys)."""
    lib = _lib.load()
    st = torch.empty(2 * channels, dtype=torch.int32, device=device)
    with torch.cuda.device(st.device):
        check(lib.sb200_minmax_init(st.data_ptr(), channels, _stream(st)))
    return st


def minmax_update(x, state, ch_axis=None):
    lib = _lib.load()
    _req(x, "data")
    with torch.cuda.device(x.device):
        if ch_axis is None:
            check(lib.sb200_observe_minmax(x.data_ptr(), x.numel(), state.data_ptr(), _stream(x)))
        else:
            outer, c, inner = channel_geometry(x.shape, ch_axis)
            if state.numel() != 2 * c:
                raise SparsebitB200Error(f"minmax state holds {state.numel() // 2} channels, data has {c}")
            check(lib.sb200_observe_minmax_perchannel(x.data_ptr(), outer, c, inner, state.data_ptr(), _stream(x)))


def minmax_read(state):
    lib = _lib.load()
    c = state.numel() // 2
    mn = torch.empty(c, dtype=torch.float32, device=state.device)
    mx = torch.empty(c, dtype=torch.float32, device=state.device)
    with torch.cuda.device(state.device):
        check(lib.sb200_minmax_read(state.data_ptr(), c, mn.data_ptr(), mx.data_ptr(), _stream(state)))
    return mn, mx


class _QparamsDesc(ctypes.Structure):  # include/sparsebit_b200.h sb200_minmax_qparams_desc
    _fields_ = [("state", ctypes.c_void_p), ("out_min", ctypes.c_void_p), ("out_max", ctypes.c_void_p), ("out_scale", ctypes.c_void_p),
                ("out_zero_point", ctypes.c_void_p), ("channels", ctypes.c_int64), ("qmin", ctypes.c_int), ("qmax", ctypes.c_int),
                ("symmetric", ctypes.c_int)]


def minmax_qparams_multi(requests):
    """``requests``: [(state int32[2C], qmin, qmax, symmetric)] -> [(min, max, scale, zero_point)] float32[C] views of one
    buffer, computed by ONE launch (sb200_minmax_qparams_multi)."""
    lib = _lib.load()
    if not requests:
        return []
    dev = requests[0][0].device
    chans = [r[0].numel() // 2 for r in requests]
    total = sum(chans)
    flat = torch.empty(4, total, dtype=torch.float32, device=dev)
    table = torch.empty(64 * len(requests), dtype=torch.uint8, device=dev)
    descs, outs, off = [], [], 0
    base, plane = flat.data_ptr(), total * 4
    for (state, qmin, qmax, sym), c in zip(requests, chans):
        p = base + off * 4
        descs.append(_QparamsDesc(state.data_ptr(), p, p + plane, p + 2 * plane, p + 3 * plane, c, int(qmin), int(qmax), int(bool(sym))))
        outs.append(tuple(flat[k, off:off + c] for k in range(4)))
        off += c
    arr = (_QparamsDesc * len(descs))(*descs)
    with torch.cuda.device(dev):
        check(lib.sb200_minmax_qparams_multi(arr, len(descs), table.data_ptr(), table.numel(), torch.cuda.current_stream(dev).cuda_stream))
    return outs


# ----------------------------------------------------------------------------- histogram / MSE
def hist_update(x, range_lo_hi, counts):
    """counts (int64[bins]) += histc(x, bins, lo, hi); ``range_lo_hi``: device float32[2]."""
    lib = _lib.load()
    _req(x, "data"), _req(range_lo_hi, "range")
    with torch.cuda.device(x.device):
        check(lib.sb200_observe_hist(x.data_ptr(), x.numel(), range_lo_hi.data_ptr(), counts.numel(), counts.data_ptr(), _stream(x)))


def mse_sweep(x2d, cand_scale, cand_zp, qmin, qmax, sse):
    """sse[rows, ncand] (fp64) += sum_j (x - qdq_i(x))^2 for every candidate i; x2d: [rows, row_len]."""
    lib = _lib.load()
    _req(x2d, "data"), _req(cand_scale, "cand_scale"), _req(cand_zp, "cand_zp")
    rows, row_len = x2d.shape
    ncand = cand_scale.numel() // rows
    ws_bytes = int(lib.sb200_mse_workspace_bytes(rows, row_len, ncand))
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=x2d.device)
    with torch.cuda.device(x2d.device):
        check(lib.sb200_observe_mse_sweep(x2d.data_ptr(), rows, row_len, cand_scale.data_ptr(), cand_zp.data_ptr(), ncand,
                                          int(qmin), int(qmax), sse.data_ptr(), ws.data_ptr(), ws_bytes, _stream(x2d)))


# ----------------------------------------------------------------------------- radix select
class RadixSelect:
    """Exact order statistics over one or more device tensors (3 passes x 4 B/elem).

    rows x ntargets_per_row independent selections; ``add_pass(p, tensors)`` accumulates the
    digit histograms of pass p for every tensor (each viewed as [rows, row_len]); an optional
    ``reduce`` callback (SUM all-reduce across GPUs) runs between histogram and scan."""

    def __init__(self, rows, ntargets_per_row, device, key_mode=0):
        self.lib = _lib.load()
        self.rows, self.ntpr, self.key_mode = rows, ntargets_per_row, key_mode
        n = rows * ntargets_per_row
        self.sel = torch.zeros(n * _lib.SELECT_STATE_WORDS, dtype=torch.int64, device=device)
        self.hist = torch.zeros(n * _lib.SELECT_BINS, dtype=torch.int64, device=device)
        self.counts = torch.zeros(rows * 2, dtype=torch.int64, device=device)
        with torch.cuda.device(device):
            check(self.lib.sb200_select_init(self.sel.data_ptr(), self.hist.data_ptr(), n, None, _stream(self.sel)))

    def set_ranks(self, ranks):
        """ranks: int64 device tensor [rows * ntpr] of 0-based ranks."""
        self.sel.view(-1, _lib.SELECT_STATE_WORDS)[:, 1] = ranks.to(torch.int64)

    def hist_pass(self, p, x2d, with_counts=False):
        _req(x2d, "data")
        rows, row_len = x2d.shape
        with torch.cuda.device(x2d.device):
            if with_counts and p == 0:
                check(self.lib.sb200_select_hist_counts(x2d.data_ptr(), rows, row_len, self.ntpr, self.sel.data_ptr(),
                                                        self.hist.data_ptr(), p, self.key_mode, self.counts.data_ptr(), _stream(x2d)))
            else:
                check(self.lib.sb200_select_hist(x2d.data_ptr(), rows, row_len, self.ntpr, self.sel.data_ptr(),
                                                 self.hist.data_ptr(), p, self.key_mode, _stream(x2d)))

    def percentile_ranks(self, total, alpha):
        """total: int64 device tensor [rows] (elements per row incl. NaN)."""
        with torch.cuda.device(self.sel.device):
            check(self.lib.sb200_percentile_ranks(self.counts.data_ptr(), total.data_ptr(), self.rows, float(alpha),
                                                  self.sel.data_ptr(), _stream(self.sel)))

    def scan(self, p):
        with torch.cuda.device(self.sel.device):
            check(self.lib.sb200_select_scan(self.sel.data_ptr(), self.hist.data_ptr(), self.rows, self.ntpr, p, _stream(self.sel)))

    def values(self):
        n = self.rows * self.ntpr
        out = torch.empty(n, dtype=torch.float32, device=self.sel.device)
        with torch.cuda.device(self.sel.device):
            check(self.lib.sb200_select_read(self.sel.data_ptr(), n, self.key_mode, out.data_ptr(), _stream(self.sel)))
        return out


def kth_value(x, k, key_mode=0):
    """k-th smallest (0-based) of a flat tensor, exact; key_mode 1 ranks |x|."""
    if not 0 <= int(k) < x.numel():
        raise SparsebitB200Error(f"kth_value: k must be in [0, {x.numel()}) (got {k})")
    rs = RadixSelect(1, 1, x.device, key_mode)
    rs.set_ranks(torch.tensor([k], dtype=torch.int64, device=x.device))
    x2 = x.reshape(1, -1)
    for p in range(3):
        rs.hist_pass(p, x2)
        rs.scan(p)
    return rs.values()


# ----------------------------------------------------------------------------- sparser
def mask_gt(w, thresh):
    lib = _lib.load()
    _req(w, "weight"), _req(thresh, "thresh")
    mask = torch.empty(w.shape, dtype=torch.bool, device=w.device)
    with torch.cuda.device(w.device):
        check(lib.sb200_mask_gt(w.data_ptr(), thresh.data_ptr(), mask.data_ptr(), w.numel(), _stream(w)))
    return mask


def mask_rows_gt(score, thresh, shape):
    """Float mask of ``shape`` = [rows, ...]: row r is all ones if score[r] > thresh else all zeros."""
    lib = _lib.load()
    _req(score, "score"), _req(thresh, "thresh")
    rows = int(shape[0])
    if score.numel() != rows:
        raise SparsebitB200Error("mask_rows_gt: one score per row expected")
    mask = torch.empty(tuple(shape), dtype=torch.float32, device=score.device)
    with torch.cuda.device(score.device):
        check(lib.sb200_mask_rows_gt(score.data_ptr(), thresh.data_ptr(), mask.data_ptr(), rows, mask.numel() // rows,
                                     _stream(score)))
    return mask


def mask_apply(w, mask, out=None):
    lib = _lib.load()
    _req(w, "weight")
    if mask.shape != w.shape or not mask.is_cuda or not mask.is_contiguous():
        raise SparsebitB200Error("mask must be a contiguous CUDA tensor of the weight's shape")
    out = torch.empty_like(w) if out is None else out
    with torch.cuda.device(w.device):
        if mask.dtype in (torch.bool, torch.uint8):
            check(lib.sb200_mask_apply(w.data_ptr(), mask.data_ptr(), out.data_ptr(), w.numel(), _stream(w)))
        elif mask.dtype == torch.float32:
            check(lib.sb200_mask_apply_f32(w.data_ptr(), mask.data_ptr(), out.data_ptr(), w.numel(), _stream(w)))
        else:
            raise SparsebitB200Error(f"unsupported mask dtype {mask.dtype}")
    return out


def mask_apply_qdq_perchannel(w, mask, scale, zero_point, qmin, qmax, ch_axis=0, rounding=0, out=None):
    lib = _lib.load()
    _req(w, "weight"), _req(scale, "scale"), _req(zero_point, "zero_point")
    if mask.dtype not in (torch.bool, torch.uint8) or mask.shape != w.shape or not mask.is_contiguous():
        raise SparsebitB200Error("fused mask+QDQ needs a contiguous bool mask of the weight's shape")
    outer, c, inner = channel_geometry(w.shape, ch_axis)
    out = torch.empty_like(w) if out is None else out
    with torch.cuda.device(w.device):
        check(lib.sb200_mask_apply_qdq_perchannel(w.data_ptr(), mask.data_ptr(), scale.data_ptr(), zero_point.data_ptr(),
                                                  out.data_ptr(), outer, c, inner, int(qmin), int(qmax), int(rounding), _stream(w)))
    return out


# ----------------------------------------------------------------------------- GPTQ
_gptq_ws = {}


class _Gptq4Options(ctypes.Structure):  # include/sparsebit_b200.h sb200_gptq4_options
    _fields_ = [("impl", ctypes.c_int), ("chunk_k", ctypes.c_int), ("flags", ctypes.c_int), ("reserved", ctypes.c_int * 5)]


GPTQ4_STATIC_WEIGHTS = 1  # include/sparsebit_b200.h SB200_GPTQ4_STATIC_WEIGHTS


def gptq4_matmul(x, qweight, out, scales, zeros, group_size=0, impl=None, chunk_k=0, static_weights=False):
    """In-place ``out += x @ dequant(qweight)`` (vecquant4matmul contract, cuda_kernel.cpp:10-23).
    ``impl`` / ``chunk_k``: per-call kernel selection (sb200_gptq4_matmul_ex); None = the library default.
    ``static_weights``: qweight / scales / zeros are constants of the model (not written by the kernel just in front on
    the stream), so the decode kernel may fetch them while its predecessor is still draining."""
    lib = _lib.load()
    _req(x, "inp1"), _req(out, "out"), _req(scales, "scales"), _req(zeros, "zeros")
    _req(qweight, "inp2", torch.int32)
    if x.dim() < 2:
        raise SparsebitB200Error("input1 must be with dimension >= 2")  # cuda_kernel_4bit.cu:44
    if qweight.dim() != 2:
        raise SparsebitB200Error("input2 must be with dimension == 2")  # cuda_kernel_4bit.cu:48
    k = x.shape[-1]
    m = x.numel() // k
    n = qweight.shape[1]
    if out.shape[-1] != n:
        raise SparsebitB200Error("output channel must be the same with input2 out_channel")  # :52
    ws_bytes = int(lib.sb200_gptq4_workspace_bytes(m, k, n, int(group_size)))
    ws = None
    if ws_bytes:
        key = (x.device, torch.cuda.current_stream(x.device).cuda_stream)
        ws = _gptq_ws.get(key)
        if ws is None or ws.numel() < ws_bytes:
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
            _gptq_ws[key] = ws
    with torch.cuda.device(x.device):
        if impl is None and not chunk_k and not static_weights:
            check(lib.sb200_gptq4_matmul(x.data_ptr(), qweight.data_ptr(), out.data_ptr(), scales.data_ptr(), zeros.data_ptr(),
                                         m, k, n, qweight.shape[0], int(group_size), ws.data_ptr() if ws is not None else None,
                                         ws_bytes, _stream(x)))
        else:
            opts = _Gptq4Options(int(impl or 0), int(chunk_k), GPTQ4_STATIC_WEIGHTS if static_weights else 0)
            check(lib.sb200_gptq4_matmul_ex(x.data_ptr(), qweight.data_ptr(), out.data_ptr(), scales.data_ptr(),
                                            zeros.data_ptr(), m, k, n, qweight.shape[0], int(group_size), ctypes.byref(opts),
                                            ws.data_ptr() if ws is not None else None, ws_bytes, _stream(x)))
    return out


class _Gptq4Problem(ctypes.Structure):  # include/sparsebit_b200.h sb200_gptq4_problem
    _fields_ = [("x", ctypes.c_void_p), ("qweight", ctypes.c_void_p), ("out", ctypes.c_void_p), ("scales", ctypes.c_void_p),
                ("zeros", ctypes.c_void_p), ("k", ctypes.c_int64), ("n", ctypes.c_int64), ("qweight_rows", ctypes.c_int64),
                ("group_size", ctypes.c_int)]


def gptq4_matmul_batch(problems, group_size=0, static_weights=False):
    """Up to 4 decode-sized linears sharing M in ONE launch (q / k / v, gate / up): ``problems`` = [(x, qweight, out, scales,
    zeros)], every ``out`` pre-initialised and accumulated in place (sb200_gptq4_matmul_batch[_ex])."""
    lib = _lib.load()
    m = None
    arr = (_Gptq4Problem * len(problems))()
    for i, (x, qw, out, sc, zr) in enumerate(problems):
        _req(x, "inp1"), _req(out, "out"), _req(sc, "scales"), _req(zr, "zeros"), _req(qw, "inp2", torch.int32)
        k = x.shape[-1]
        mi = x.numel() // k
        if m is None:
            m = mi
        elif mi != m:
            raise SparsebitB200Error("gptq4_matmul_batch: all problems must have the same number of tokens")
        if out.shape[-1] != qw.shape[1]:
            raise SparsebitB200Error("output channel must be the same with input2 out_channel")
        arr[i] = _Gptq4Problem(x.data_ptr(), qw.data_ptr(), out.data_ptr(), sc.data_ptr(), zr.data_ptr(), k, qw.shape[1], qw.shape[0],
                               int(group_size))
    dev = problems[0][0].device
    with torch.cuda.device(dev):
        check(lib.sb200_gptq4_matmul_batch_ex(arr, len(problems), m, GPTQ4_STATIC_WEIGHTS if static_weights else 0,
                                              torch.cuda.current_stream(dev).cuda_stream))
    return [p[2] for p in problems]


_gptq_state = {}  # (device, stream) -> zero-initialised, self-resetting arrival counters of the single-launch decode path


def gptq4_linear_f16(x, qweight, scales, zeros, bias=None, group_size=0, static_weights=False, single_launch=True):
    """fp16 activations in, fp16 ``bias + x @ dequant(qweight)`` out, no eager casts (sb200_gptq4_linear_f16_ex).
    Decode-sized M (<= 32) is ONE kernel launch; ``single_launch=False`` keeps the staged path (cast, bias, kernel, cast).
    ``static_weights``: see ``gptq4_matmul``."""
    lib = _lib.load()
    _req(x, "inp1", torch.float16), _req(scales, "scales"), _req(zeros, "zeros"), _req(qweight, "inp2", torch.int32)
    if bias is not None:
        _req(bias, "bias")
    k = x.shape[-1]
    m = x.numel() // k
    n = qweight.shape[1]
    out = torch.empty(x.shape[:-1] + (n,), dtype=torch.float16, device=x.device)
    ws_bytes = int(lib.sb200_gptq4_linear_f16_workspace_bytes(m, k, n, int(group_size)))
    key = (x.device, torch.cuda.current_stream(x.device).cuda_stream, "f16")
    ws = _gptq_ws.get(key)
    if ws is None or ws.numel() < ws_bytes:
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        _gptq_ws[key] = ws
    state = None
    if single_launch and m <= 32:
        skey = key[:2]
        state = _gptq_state.get(skey)
        if state is None:
            state = torch.zeros(int(lib.sb200_gptq4_linear_f16_state_bytes()), dtype=torch.uint8, device=x.device)
            _gptq_state[skey] = state
    with torch.cuda.device(x.device):
        check(lib.sb200_gptq4_linear_f16_ex(x.data_ptr(), qweight.data_ptr(), out.data_ptr(), bias.data_ptr() if bias is not None else None,
                                            scales.data_ptr(), zeros.data_ptr(), m, k, n, qweight.shape[0], int(group_size),
                                            state.data_ptr() if state is not None else None,
                                            GPTQ4_STATIC_WEIGHTS if static_weights else 0, ws.data_ptr(), ws_bytes, _stream(x)))
    return out


def gptq_matmul(x, qweight, out, scales, zeros, bits, group_size=0):
    """In-place ``out += x @ dequant(qweight)`` for 2 / 3 / 4-bit GPTQ weights
    (vecquant{2,3,4}matmul / vecgroupquant{2,3,4}matmul, cuda_kernel.cpp:10-57)."""
    if int(bits) == 4:
        return gptq4_matmul(x, qweight, out, scales, zeros, group_size)
    lib = _lib.load()
    _req(x, "inp1"), _req(out, "out"), _req(scales, "scales"), _req(zeros, "zeros")
    _req(qweight, "inp2", torch.int32)
    if x.dim() < 2:
        raise SparsebitB200Error("input1 must be with dimension >= 2")  # cuda_kernel_3bit.cu:40
    if qweight.dim() != 2:
        raise SparsebitB200Error("input2 must be with dimension == 2")  # cuda_kernel_3bit.cu:44
    k = x.shape[-1]
    m = x.numel() // k
    n = qweight.shape[1]
    if out.shape[-1] != n:
        raise SparsebitB200Error("output channel must be the same with input2 out_channel")  # :48
    with torch.cuda.device(x.device):
        check(lib.sb200_gptq_matmul(x.data_ptr(), qweight.data_ptr(), out.data_ptr(), scales.data_ptr(), zeros.data_ptr(),
                                    m, k, n, qweight.shape[0], int(bits), int(group_size), None, 0, _stream(x)))
    return out
