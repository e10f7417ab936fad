"""Oracle: GPTQ int4 (and 3 / 2-bit) group-wise packing, parameter search and dequant-matmul (numpy)."""
import numpy as np

F32 = np.float32


def find_params_int4(w, groupsize=-1):
    """Quantizer.configure(bit=4, perchannel=True, sym=False, mse=False) + find_params(weight=True)
    -- large_language_models/llama/quantization/utils/quant.py:43-89,117-124.
    w: [N, K] fp32.  Returns scale, zero of shape [N, G] (G = K // groupsize or 1)."""
    w = np.asarray(w, dtype=F32)
    n, k = w.shape
    g = 1 if groupsize == -1 else k // groupsize
    x = w.reshape(n * g, -1)
    maxq = F32(15)
    xmin = np.minimum(x.min(1), F32(0))
    xmax = np.maximum(x.max(1), F32(0))
    both0 = (xmin == 0) & (xmax == 0)
    xmin = np.where(both0, F32(-1), xmin)
    xmax = np.where(both0, F32(1), xmax)
    scale = ((xmax - xmin) / maxq).astype(F32)
    zero = np.rint((-xmin / scale).astype(F32)).astype(F32)
    return scale.reshape(n, g), zero.reshape(n, g)


def quantize_weight(w, scale, zero, groupsize=-1, bit=4):
    """quantize() utils/quant.py:8-10 applied group-wise as in test_cuda_kernel.py:31-36."""
    w = np.asarray(w, dtype=F32)
    n, k = w.shape
    g = scale.shape[1]
    x = w.reshape(n, g, -1)
    s = scale.reshape(n, g, 1)
    z = zero.reshape(n, g, 1)
    q = np.clip(np.rint((x / s).astype(F32)) + z, 0, 2**bit - 1).astype(F32)
    return (s * (q - z)).astype(F32).reshape(n, k)


def pack_int4(w, scale, zero):
    """QuantLinear.pack for bit=4 -- utils/quant.py:187-225: zeros = zero*scale;
    intweight = round((w + zeros) / scales); 8 nibbles per int32 along K, LSB = lowest k;
    qweight [ceil(K/8), N]."""
    w = np.asarray(w, dtype=F32)
    n, k = w.shape
    g = scale.shape[1]
    zeros = (zero * scale).astype(F32)
    iw = np.rint(((w.reshape(n, g, -1) + zeros[:, :, None]) / scale[:, :, None]).astype(F32)).astype(np.int64)
    iw = iw.reshape(n, k).T.astype(np.uint32)  # [K, N]
    rows = (k + 7) // 8
    pad = np.zeros((rows * 8, n), dtype=np.uint32)
    pad[:k] = iw
    q = np.zeros((rows, n), dtype=np.uint32)
    for j in range(8):
        q |= pad[j::8] << np.uint32(4 * j)
    return q.view(np.int32), scale.astype(F32), zeros


def unpack_int4(qweight, k):
    """Inverse of the packing: returns uint nibbles [K, N]."""
    q = np.asarray(qweight).view(np.uint32)
    rows, n = q.shape
    out = np.zeros((rows * 8, n), dtype=np.uint32)
    for j in range(8):
        out[j::8] = (q >> np.uint32(4 * j)) & np.uint32(0xF)
    return out[:k]


def find_params(w, bit=4, groupsize=-1):
    """find_params_int4 for any bit width: maxq = 2^bit - 1 (utils/quant.py:43-89)."""
    w = np.asarray(w, dtype=F32)
    n, k = w.shape
    g = 1 if groupsize == -1 else k // groupsize
    x = w.reshape(n * g, -1)
    xmin = np.minimum(x.min(1), F32(0))
    xmax = np.maximum(x.max(1), F32(0))
    both0 = (xmin == 0) & (xmax == 0)
    xmin = np.where(both0, F32(-1), xmin)
    xmax = np.where(both0, F32(1), xmax)
    scale = ((xmax - xmin) / F32(2**bit - 1)).astype(F32)
    zero = np.rint((-xmin / scale).astype(F32)).astype(F32)
    return scale.reshape(n, g), zero.reshape(n, g)


def _bit_slots(bit, k):
    """For every input channel i < k: (row, shift, spill_row, spill_shift) of QuantLinear.pack's layout
    (utils/quant.py:210-258).  2/4-bit: 32/bit values per word.  3-bit: 32 values in 3 words; value 10
    keeps 2 bits in word 0 (<< 30) and 1 in word 1 (>> 2); value 21 keeps 1 bit in word 1 (<< 31) and 2 in
    word 2 (>> 1)."""
    slots = []
    for i in range(k):
        if bit in (2, 4):
            per = 32 // bit
            slots.append((i // per, bit * (i % per), None, 0))
            continue
        u, j = divmod(i, 32)
        if j < 10:
            slots.append((3 * u, 3 * j, None, 0))
        elif j == 10:
            slots.append((3 * u, 30, 3 * u + 1, 2))
        elif j < 21:
            slots.append((3 * u + 1, 3 * (j - 11) + 1, None, 0))
        elif j == 21:
            slots.append((3 * u + 1, 31, 3 * u + 2, 1))
        else:
            slots.append((3 * u + 2, 3 * (j - 22) + 2, None, 0))
    return slots


def packed_rows(k, bit):
    """ceil(K*bit / (32*p)) * p, p = 3 for 3-bit (utils/quant.py:172-184)."""
    p = 3 if bit == 3 else 1
    return -(-k * bit // (32 * p)) * p


def pack_bits(w, scale, zero, bit):
    """QuantLinear.pack for bit in {2, 3, 4} -- utils/quant.py:187-260."""
    w = np.asarray(w, dtype=F32)
    n, k = w.shape
    g = scale.shape[1]
    zeros = (zero * scale).astype(F32)
    iw = np.rint(((w.reshape(n, g, -1) + zeros[:, :, None]) / scale[:, :, None]).astype(F32)).astype(np.int64)
    return pack_values(iw.reshape(n, k).T, bit), scale.astype(F32), zeros


def pack_values(iw, bit):
    """The packing step of QuantLinear.pack alone: unsigned integer weights iw [K, N] (< 2^bit) ->
    int32 qweight [packed_rows(K, bit), N].  Any K: no group structure is involved."""
    iw = np.asarray(iw).astype(np.uint64)
    k, n = iw.shape
    q = np.zeros((packed_rows(k, bit), n), dtype=np.uint64)
    for i, (row, shift, srow, sshift) in enumerate(_bit_slots(bit, k)):
        q[row] |= (iw[i] << np.uint64(shift)) & np.uint64(0xFFFFFFFF)
        if srow is not None:
            q[srow] |= iw[i] >> np.uint64(sshift)
    return q.astype(np.uint32).view(np.int32)


def unpack_bits(qweight, k, bit):
    """Inverse of pack_bits: unsigned integer weights [K, N]."""
    q = np.asarray(qweight).view(np.uint32).astype(np.uint64)
    mask = np.uint64(2**bit - 1)
    out = np.zeros((k, q.shape[1]), dtype=np.uint32)
    for i, (row, shift, srow, sshift) in enumerate(_bit_slots(bit, k)):
        v = q[row] >> np.uint64(shift)
        if srow is not None:
            v = v | (q[srow] << np.uint64(sshift))
        out[i] = (v & mask).astype(np.uint32)
    return out


def dequant_matmul(x, qweight, out_init, scales, zeros, group_size=0, dtype=np.float64, bit=4):
    """VecQuant{2,3,4}MatMulKernel contract -- cuda/cuda_kernel_4bit.cu:88-180 / cuda_kernel.cpp:10-57:
        out[m, n] = out_init[m, n] + sum_k (scales[n, k//gs] * q[k, n] - zeros[n, k//gs]) * x[m, k]
    computed in ``dtype`` (fp64 by default: the tolerance anchor for the fp32 kernels)."""
    x = np.asarray(x)
    k = x.shape[-1]
    xm = x.reshape(-1, k).astype(dtype)
    q = (unpack_int4(qweight, k) if bit == 4 else unpack_bits(qweight, k, bit)).astype(dtype)  # [K, N]
    n = q.shape[1]
    gs = k if group_size in (0, -1) else group_size
    g = (k + gs - 1) // gs
    s = np.asarray(scales, dtype=F32).reshape(n, g).astype(dtype)
    z = np.asarray(zeros, dtype=F32).reshape(n, g).astype(dtype)
    gi = np.arange(k) // gs
    w = s.T[gi] * q - z.T[gi]  # [K, N]
    y = np.asarray(out_init).reshape(-1, n).astype(dtype) + xm @ w
    return y.reshape(x.shape[:-1] + (n,))
