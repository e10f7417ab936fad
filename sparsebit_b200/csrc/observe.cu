// observe.cu -- Observer calibration reductions for sm_100a.
//
// Replaces the ATen op chains inside the reference observers (megvii-research/Sparsebit):
//   observers/minmax.py:14-25        torch.cat + min/max                  -> minmax_* kernels
//   observers/kl_histogram.py:47-50  data.cpu(); torch.histc(2048 bins)   -> hist_kernel
//   observers/mse.py:46-61           80 x (QDQ + (x-x_dq)^2.mean())       -> mse_sweep_kernel (1 pass)
//   observers/percentile.py:27-43    (x<0).sum, (x>=0).sum, kthvalue x2   -> select_* kernels
//   sparse/sparsers/l1norm.py:18-22  torch.sort(|w|)[k]                   -> select_* (key_mode 1)
//
// All of them are 4 B/elem streaming reads; statistics are combined with warp shuffles, a
// shared-memory stage and integer atomics (exact, order independent).  Floating-point sums that
// the reference produces (MSE) are accumulated fp32 per thread over a bounded tile, fp64 across
// tiles in a fixed order, so results are deterministic.
#include "common.cuh"

namespace sb200 {

constexpr int kThreads = 256;

// =========================================================================================
// Per-channel MinMax over x viewed as [outer, C, inner]
// =========================================================================================

// Reduce `len` contiguous floats starting at `p` into acc, cooperatively by `nthr` threads with
// rank `t`; uses 128-bit loads on the 16-byte aligned middle part.
__device__ __forceinline__ void span_minmax(const float* __restrict__ p, long long len, int t, int nthr,
                                            MinMaxAcc& acc) {
  long long head = ((16 - (reinterpret_cast<uintptr_t>(p) & 15u)) & 15u) >> 2;
  if (head > len) head = len;
  for (long long i = t; i < head; i += nthr) acc.add(__ldcs(p + i));
  const float4* q = reinterpret_cast<const float4*>(p + head);
  const long long nv = (len - head) >> 2;
  long long i = t;
  for (; i + 3LL * nthr < nv; i += 4LL * nthr) {
    const float4 a = ld_stream4(q + i), b = ld_stream4(q + i + nthr), c = ld_stream4(q + i + 2LL * nthr),
                 d = ld_stream4(q + i + 3LL * nthr);
    acc.add4(a); acc.add4(b); acc.add4(c); acc.add4(d);
  }
  for (; i < nv; i += nthr) acc.add4(ld_stream4(q + i));
  for (long long e = head + (nv << 2) + t; e < len; e += nthr) acc.add(__ldcs(p + e));
}

// Regime A: long rows -- one CTA per (row, tile) of up to kRowTile elements.
constexpr long long kRowTile = 8192;
__global__ void __launch_bounds__(kThreads) minmax_rows_cta_kernel(const float* __restrict__ x, long long rows,
                                                                   long long inner, int channels,
                                                                   uint32_t* __restrict__ state) {
  __shared__ float red[96];
  const long long tpr = (inner + kRowTile - 1) / kRowTile;
  const long long total = rows * tpr;
  for (long long tile = blockIdx.x; tile < total; tile += gridDim.x) {
    const long long row = tile / tpr, j = tile - row * tpr;
    const long long off = j * kRowTile;
    const long long len = (inner - off) < kRowTile ? (inner - off) : kRowTile;
    MinMaxAcc acc;
    acc.init();
    span_minmax(x + row * inner + off, len, threadIdx.x, blockDim.x, acc);
    block_reduce_minmax(acc, red);
    if (threadIdx.x == 0) acc.publish(state + 2 * (row % channels));
  }
}

// Regime B: mid-length rows (64 < inner < 4096) -- a warp takes 4 consecutive rows per iteration and
// keeps one 128-bit load per row in flight per lane (one row alone is only a few hundred bytes).
__global__ void __launch_bounds__(kThreads) minmax_rows_warp_kernel(const float* __restrict__ x, long long rows,
                                                                    long long inner, int channels,
                                                                    uint32_t* __restrict__ state) {
  const int lane = threadIdx.x & 31;
  const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
  const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const bool vec = ((inner & 3) == 0) && ((reinterpret_cast<uintptr_t>(x) & 15u) == 0);
  for (long long row0 = gw * 4; row0 < rows; row0 += warps * 4) {
    MinMaxAcc acc[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[j].init();
    if (vec && row0 + 3 < rows) {
      const long long nv = inner >> 2;
      const float4* base = reinterpret_cast<const float4*>(x + row0 * inner);
      for (long long i = lane; i < nv; i += 32) {
        const float4 v0 = ld_stream4(base + i), v1 = ld_stream4(base + nv + i), v2 = ld_stream4(base + 2 * nv + i),
                     v3 = ld_stream4(base + 3 * nv + i);
        acc[0].add4(v0); acc[1].add4(v1); acc[2].add4(v2); acc[3].add4(v3);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (row0 + j < rows) span_minmax(x + (row0 + j) * inner, inner, lane, 32, acc[j]);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      acc[j].warp_reduce();
      if (lane == 0 && row0 + j < rows) acc[j].publish(state + 2 * ((row0 + j) % channels));
    }
  }
}

// Regime B': tiny rows (inner <= 64, e.g. 7x7 feature maps) -- a warp stages 32 consecutive rows
// (one contiguous chunk, read with full coalescing) in shared memory, then lane l reduces row l.
__global__ void __launch_bounds__(kThreads) minmax_rows_tiny_kernel(const float* __restrict__ x, long long rows,
                                                                    int inner, int channels,
                                                                    uint32_t* __restrict__ state) {
  extern __shared__ __align__(16) float s_rows[];  // [warps per CTA][32 * inner]
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float* mine = s_rows + (size_t)wid * 32 * inner;
  const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
  const bool base_ok = (reinterpret_cast<uintptr_t>(x) & 15u) == 0;
  for (long long row0 = ((((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5)) * 32; row0 < rows; row0 += warps * 32) {
    const int nrows = (int)((rows - row0) < 32 ? (rows - row0) : 32);
    const int cnt = nrows * inner;
    const float* src = x + row0 * inner;
    if (base_ok && ((cnt & 3) == 0) && (((row0 * inner) & 3) == 0)) {
      const float4* s4 = reinterpret_cast<const float4*>(src);
      float4* d4 = reinterpret_cast<float4*>(mine);
      for (int i = lane; i < (cnt >> 2); i += 32) d4[i] = ld_stream4(s4 + i);
    } else {
      for (int i = lane; i < cnt; i += 32) mine[i] = __ldcs(src + i);
    }
    __syncwarp();
    if (lane < nrows) {
      MinMaxAcc acc;
      acc.init();
      const float* r = mine + lane * inner;
      const bool rot = (inner & 1) == 0;  // even row pitch: rotate the start column to spread banks
      for (int i = 0; i < inner; ++i) {
        const int col = rot ? (i + lane) % inner : i;
        acc.add(r[col]);
      }
      acc.publish(state + 2 * ((row0 + lane) % channels));
    }
    __syncwarp();
  }
}

// Regime C: channel-last ([R, C], inner == 1) -- a thread owns VEC adjacent channels and walks rows.
template <int VEC>
__global__ void __launch_bounds__(128) minmax_cols_kernel(const float* __restrict__ x, long long R, int channels,
                                                          long long rows_per_block, uint32_t* __restrict__ state) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;  // vector column
  const int nq = channels / VEC;
  if (q >= nq) return;
  long long r0 = (long long)blockIdx.y * rows_per_block;
  long long r1 = r0 + rows_per_block < R ? r0 + rows_per_block : R;
  MinMaxAcc acc[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) acc[j].init();
  if (VEC == 4) {
    const float4* base = reinterpret_cast<const float4*>(x) + q;
    long long r = r0;
    for (; r + 3 < r1; r += 4) {
      const float4 a = ld_stream4(base + r * nq), b = ld_stream4(base + (r + 1) * nq),
                   c = ld_stream4(base + (r + 2) * nq), d = ld_stream4(base + (r + 3) * nq);
      acc[0].add(a.x); acc[1 % VEC].add(a.y); acc[2 % VEC].add(a.z); acc[3 % VEC].add(a.w);
      acc[0].add(b.x); acc[1 % VEC].add(b.y); acc[2 % VEC].add(b.z); acc[3 % VEC].add(b.w);
      acc[0].add(c.x); acc[1 % VEC].add(c.y); acc[2 % VEC].add(c.z); acc[3 % VEC].add(c.w);
      acc[0].add(d.x); acc[1 % VEC].add(d.y); acc[2 % VEC].add(d.z); acc[3 % VEC].add(d.w);
    }
    for (; r < r1; ++r) {
      const float4 a = ld_stream4(base + r * nq);
      acc[0].add(a.x); acc[1 % VEC].add(a.y); acc[2 % VEC].add(a.z); acc[3 % VEC].add(a.w);
    }
  } else {
    for (long long r = r0; r < r1; ++r) acc[0].add(__ldcs(x + r * channels + q));
  }
#pragma unroll
  for (int j = 0; j < VEC; ++j) acc[j].publish(state + 2 * (q * VEC + j));
}

// =========================================================================================
// histc-compatible histogram
// =========================================================================================
// ATen CPU histc rule: pos = (int64)(((x - lo) * bins) / (hi - lo)) in fp32 (IEEE division),
// pos == bins -> bins - 1, x outside [lo, hi] (or NaN) dropped.
__global__ void __launch_bounds__(kThreads) hist_kernel(const float* __restrict__ x, long long n,
                                                        const float* __restrict__ range, int bins,
                                                        unsigned long long* __restrict__ counts) {
  extern __shared__ unsigned int s_cnt[];  // bins
  for (int i = threadIdx.x; i < bins; i += blockDim.x) s_cnt[i] = 0;
  __syncthreads();
  const float lo = __ldg(range), hi = __ldg(range + 1);
  const float fb = (float)bins;
  QP dv;
  dv.set(__fsub_rn(hi, lo), 0.f);
  const long long T = (long long)gridDim.x * blockDim.x;
  auto add = [&](float v) {
    if (!(v >= lo && v <= hi)) return;  // also drops NaN
    const float pos = div_exact(__fmul_rn(__fsub_rn(v, lo), fb), dv);
    int b = (int)pos;  // truncation toward zero like static_cast<int64_t>
    b = b > bins - 1 ? bins - 1 : (b < 0 ? 0 : b);
    atomicAdd(&s_cnt[b], 1u);
  };
  const bool vec = (reinterpret_cast<uintptr_t>(x) & 15u) == 0;
  const long long gt = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (vec) {
    const long long nv = n >> 2;
    const float4* x4 = reinterpret_cast<const float4*>(x);
    long long i = gt;
    for (; i + 3 * T < nv; i += 4 * T) {  // four independent 128-bit loads in flight per thread
      const float4 a = ld_stream4(x4 + i), b = ld_stream4(x4 + i + T), c = ld_stream4(x4 + i + 2 * T), d = ld_stream4(x4 + i + 3 * T);
      add(a.x); add(a.y); add(a.z); add(a.w);
      add(b.x); add(b.y); add(b.z); add(b.w);
      add(c.x); add(c.y); add(c.z); add(c.w);
      add(d.x); add(d.y); add(d.z); add(d.w);
    }
    for (; i < nv; i += T) {
      const float4 a = ld_stream4(x4 + i);
      add(a.x); add(a.y); add(a.z); add(a.w);
    }
    for (long long e = (nv << 2) + gt; e < n; e += T) add(__ldcs(x + e));
  } else {
    for (long long e = gt; e < n; e += T) add(__ldcs(x + e));
  }
  __syncthreads();
  for (int i = threadIdx.x; i < bins; i += blockDim.x) {
    const unsigned int c = s_cnt[i];
    if (c) atomicAdd(counts + i, (unsigned long long)c);
  }
}

// =========================================================================================
// MSE sweep: all candidates in one pass; x tile staged in shared memory by TMA (cp.async.bulk)
// =========================================================================================
constexpr int kMseTile = 8192;      // floats per tile (32 KB of shared memory)
constexpr int kMseCandChunk = 8;    // accumulators live per thread
constexpr int kMseMaxCand = 128;

// Per-candidate quantisation error of one value.  The quotient uses a reciprocal plus one
// Newton correction (q1 = q0 + (x - q0*s)*r), which is the correctly rounded x/s except in
// measure-zero corner cases -- sufficient for a loss that is compared at 1e-5 (Q: mse.py:51-55).
__device__ __forceinline__ float mse_err2(float x, float s, float r, float zp, float qmin, float qmax) {
  const float q0 = x * r;
  const float e = fmaf(-q0, s, x);
  const float q = fmaf(e, r, q0);
  float v = rintf(q) + zp;
  v = fminf(fmaxf(v, qmin), qmax);
  const float d = x - (v - zp) * s;
  return d * d;
}

// grid: persistent over tiles; tile t -> (row, j) with tpr tiles per row.
// partial[tile * ncand + i] = sum over the tile of err2 for candidate i (fp64).
__global__ void __launch_bounds__(kThreads) mse_sweep_kernel(const float* __restrict__ x, long long rows,
                                                             long long row_len, const float* __restrict__ cand_scale,
                                                             const float* __restrict__ cand_zp, int ncand,
                                                             float qmin, float qmax, double* __restrict__ partial) {
  __shared__ __align__(128) float s_x[kMseTile];
  __shared__ float s_s[kMseMaxCand], s_r[kMseMaxCand], s_z[kMseMaxCand];
  __shared__ double s_w[kThreads / 32][kMseCandChunk];
  __shared__ __align__(8) uint64_t s_bar;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const long long tpr = (row_len + kMseTile - 1) / kMseTile;
  const long long total = rows * tpr;
  if (tid == 0) {
    mbar_init(&s_bar, 1);
    mbar_fence_init();
  }
  __syncthreads();
  uint32_t phase = 0;
  long long prev_row = -1;
  for (long long tile = blockIdx.x; tile < total; tile += gridDim.x) {
    const long long row = tile / tpr, j = tile - row * tpr;
    const long long off = j * kMseTile;
    const int len = (int)((row_len - off) < kMseTile ? (row_len - off) : kMseTile);
    const float* src = x + row * row_len + off;
    const bool bulk = ((reinterpret_cast<uintptr_t>(src) & 15u) == 0) && ((len & 3) == 0);
    if (bulk) {
      if (tid == 0) {
        mbar_expect_tx(&s_bar, (uint32_t)len * 4u);
        tma_bulk_g2s(s_x, src, (uint32_t)len * 4u, &s_bar);
      }
    } else {
      for (int i = tid; i < len; i += blockDim.x) s_x[i] = __ldcs(src + i);
    }
    if (row != prev_row) {  // (re)load this row's candidate table
      for (int i = tid; i < ncand; i += blockDim.x) {
        const float s = __ldg(cand_scale + row * ncand + i);
        s_s[i] = s;
        s_r[i] = __frcp_rn(s);
        s_z[i] = rintf(__ldg(cand_zp + row * ncand + i));
      }
      prev_row = row;
    }
    if (bulk) {
      mbar_wait(&s_bar, phase);
      phase ^= 1;
    }
    __syncthreads();
    for (int c0 = 0; c0 < ncand; c0 += kMseCandChunk) {
      float acc[kMseCandChunk];
#pragma unroll
      for (int k = 0; k < kMseCandChunk; ++k) acc[k] = 0.f;
      for (int i = tid; i < len; i += kThreads) {
        const float v = s_x[i];
#pragma unroll
        for (int k = 0; k < kMseCandChunk; ++k) {
          const int ci = (c0 + k < ncand) ? (c0 + k) : (ncand - 1);
          acc[k] += mse_err2(v, s_s[ci], s_r[ci], s_z[ci], qmin, qmax);
        }
      }
#pragma unroll
      for (int k = 0; k < kMseCandChunk; ++k) {
        const double w = warp_sum((double)acc[k]);
        if (lane == 0) s_w[wid][k] = w;
      }
      __syncthreads();
      if (tid < kMseCandChunk && c0 + tid < ncand) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < kThreads / 32; ++w) t += s_w[w][tid];
        partial[tile * ncand + c0 + tid] = t;
      }
      __syncthreads();
    }
  }
}

// sse[row*ncand + i] += sum_j partial[(row*tpr + j)*ncand + i]   (fixed order): strided_finish_kernel below

// =========================================================================================
// Radix select (3 passes: 11 + 11 + 10 key bits) and sign counting
// =========================================================================================
// Elements per (row, segment) tile, chosen per call (sel_seg): 65536 when that still gives every SM several CTAs, halved
// down to 16384 otherwise.  (A fixed 65536 made 296 CTAs out of a 19 M-element tensor -- two per SM, 16 KB of loads in
// flight per SM, every pass at 2 TB/s; a fixed 16384 costs large tensors 10 % in per-tile histogram flushes.)
constexpr long long kSelSegMax = 65536, kSelSegMin = 16384;
constexpr int kSelMaxTargets = 2;
constexpr int kSelCopies = 4;  // pass-0 sub-histograms per CTA (spreads hot exponent buckets)

__device__ __forceinline__ uint32_t sel_key(float v, int key_mode) {
  if (v != v) return 0xFFFFFFFFu;  // NaN sorts last (torch.kthvalue / torch.sort)
  return enc_f32(key_mode ? fabsf(v) : v);
}
__device__ __forceinline__ int pass_shift(int pass) { return pass == 0 ? 21 : (pass == 1 ? 10 : 0); }
__device__ __forceinline__ int pass_bits(int pass) { return pass == 2 ? 10 : 11; }

// sel layout per target: [0] prefix (bits decided so far, right aligned), [1] remaining rank,
// [2] final key, [3] reserved.
template <int PASS>
__global__ void __launch_bounds__(kThreads) select_hist_kernel(const float* __restrict__ x, long long rows,
                                                               long long row_len, long long seg, int ntpr,
                                                               const unsigned long long* __restrict__ sel,
                                                               unsigned long long* __restrict__ hist, int key_mode,
                                                               unsigned long long* __restrict__ sign_counts) {
  extern __shared__ unsigned int s_hist[];  // PASS 0: kSelCopies * 2048 ; else ntpr * 2048
  const int nslots = (PASS == 0) ? kSelCopies : ntpr;
  const long long spr = (row_len + seg - 1) / seg;
  const long long total = rows * spr;
  const int lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < nslots * SB200_SELECT_BINS; i += blockDim.x) s_hist[i] = 0;
  __syncthreads();
  for (long long tile = blockIdx.x; tile < total; tile += gridDim.x) {
    const long long row = tile / spr, j = tile - row * spr;
    const long long off = j * seg;
    const long long len = (row_len - off) < seg ? (row_len - off) : seg;
    const float* p = x + row * row_len + off;
    uint32_t pre[kSelMaxTargets] = {0, 0};
    if (PASS > 0) {
      for (int t = 0; t < ntpr; ++t) pre[t] = (uint32_t)sel[(row * ntpr + t) * SB200_SELECT_STATE_WORDS + 0];
    }
    unsigned int neg = 0, pos = 0;
    auto add = [&](float v) {
      const uint32_t k = sel_key(v, key_mode);
      if (PASS == 0) {
        atomicAdd(&s_hist[(lane & (kSelCopies - 1)) * SB200_SELECT_BINS + (k >> 21)], 1u);
        neg += (v < 0.f);
        pos += (v >= 0.f);
      } else {
        const uint32_t hi = k >> (PASS == 1 ? 21 : 10);
        const uint32_t dg = (PASS == 1) ? ((k >> 10) & 0x7FFu) : (k & 0x3FFu);
#pragma unroll
        for (int t = 0; t < kSelMaxTargets; ++t)
          if (t < ntpr && hi == pre[t]) atomicAdd(&s_hist[t * SB200_SELECT_BINS + dg], 1u);
      }
    };
    long long head = ((16 - (reinterpret_cast<uintptr_t>(p) & 15u)) & 15u) >> 2;
    if (head > len) head = len;
    for (long long i = threadIdx.x; i < head; i += blockDim.x) add(__ldcs(p + i));
    const float4* q = reinterpret_cast<const float4*>(p + head);
    const long long nv = (len - head) >> 2;
    long long i = threadIdx.x;
    for (; i + 3LL * blockDim.x < nv; i += 4LL * blockDim.x) {  // four independent 128-bit loads in flight per thread
      const float4 a = ld_stream4(q + i), b = ld_stream4(q + i + blockDim.x), c = ld_stream4(q + i + 2LL * blockDim.x),
                   d = ld_stream4(q + i + 3LL * blockDim.x);
      add(a.x); add(a.y); add(a.z); add(a.w);
      add(b.x); add(b.y); add(b.z); add(b.w);
      add(c.x); add(c.y); add(c.z); add(c.w);
      add(d.x); add(d.y); add(d.z); add(d.w);
    }
    for (; i < nv; i += blockDim.x) {
      const float4 a = ld_stream4(q + i);
      add(a.x); add(a.y); add(a.z); add(a.w);
    }
    for (long long e = head + (nv << 2) + threadIdx.x; e < len; e += blockDim.x) add(__ldcs(p + e));
    __syncthreads();
    // flush this tile's histogram(s) to global and clear
    if (PASS == 0) {
      unsigned long long* g = hist + (row * ntpr) * SB200_SELECT_BINS;  // target 0 of the row
      for (int b = threadIdx.x; b < SB200_SELECT_BINS; b += blockDim.x) {
        unsigned int c = 0;
#pragma unroll
        for (int k = 0; k < kSelCopies; ++k) {
          c += s_hist[k * SB200_SELECT_BINS + b];
          s_hist[k * SB200_SELECT_BINS + b] = 0;
        }
        if (c) atomicAdd(g + b, (unsigned long long)c);
      }
      if (sign_counts) {
        neg = __reduce_add_sync(0xffffffffu, neg);
        pos = __reduce_add_sync(0xffffffffu, pos);
        if (lane == 0) {
          if (neg) atomicAdd(sign_counts + row * 2, (unsigned long long)neg);
          if (pos) atomicAdd(sign_counts + row * 2 + 1, (unsigned long long)pos);
        }
      }
    } else {
      for (int t = 0; t < ntpr; ++t) {
        unsigned long long* g = hist + (row * ntpr + t) * SB200_SELECT_BINS;
        for (int b = threadIdx.x; b < SB200_SELECT_BINS; b += blockDim.x) {
          const unsigned int c = s_hist[t * SB200_SELECT_BINS + b];
          if (c) {
            atomicAdd(g + b, (unsigned long long)c);
            s_hist[t * SB200_SELECT_BINS + b] = 0;
          }
        }
      }
    }
    __syncthreads();
  }
}

// One CTA per row: for each target of the row find the bucket holding its rank.
__global__ void __launch_bounds__(kThreads) select_scan_kernel(unsigned long long* __restrict__ sel,
                                                               unsigned long long* __restrict__ hist, int ntpr,
                                                               int pass) {
  __shared__ unsigned long long s_part[kThreads];
  __shared__ unsigned long long s_found[2];
  const long long row = blockIdx.x;
  const int bits = pass_bits(pass);
  const int nb = 1 << bits;
  const int per = SB200_SELECT_BINS / kThreads;  // 8 bins per thread
  for (int t = 0; t < ntpr; ++t) {
    const unsigned long long* h = hist + (row * ntpr + (pass == 0 ? 0 : t)) * SB200_SELECT_BINS;
    unsigned long long* st = sel + (row * ntpr + t) * SB200_SELECT_STATE_WORDS;
    const unsigned long long rank = st[1];
    unsigned long long loc[per];
    unsigned long long sum = 0;
#pragma unroll
    for (int k = 0; k < per; ++k) {
      const int b = threadIdx.x * per + k;
      loc[k] = b < nb ? h[b] : 0ull;
      sum += loc[k];
    }
    s_part[threadIdx.x] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {  // exclusive scan of 256 partials (tiny, once per pass)
      unsigned long long run = 0;
      for (int i = 0; i < kThreads; ++i) {
        const unsigned long long v = s_part[i];
        s_part[i] = run;
        run += v;
      }
      s_found[0] = 0xFFFFFFFFFFFFFFFFull;
    }
    __syncthreads();
    unsigned long long base = s_part[threadIdx.x];
#pragma unroll
    for (int k = 0; k < per; ++k) {
      if (loc[k] && rank >= base && rank < base + loc[k]) {
        s_found[0] = (unsigned long long)(threadIdx.x * per + k);
        s_found[1] = base;
      }
      base += loc[k];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned long long b = s_found[0];
      unsigned long long below = s_found[1];
      if (b == 0xFFFFFFFFFFFFFFFFull) {  // rank beyond the population: no bin holds it, bin 0 is taken and the value
        // read back is meaningless.  Callers keep ranks below the row length (ops.kth_value rejects k >= n,
        // percentile_ranks_kernel clamps to the row total).
        b = 0;
        below = 0;
      }
      st[0] = (st[0] << bits) | b;
      st[1] = rank - below;
      if (pass == 2) st[2] = st[0];
    }
    __syncthreads();
  }
  // clear this row's histograms for the next pass
  for (int i = threadIdx.x; i < ntpr * SB200_SELECT_BINS; i += blockDim.x) hist[row * ntpr * SB200_SELECT_BINS + i] = 0ull;
}

__global__ void select_init_kernel(unsigned long long* sel, unsigned long long* hist, long long ntargets,
                                   const long long* ranks) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < ntargets * SB200_SELECT_BINS) hist[i] = 0ull;
  if (i < ntargets) {
    sel[i * SB200_SELECT_STATE_WORDS + 0] = 0ull;
    sel[i * SB200_SELECT_STATE_WORDS + 1] = ranks ? (unsigned long long)ranks[i] : 0ull;
    sel[i * SB200_SELECT_STATE_WORDS + 2] = 0ull;
    sel[i * SB200_SELECT_STATE_WORDS + 3] = 0ull;
  }
}

__global__ void select_read_kernel(const unsigned long long* __restrict__ sel, long long ntargets, int key_mode,
                                   float* __restrict__ values) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < ntargets) {
    const uint32_t k = (uint32_t)sel[i * SB200_SELECT_STATE_WORDS + 2];
    values[i] = (k == 0xFFFFFFFFu) ? __int_as_float(0x7fc00000) : dec_f32(k);
  }
}

// counts[row*2] = #(x<0), counts[row*2+1] = #(x>=0);  total[row] = row length incl. NaN.
// ranks written straight into the select state (min side = target 0, max side = target 1).
__global__ void percentile_ranks_kernel(const unsigned long long* __restrict__ counts,
                                        const long long* __restrict__ total, long long rows, double alpha,
                                        unsigned long long* __restrict__ sel) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const double neg = (double)counts[2 * r], pos = (double)counts[2 * r + 1];
  // Python round(): half-to-even on the double product == rint()
  long long kmin = (long long)rint(neg * alpha);
  if (kmin < 1) kmin = 1;
  long long kpos = (long long)rint(pos * alpha);
  if (kpos < 0) kpos = 0;
  long long kmax = total[r] - kpos;  // 1-based k for kthvalue
  if (kmax < 1) kmax = 1;
  if (kmin > total[r]) kmin = total[r];
  sel[(r * 2 + 0) * SB200_SELECT_STATE_WORDS + 1] = (unsigned long long)(kmin - 1);
  sel[(r * 2 + 1) * SB200_SELECT_STATE_WORDS + 1] = (unsigned long long)(kmax - 1);
}

__global__ void count_sign_kernel(const float* __restrict__ x, long long rows, long long row_len, long long seg,
                                  unsigned long long* __restrict__ counts) {
  const long long spr = (row_len + seg - 1) / seg;
  const long long total = rows * spr;
  const int lane = threadIdx.x & 31;
  for (long long tile = blockIdx.x; tile < total; tile += gridDim.x) {
    const long long row = tile / spr, j = tile - row * spr;
    const long long off = j * seg;
    const long long len = (row_len - off) < seg ? (row_len - off) : seg;
    const float* p = x + row * row_len + off;
    unsigned int neg = 0, pos = 0;
    for (long long i = threadIdx.x; i < len; i += blockDim.x) {
      const float v = __ldcs(p + i);
      neg += (v < 0.f);
      pos += (v >= 0.f);
    }
    neg = __reduce_add_sync(0xffffffffu, neg);
    pos = __reduce_add_sync(0xffffffffu, pos);
    if (lane == 0) {
      if (neg) atomicAdd(counts + row * 2, (unsigned long long)neg);
      if (pos) atomicAdd(counts + row * 2 + 1, (unsigned long long)pos);
    }
  }
}

static inline int persistent_grid(long long tiles, int ctas_per_sm) {
  long long cap = (long long)sm_count() * ctas_per_sm;
  if (tiles < 1) tiles = 1;
  return (int)(tiles < cap ? tiles : cap);
}
static inline long long sel_seg(long long rows, long long row_len) {
  long long seg = kSelSegMax;
  const long long want = (long long)sm_count() * 6;
  while (seg > kSelSegMin && rows * ((row_len + seg - 1) / seg) < want) seg >>= 1;
  return seg;
}


// =========================================================================================
// Row moments (LSQ / LSQ+ step-size initialisation, ACIQ-laplace): per row of x [rows, row_len]
//   S[0] += sum x, S[1] += sum x^2, S[2] += sum |x|, S[3] += sum |x - c|, S[4] += sum (x - c)^2
// (c = centre[row], 0 when centre is NULL).  fp32 loads, fp64 accumulation; one CTA per (row, tile)
// writes its partial, a finish kernel adds the tiles of a row in index order -> deterministic.
// =========================================================================================
constexpr long long kMomTile = 16384;
constexpr int kMomVals = 5;

__global__ void __launch_bounds__(kThreads) moments_tile_kernel(const float* __restrict__ x, long long rows,
                                                                long long row_len, const double* __restrict__ centre,
                                                                double* __restrict__ partial) {
  __shared__ double red[kMomVals][kThreads / 32];
  const long long tpr = (row_len + kMomTile - 1) / kMomTile;
  const long long total = rows * tpr;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (long long tile = blockIdx.x; tile < total; tile += gridDim.x) {
    const long long row = tile / tpr, j = tile - row * tpr;
    const long long off = j * kMomTile;
    const long long len = (row_len - off) < kMomTile ? (row_len - off) : kMomTile;
    const float* p = x + row * row_len + off;
    const float c = centre ? (float)centre[row] : 0.f;
    const double cd = centre ? centre[row] : 0.0;
    // per thread: fp32 partial sums over at most 64 elements would already lose bits for sum x^2; keep fp64
    double a0 = 0, a1 = 0, a2 = 0, a3 = 0, a4 = 0;
    (void)c;
    for (long long i = threadIdx.x; i < len; i += kThreads) {
      const double v = (double)__ldcs(p + i);
      const double d = v - cd;
      a0 += v;
      a1 += v * v;
      a2 += fabs(v);
      a3 += fabs(d);
      a4 += d * d;
    }
    double acc[kMomVals] = {a0, a1, a2, a3, a4};
#pragma unroll
    for (int k = 0; k < kMomVals; ++k) {
      const double w = warp_sum(acc[k]);
      if (lane == 0) red[k][wid] = w;
    }
    __syncthreads();
    if (threadIdx.x < kMomVals) {
      double t = 0;
#pragma unroll
      for (int w = 0; w < kThreads / 32; ++w) t += red[threadIdx.x][w];
      partial[tile * kMomVals + threadIdx.x] = t;
    }
    __syncthreads();
  }
}

__global__ void strided_finish_kernel(const double* __restrict__ partial, long long tpr, int nval, double* __restrict__ out) {
  extern __shared__ double s_fin[];  // [S][nval]
  const int S = blockDim.x / nval;
  const int s = threadIdx.x / nval, k = threadIdx.x - s * nval;
  const long long row = blockIdx.x;
  if (s < S) {
    const double* base = partial + row * tpr * nval + k;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    long long j = s;
    for (; j + 3LL * S < tpr; j += 4LL * S) {
      const double v0 = base[j * nval], v1 = base[(j + S) * nval], v2 = base[(j + 2LL * S) * nval], v3 = base[(j + 3LL * S) * nval];
      a0 += v0; a1 += v1; a2 += v2; a3 += v3;
    }
    for (; j < tpr; j += S) a0 += base[j * nval];
    s_fin[s * nval + k] = (a0 + a1) + (a2 + a3);
  }
  __syncthreads();
  if (threadIdx.x < nval) {
    double t = 0.0;
    for (int q = 0; q < S; ++q) t += s_fin[q * nval + threadIdx.x];
    out[row * nval + threadIdx.x] += t;
  }
}

}  // namespace sb200

using namespace sb200;

extern "C" {

int sb200_observe_minmax_perchannel(const float* x, int64_t outer, int64_t channels, int64_t inner,
                                    uint32_t* state, void* stream) {
  SB_REQUIRE(x && state, "sb200_observe_minmax_perchannel: null pointer argument");
  SB_REQUIRE(outer > 0 && channels > 0 && inner > 0, "sb200_observe_minmax_perchannel: empty tensor");
  SB_REQUIRE(channels < (1LL << 31), "sb200_observe_minmax_perchannel: too many channels");
  cudaStream_t st = (cudaStream_t)stream;
  const long long rows = outer * channels;
  if (inner == 1) {
    const bool vec = (channels % 4 == 0) && aligned16(x);
    const long long nq = vec ? channels / 4 : channels;
    // (64-thread CTAs, which leave no idle lanes for 192 vector columns, measured slower here: 155 vs 139 us on
    // [1024, 197, 768] -- unlike the backward kernel, which gained from them)
    const int bt = 128;
    const unsigned gx = (unsigned)((nq + bt - 1) / bt);
    long long want_y = ((long long)sm_count() * 8 * (128 / bt) + gx - 1) / gx;
    if (want_y > outer) want_y = outer;
    if (want_y > 65535) want_y = 65535;
    if (want_y < 1) want_y = 1;
    const long long rpb = (outer + want_y - 1) / want_y;
    const unsigned gy = (unsigned)((outer + rpb - 1) / rpb);
    if (vec)
      minmax_cols_kernel<4><<<dim3(gx, gy), bt, 0, st>>>(x, outer, (int)channels, rpb, state);
    else
      minmax_cols_kernel<1><<<dim3(gx, gy), bt, 0, st>>>(x, outer, (int)channels, rpb, state);
  } else if (inner >= 4096) {
    const long long tiles = rows * ((inner + kRowTile - 1) / kRowTile);
    minmax_rows_cta_kernel<<<persistent_grid(tiles, 8), kThreads, 0, st>>>(x, rows, inner, (int)channels, state);
  } else if (inner <= 64) {
    const long long ctas = (rows + 32 * (kThreads / 32) - 1) / (32 * (kThreads / 32));
    const size_t smem = (size_t)(kThreads / 32) * 32 * inner * sizeof(float);  // <= 64 KB
    static std::atomic<int> attr_done[64];  // per device
    SB_CUDA(ensure_dyn_smem(minmax_rows_tiny_kernel, 64 * 1024, attr_done));
    minmax_rows_tiny_kernel<<<persistent_grid(ctas, 3), kThreads, smem, st>>>(x, rows, (int)inner, (int)channels, state);
  } else {
    const long long ctas = (rows + 4 * (kThreads / 32) - 1) / (4 * (kThreads / 32));
    minmax_rows_warp_kernel<<<persistent_grid(ctas, 8), kThreads, 0, st>>>(x, rows, inner, (int)channels, state);
  }
  SB_LAUNCHED();
  return SB200_OK;
}

int sb200_observe_hist(const float* x, int64_t n, const float* range, int bins, int64_t* counts, void* stream) {
  SB_REQUIRE(x && range && counts, "sb200_observe_hist: null pointer argument");
  SB_REQUIRE(n > 0, "sb200_observe_hist: empty tensor");
  SB_REQUIRE(bins > 0 && bins <= 8192, "sb200_observe_hist: bins must be in [1, 8192] (got %d)", bins);
  const size_t smem = (size_t)bins * 4;
  const long long blocks = (n / 4 + kThreads * 4 - 1) / (kThreads * 4);
  hist_kernel<<<persistent_grid(blocks, 8), kThreads, smem, (cudaStream_t)stream>>>(
      x, n, range, bins, reinterpret_cast<unsigned long long*>(counts));
  SB_LAUNCHED();
  return SB200_OK;
}

size_t sb200_mse_workspace_bytes(int64_t rows, int64_t row_len, int ncand) {
  if (rows <= 0 || row_len <= 0 || ncand <= 0) return 0;
  const long long tpr = (row_len + kMseTile - 1) / kMseTile;
  return (size_t)(rows * tpr) * (size_t)ncand * sizeof(double);
}

int sb200_observe_mse_sweep(const float* x, int64_t rows, int64_t row_len, const float* cand_scale,
                            const float* cand_zp, int ncand, int qmin, int qmax, double* sse, void* workspace,
                            size_t workspace_bytes, void* stream) {
  SB_REQUIRE(x && cand_scale && cand_zp && sse, "sb200_observe_mse_sweep: null pointer argument");
  SB_REQUIRE(rows > 0 && row_len > 0, "sb200_observe_mse_sweep: empty tensor");
  SB_REQUIRE(ncand > 0 && ncand <= kMseMaxCand, "sb200_observe_mse_sweep: ncand must be in [1, %d]", kMseMaxCand);
  const size_t need = sb200_mse_workspace_bytes(rows, row_len, ncand);
  if (!workspace || workspace_bytes < need) {
    set_error("sb200_observe_mse_sweep: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    return SB200_E_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const long long tpr = (row_len + kMseTile - 1) / kMseTile;
  const long long tiles = rows * tpr;
  mse_sweep_kernel<<<persistent_grid(tiles, 4), kThreads, 0, st>>>(x, rows, row_len, cand_scale, cand_zp, ncand,
                                                                    (float)qmin, (float)qmax, (double*)workspace);
  SB_LAUNCHED();
  const long long outn = rows * ncand;
  {
    const int ft = strided_finish_threads(tpr, ncand);
    strided_finish_kernel<<<(unsigned)rows, ft, (size_t)(ft / ncand) * ncand * sizeof(double), st>>>((const double*)workspace, tpr, ncand, sse);
  }
  SB_LAUNCHED();
  return SB200_OK;
}

int sb200_select_init(uint64_t* sel, int64_t* hist, int64_t ntargets_total, const int64_t* ranks, void* stream) {
  SB_REQUIRE(sel && hist && ntargets_total > 0, "sb200_select_init: bad arguments");
  const long long n = ntargets_total * SB200_SELECT_BINS;
  select_init_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      (unsigned long long*)sel, (unsigned long long*)hist, ntargets_total, (const long long*)ranks);
  SB_LAUNCHED();
  return SB200_OK;
}

int sb200_select_hist(const float* x, int64_t rows, int64_t row_len, int ntargets_per_row, const uint64_t* sel,
                      int64_t* hist, int pass, int key_mode, void* stream) {
  return sb200_select_hist_counts(x, rows, row_len, ntargets_per_row, sel, hist, pass, key_mode, nullptr, stream);
}

int sb200_select_hist_counts(const float* x, int64_t rows, int64_t row_len, int ntargets_per_row,
                             const uint64_t* sel, int64_t* hist, int pass, int key_mode, int64_t* sign_counts,
                             void* stream) {
  SB_REQUIRE(x && sel && hist, "sb200_select_hist: null pointer argument");
  SB_REQUIRE(rows > 0 && row_len > 0, "sb200_select_hist: empty tensor");
  SB_REQUIRE(ntargets_per_row >= 1 && ntargets_per_row <= kSelMaxTargets,
             "sb200_select_hist: ntargets_per_row must be 1 or 2 (got %d)", ntargets_per_row);
  SB_REQUIRE(pass >= 0 && pass <= 2, "sb200_select_hist: pass must be 0, 1 or 2");
  cudaStream_t st = (cudaStream_t)stream;
  const long long seg = sel_seg(rows, row_len);
  const long long tiles = rows * ((row_len + seg - 1) / seg);
  const int grid = persistent_grid(tiles, 6);  // pass 0 holds 32 KB of sub-histograms per CTA: 6 fit next to each other
  auto* sl = reinterpret_cast<const unsigned long long*>(sel);
  auto* hs = reinterpret_cast<unsigned long long*>(hist);
  auto* sc = reinterpret_cast<unsigned long long*>(sign_counts);
  if (pass == 0) {
    const size_t smem = (size_t)kSelCopies * SB200_SELECT_BINS * 4;
    select_hist_kernel<0><<<grid, kThreads, smem, st>>>(x, rows, row_len, seg, ntargets_per_row, sl, hs, key_mode, sc);
  } else {
    const size_t smem = (size_t)ntargets_per_row * SB200_SELECT_BINS * 4;
    if (pass == 1)
      select_hist_kernel<1><<<grid, kThreads, smem, st>>>(x, rows, row_len, seg, ntargets_per_row, sl, hs, key_mode, nullptr);
    else
      select_hist_kernel<2><<<grid, kThreads, smem, st>>>(x, rows, row_len, seg, ntargets_per_row, sl, hs, key_mode, nullptr);
  }
  SB_LAUNCHED();
  return SB200_OK;
}

int sb200_select_scan(uint64_t* sel, int64_t* hist, int64_t rows, int ntargets_per_row, int pass, void* stream) {
  SB_REQUIRE(sel && hist && rows > 0, "sb200_select_scan: bad arguments");
  SB_REQUIRE(ntargets_per_row >= 1 && ntargets_per_row <= kSelMaxTargets, "sb200_select_scan: bad ntargets_per_row");
  SB_REQUIRE(pass >= 0 && pass <= 2, "sb200_select_scan: pass must be 0, 1 or 2");
  select_scan_kernel<<<(unsigned)rows, kThreads, 0, (cudaStream_t)stream>>>(
      (unsigned long long*)sel, (unsigned long long*)hist, ntargets_per_row, pass);
  SB_LAUNCHED();
  return SB200_OK;
}

int sb200_select_read(const uint64_t* sel, int64_t ntargets_total, int key_mode, float* values, void* stream) {
  SB_REQUIRE(sel && values && ntargets_total > 0, "sb200_select_read: bad arguments");
  select_read_kernel<<<(unsigned)((ntargets_total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      (const unsigned long long*)sel, ntargets_total, key_mode, values);
  SB_LAUNCHED();
  return SB200_OK;
}

int sb200_count_sign(const float* x, int64_t rows, int64_t row_len, int64_t* counts, void* stream) {
  SB_REQUIRE(x && counts, "sb200_count_sign: null pointer argument");
  SB_REQUIRE(rows > 0 && row_len > 0, "sb200_count_sign: empty tensor");
  const long long seg = sel_seg(rows, row_len);
  const long long tiles = rows * ((row_len + seg - 1) / seg);
  count_sign_kernel<<<persistent_grid(tiles, 8), kThreads, 0, (cudaStream_t)stream>>>(
      x, rows, row_len, seg, (unsigned long long*)counts);
  SB_LAUNCHED();
  return SB200_OK;
}

int sb200_percentile_ranks(const int64_t* counts, const int64_t* total, int64_t rows, double alpha, uint64_t* sel,
                           void* stream) {
  SB_REQUIRE(counts && total && sel && rows > 0, "sb200_percentile_ranks: bad arguments");
  percentile_ranks_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      (const unsigned long long*)counts, (const long long*)total, rows, alpha, (unsigned long long*)sel);
  SB_LAUNCHED();
  return SB200_OK;
}

size_t sb200_moments_workspace_bytes(int64_t rows, int64_t row_len) {
  if (rows <= 0 || row_len <= 0) return 0;
  return (size_t)(rows * ((row_len + kMomTile - 1) / kMomTile)) * kMomVals * sizeof(double);
}

int sb200_observe_moments(const float* x, int64_t rows, int64_t row_len, const double* centre, double* out,
                          void* workspace, size_t workspace_bytes, void* stream) {
  SB_REQUIRE(x && out && workspace, "sb200_observe_moments: null pointer argument");
  SB_REQUIRE(rows > 0 && row_len > 0, "sb200_observe_moments: empty tensor");
  SB_REQUIRE(workspace_bytes >= sb200_moments_workspace_bytes(rows, row_len), "sb200_observe_moments: workspace too small");
  const long long tpr = (row_len + kMomTile - 1) / kMomTile;
  const long long tiles = rows * tpr;
  double* partial = reinterpret_cast<double*>(workspace);
  moments_tile_kernel<<<persistent_grid(tiles, 8), kThreads, 0, (cudaStream_t)stream>>>(x, rows, row_len, centre, partial);
  SB_LAUNCHED();
  const long long n = rows * kMomVals;
  {
    const int ft = strided_finish_threads(tpr, kMomVals);
    strided_finish_kernel<<<(unsigned)rows, ft, (size_t)(ft / kMomVals) * kMomVals * sizeof(double), (cudaStream_t)stream>>>(partial, tpr, kMomVals, out);
  }
  SB_LAUNCHED();
  return SB200_OK;
}

}  // extern "C"
