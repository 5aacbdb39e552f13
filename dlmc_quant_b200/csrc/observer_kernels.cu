// observer_kernels.cu - PTQ observers (dlmc/quantization/scalar/ops.py) as single-pass kernels.
//
//   obs_stats            one read of x -> {min, max, max|x|, sum|x|} per tensor / per channel
//   *_finalize           O(channels) kernels turning statistics into (scale, offset); multi-GPU
//                        callers all-reduce the statistics between the two calls
//   sweep_tensor         ops.py:36-68   80-candidate clip-ratio MSE search, per tensor: every thread
//                        keeps its elements in registers and evaluates all 80 candidates on them,
//                        so x is read from HBM exactly once (the reference reads it 80 x 9 times)
//   sweep_channel        ops.py:169-196 per-channel search: one warp per row, the row staged once in
//                        shared memory by a bulk async copy (TMA, cp.async.bulk + mbarrier) and swept
//                        80 times on chip, including the reference's sequential accept rule
//   l2norm_step          ops.py:71-83,198-215 one fixed-point iteration (two dot products per row)
//
// Rooflines: stats / l2norm are HBM-bound (4 B/elem fp32).  The sweeps are fp32-issue-bound once
// staged (80 x ~20 instructions per element against 4 B of traffic).
#include "fq_math.cuh"

namespace dlmcq {

constexpr int kNC = DLMCQ_SWEEP_CANDIDATES;

// ---------------------------------------------------------------------------------------
// statistics
// ---------------------------------------------------------------------------------------
struct Stat4 {
  float mn, mx, am, sm;
};
__device__ __forceinline__ void stat_init(Stat4& s) {
  s.mn = INFINITY; s.mx = -INFINITY; s.am = 0.f; s.sm = 0.f;
}
template <bool ABS = false>
__device__ __forceinline__ void stat_add(Stat4& s, float v) {
  const float a = fabsf(v);
  if (ABS) v = a;
  s.mn = fminf(s.mn, v); s.mx = fmaxf(s.mx, v); s.am = fmaxf(s.am, a); s.sm += a;   // NaN reaches sm
}
__device__ __forceinline__ void stat_merge(Stat4& s, const Stat4& o) {
  s.mn = fminf(s.mn, o.mn); s.mx = fmaxf(s.mx, o.mx); s.am = fmaxf(s.am, o.am); s.sm += o.sm;
}
__device__ __forceinline__ Stat4 stat_warp(Stat4 s) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    Stat4 t;
    t.mn = __shfl_xor_sync(0xffffffffu, s.mn, o);
    t.mx = __shfl_xor_sync(0xffffffffu, s.mx, o);
    t.am = __shfl_xor_sync(0xffffffffu, s.am, o);
    t.sm = __shfl_xor_sync(0xffffffffu, s.sm, o);
    stat_merge(s, t);
  }
  return s;
}
// torch.min / torch.max propagate NaN; fminf/fmaxf do not.  Any NaN input makes sum|x| NaN,
// which is then used to poison the other three statistics.
__device__ __forceinline__ void stat_store(float* out, const Stat4& s) {
  const bool nan = s.sm != s.sm;
  out[0] = nan ? s.sm : s.mn;
  out[1] = nan ? s.sm : s.mx;
  out[2] = nan ? s.sm : s.am;
  out[3] = s.sm;
}

template <typename T, bool ABS>
__global__ void __launch_bounds__(kThreads, 4)
stats_flat_kernel(const T* __restrict__ x, int64_t n, float* __restrict__ stats, void* ws) {
  using V = Vec<T>;
  using raw = typename V::raw;
  __shared__ Stat4 sh[32];
  Stat4 s;
  stat_init(s);
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if ((reinterpret_cast<uintptr_t>(x) & 15u) == 0) {
    const int64_t nvec = n / V::N;
    const raw* xv = reinterpret_cast<const raw*>(x);
    constexpr int U = 4;
    for (; i + (U - 1) * stride < nvec; i += U * stride) {
      raw r[U];
#pragma unroll
      for (int k = 0; k < U; ++k) r[k] = ld_stream(xv + i + k * stride);
#pragma unroll
      for (int k = 0; k < U; ++k) {
        float f[V::N];
        V::unpack(r[k], f);
#pragma unroll
        for (int e = 0; e < V::N; ++e) stat_add<ABS>(s, f[e]);
      }
    }
    for (; i < nvec; i += stride) {
      float f[V::N];
      V::unpack(ld_stream(xv + i), f);
#pragma unroll
      for (int e = 0; e < V::N; ++e) stat_add<ABS>(s, f[e]);
    }
    if (blockIdx.x == 0) {
      const int64_t t = nvec * V::N + threadIdx.x;
      if (t < n) stat_add<ABS>(s, to_f32<T>(x[t]));
    }
  } else {
    for (; i < n; i += stride) stat_add<ABS>(s, to_f32<T>(x[i]));
  }
  s = stat_warp(s);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  if (lane == 0) sh[warp] = s;
  __syncthreads();
  Stat4* part = reinterpret_cast<Stat4*>(ws_partials(ws));
  if (threadIdx.x == 0) {
    for (int w = 1; w < nwarp; ++w) stat_merge(s, sh[w]);
    part[blockIdx.x] = s;
  }
  if (take_last_ticket(ws_counter(ws), gridDim.x)) {
    Stat4 t;
    stat_init(t);
    for (int b = threadIdx.x; b < static_cast<int>(gridDim.x); b += blockDim.x) stat_merge(t, part[b]);
    t = stat_warp(t);
    __syncthreads();
    if (lane == 0) sh[warp] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int w = 1; w < nwarp; ++w) stat_merge(t, sh[w]);
      stat_store(stats, t);
      *ws_counter(ws) = 0u;
    }
  }
}

template <typename T, bool ABS>
__global__ void __launch_bounds__(kRowWarps * 32)
stats_rows_kernel(const T* __restrict__ x, RowGeom gm, float* __restrict__ stats, Stat4* __restrict__ part, int direct) {
  using V = Vec<T>;
  using raw = typename V::raw;
  const int lane = threadIdx.x & 31;
  const int64_t item = static_cast<int64_t>(blockIdx.x) * kRowWarps + (threadIdx.x >> 5);
  if (item >= gm.rows * gm.segs) return;
  const int64_t row = item / gm.segs, seg = item - row * gm.segs;
  const int64_t beg = seg * gm.seg;
  const int64_t len = (gm.inner - beg) < gm.seg ? (gm.inner - beg) : gm.seg;
  const T* xr = x + row * gm.inner + beg;
  Stat4 s;
  stat_init(s);
  int64_t done = 0;
  if ((reinterpret_cast<uintptr_t>(xr) & 15u) == 0) {
    const int64_t nvec = len / V::N;
    const raw* xv = reinterpret_cast<const raw*>(xr);
    constexpr int U = 8;                                     // 128-bit loads in flight per lane
    int64_t j = lane;
    for (; j + 32 * (U - 1) < nvec; j += 32 * U) {
      raw r[U];
#pragma unroll
      for (int h = 0; h < U; ++h) r[h] = ld_stream(xv + j + 32 * h);
#pragma unroll
      for (int h = 0; h < U; ++h) {
        float f[V::N];
        V::unpack(r[h], f);
#pragma unroll
        for (int e = 0; e < V::N; ++e) stat_add<ABS>(s, f[e]);
      }
    }
    if (j < nvec) {                                          // last, partial block: still all loads first
      raw r[U];
#pragma unroll
      for (int h = 0; h < U; ++h)
        if (j + 32 * h < nvec) r[h] = ld_stream(xv + j + 32 * h);
#pragma unroll
      for (int h = 0; h < U; ++h) {
        if (j + 32 * h < nvec) {
          float f[V::N];
          V::unpack(r[h], f);
#pragma unroll
          for (int e = 0; e < V::N; ++e) stat_add<ABS>(s, f[e]);
        }
      }
    }
    done = nvec * V::N;
  }
  for (int64_t j = done + lane; j < len; j += 32) stat_add<ABS>(s, to_f32<T>(xr[j]));
  s = stat_warp(s);
  if (lane == 0) {
    if (direct) stat_store(stats + 4 * (row % gm.channels), s);
    else part[item] = s;
  }
}

// channel-major statistics for per-channel activations with short rows (see fq_cmaj_kernel): one warp per
// (channel, batch chunk) walks the flattened (b, e) index space; partial [channel][chunk].
template <typename T, bool ABS, int VEC>
__global__ void __launch_bounds__(kRowWarps * 32)
stats_cmaj_kernel(const T* __restrict__ x, CmajGeom gm, Stat4* __restrict__ part) {
  using V = Vec<T>;
  using raw = typename V::raw;
  const int lane = threadIdx.x & 31;
  const int64_t item = static_cast<int64_t>(blockIdx.x) * kRowWarps + (threadIdx.x >> 5);
  if (item >= gm.channels * gm.chunks) return;
  const int64_t jc = item / gm.channels, c = item - jc * gm.channels;   // adjacent warps: adjacent channels
  const int64_t b0 = jc * gm.bc;
  const int64_t nb = (gm.outer - b0) < gm.bc ? (gm.outer - b0) : gm.bc;
  const uint32_t inner = static_cast<uint32_t>(gm.inner) / VEC;          // access units per row
  const uint32_t total = static_cast<uint32_t>(nb) * inner;
  const uint32_t plane = static_cast<uint32_t>(gm.channels * gm.inner) / VEC;
  const T* xb = x + (b0 * gm.channels + c) * gm.inner;
  Stat4 s;
  stat_init(s);
  constexpr int U = VEC == 1 ? 8 : 4;
  for (uint32_t t0 = 0; t0 < total; t0 += 32 * U) {
    uint32_t off[U];
    bool ok[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const uint32_t t = t0 + u * 32 + lane;
      ok[u] = t < total;
      const uint32_t bl = static_cast<uint32_t>((static_cast<uint64_t>(t) * gm.magic) >> 24);
      off[u] = bl * plane + (t - bl * inner);
    }
    if constexpr (VEC == 1) {
      float v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) v[u] = ok[u] ? to_f32<T>(xb[off[u]]) : 0.f;
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (ok[u]) stat_add<ABS>(s, v[u]);
    } else {
      raw r[U];
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (ok[u]) r[u] = ld_stream(reinterpret_cast<const raw*>(xb) + off[u]);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (!ok[u]) continue;
        float f[V::N];
        V::unpack(r[u], f);
#pragma unroll
        for (int e = 0; e < V::N; ++e) stat_add<ABS>(s, f[e]);
      }
    }
  }
  s = stat_warp(s);
  if (lane == 0) part[c * gm.chunks + jc] = s;
}

// slab statistics (SlabGeom, common.cuh): short rows that are not whole 128-bit vectors, read as vectors anyway;
// one Stat4 per element slot of the thread's vector, folded per channel in a fixed order; partial [channel][chunk].
template <typename T, bool ABS>
__global__ void __launch_bounds__(kThreads, 2)
stats_slab_kernel(const T* __restrict__ x, SlabGeom gm, Stat4* __restrict__ part) {
  using V = Vec<T>;
  using raw = typename V::raw;
  constexpr int U = 2 * kSlabUnroll;
  __shared__ Stat4 sh[V::N * kThreads];
  const int tid = threadIdx.x;
  const int r = tid / gm.W, v = tid - r * gm.W;
  const bool active = r < gm.R;
  const int64_t j = blockIdx.x / gm.groups, grp = blockIdx.x - j * gm.groups;
  const int64_t b0 = j * gm.bc;
  const int64_t b1 = (gm.outer - b0) < gm.bc ? gm.outer : b0 + gm.bc;
  const raw* xv = reinterpret_cast<const raw*>(x) + grp * gm.W + v;
  Stat4 s[V::N];
#pragma unroll
  for (int k = 0; k < V::N; ++k) stat_init(s[k]);
  if (active) {
    for (int64_t b = b0 + r; b < b1; b += static_cast<int64_t>(gm.R) * U) {
      raw rx[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t bb = b + static_cast<int64_t>(u) * gm.R;
        if (bb < b1) rx[u] = ld_stream(xv + bb * gm.plane_vecs);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (b + static_cast<int64_t>(u) * gm.R >= b1) break;
        float f[V::N];
        V::unpack(rx[u], f);
#pragma unroll
        for (int k = 0; k < V::N; ++k) stat_add<ABS>(s[k], f[k]);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < V::N; ++k) sh[k * kThreads + tid] = s[k];
  __syncthreads();
  // channel q of the group owns the flat elements [q * inner, (q + 1) * inner) of every row: warp w folds channels
  // w, w + 8, ... in a fixed order (row-major over its entries, then the shuffle tree)
  const int warp = tid >> 5, lane = tid & 31;
  const int inner = static_cast<int>(gm.inner);
  for (int q = warp; q < gm.G; q += kThreads / 32) {
    Stat4 t;
    stat_init(t);
    for (int i = lane; i < gm.R * inner; i += 32) {
      const int rr = i / inner, e = q * inner + (i - rr * inner);
      stat_merge(t, sh[(e % V::N) * kThreads + rr * gm.W + e / V::N]);
    }
    t = stat_warp(t);
    if (lane == 0) part[(grp * gm.G + q) * gm.chunks + j] = t;
  }
}

// one CTA per channel: merge that channel's `per` partials at part[(k / inner_n) * stride_o + ch * inner_n +
// (k % inner_n)] (rows: k = (b, seg), stride_o = C * segs, inner_n = segs; channel-major: stride_o = 0).
__global__ void __launch_bounds__(128)
stats_finalize_kernel(const Stat4* __restrict__ part, int64_t per, int64_t inner_n, int64_t stride_o,
                      float* __restrict__ stats) {
  __shared__ Stat4 sh[4];
  const int64_t ch = blockIdx.x;
  Stat4 s;
  stat_init(s);
  for (int64_t k = threadIdx.x; k < per; k += blockDim.x) {
    const int64_t o = k / inner_n, i = k - o * inner_n;
    stat_merge(s, part[o * stride_o + ch * inner_n + i]);
  }
  s = stat_warp(s);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 4; ++w) stat_merge(s, sh[w]);
    stat_store(stats + 4 * ch, s);
  }
}

// ops.py:20-34 / 121-140
// recip_mul: `tensor / python_scalar` as eager PyTorch evaluates it ON CUDA - ATen's true-division kernel multiplies
// by the reciprocal of a CPU-scalar divisor, a * (1.0f / b) (BinaryDivTrueKernel.cu, "may lose one bit of precision") -
// instead of the IEEE division the CPU kernels (and the committed fixtures, minted on the CPU) perform.
__global__ void minmax_finalize_kernel(const float* __restrict__ stats, float* __restrict__ scale,
                                       float* __restrict__ offset, int64_t channels, float qdiv, int is_signed,
                                       int allow_offset, int recip_mul) {
  const int64_t c = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (c >= channels) return;
  const float* s = stats + 4 * c;
  const float inv = 1.0f / qdiv;
  if (is_signed) {
    scale[c] = recip_mul ? s[2] * inv : s[2] / qdiv;            // abs().max() / (2^(n-1)-1)
    offset[c] = 0.f;
  } else {
    const float lo = allow_offset ? s[0] : 0.f;
    const float range = s[1] - lo;
    scale[c] = recip_mul ? range * inv : range / qdiv;          // (max - min) / (2^n - 1)
    offset[c] = lo;
  }
}

// mean|x| * multiplier, computed as (sum / count) then * multiplier like the eager chain
__global__ void absmean_finalize_kernel(const float* __restrict__ stats, float* __restrict__ out, int64_t channels,
                                        float count, float mul_a, float mul_b, int mode) {
  const int64_t c = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (c >= channels) return;
  const float mean = stats[4 * c + 3] / count;
  // mode 0: modules/base.py:84   2 * mean / sqrt(qmax)        -> (mul_a * mean) / mul_b
  // mode 1: RootQ/base.py:115    2 * mean * sqrt(qmax)        -> (mul_a * mean) * mul_b
  out[c] = mode == 0 ? (mul_a * mean) / mul_b : (mul_a * mean) * mul_b;
}

// ---------------------------------------------------------------------------------------
// 80-candidate sweep, per tensor
// ---------------------------------------------------------------------------------------
// Candidate i (ops.py:53-58): r = 1 - 0.01*i (python double, cast to fp32 when it meets the
// tensor); c_hi = r*max; c_lo = r*min; scale = (c_hi - c_lo)/qmax; zp = round(-c_lo/scale).
__device__ __forceinline__ void sweep_candidate(int i, float lo, float hi, float qmax, float& sc, float& zp) {
  const float r = static_cast<float>(1.0 - 0.01 * static_cast<double>(i));
  const float c_hi = r * hi, c_lo = r * lo;
  sc = (c_hi - c_lo) / qmax;
  zp = rintf((-c_lo) / sc);
}
// squared error of one element under one candidate (ops.py:59-61), literal chain
__device__ __forceinline__ float sweep_err2(float x, float sc, float zp, float qmax) {
  float q = rintf(x / sc) + zp;
  q = (clamp_ref(q, 0.f, qmax) - zp) * sc;
  const float d = q - x;
  return d * d;
}
// same value on the fast-path domain (|x| <= 2^60, candidate scale in [2^-40, 2^40]): residual-corrected
// division by the candidate's hoisted reciprocal, NaN-propagating min/max clamp (a zero's sign is erased
// by the following "- zp").  11 instructions instead of ~22: the sweep is fp32-issue-bound.
__device__ __forceinline__ float sweep_err2_fast(float x, const FastDiv& fd, float zp, float qmax) {
  float q = rintf(fast_div(x, fd)) + zp;
  q = (clamp_fast(q, 0.f, qmax) - zp) * fd.s;
  const float d = q - x;
  return d * d;
}

// ---- fast candidate evaluation ---------------------------------------------------------------
// With an integer zero-point zp and integer bounds, clamp(rint(q) + zp, 0, qmax) - zp ==
// rint(clamp(q, -zp, qmax - zp)) (rint is monotonic and integers are its fixed points), and for |c| < 2^22
// rint(c) == (c + 1.5*2^23) - 1.5*2^23.  That removes the half-rate FRND and two adds per element; what is
// left per candidate-element is: 3 (exact division) + 2 (max.NaN/min.NaN) + 2 (round) + 1 (x scale) +
// 1 (- x) + 1 (fma into the running sum) = 10 instructions, 8 of them on the fp32 pipe.  The fp32-pipe ops
// are issued as packed f32x2 instructions (sm_100 FFMA2 / FMUL2 / FADD2: two IEEE-RN results per lane per
// issue slot), which is what the sweep - issue-bound once x sits in registers - is limited by.
// Valid when the candidate scale is in the fast-division domain, |zp| <= 2^21 and qmax <= 2^21; every
// per-element value is bit-identical to sweep_err2, only the summation order differs.
struct SweepCand {
  float ns;   // -scale
  float r;    // RN(1 / scale)
  float a;    // -zp
  float b;    // qmax - zp
};
__device__ __forceinline__ bool sweep_cand_fast(float sc, float zp, float qmax, SweepCand& c) {
  const FastDiv fd = make_fastdiv(sc);
  c.ns = -sc;
  c.r = fd.r;
  c.a = -zp;
  c.b = qmax - zp;
  return fd.ok && (fabsf(zp) <= 0x1p21f) && (qmax <= 0x1p21f);   // NaN zp -> false
}
__device__ __forceinline__ float2 sweep_pair_fast(float2 x, const SweepCand& c, float2 acc) {
  const float2 r2 = make_float2(c.r, c.r), ns2 = make_float2(c.ns, c.ns);
  const float2 q0 = __fmul2_rn(x, r2);
  const float2 e = __ffma2_rn(ns2, q0, x);
  const float2 q = __ffma2_rn(e, r2, q0);
  float2 k;
  k.x = min_nan(max_nan(q.x, c.a), c.b);
  k.y = min_nan(max_nan(q.y, c.a), c.b);
  const float2 t = __fadd2_rn(k, make_float2(kRoundMagic, kRoundMagic));
  const float2 rr = __fadd2_rn(t, make_float2(-kRoundMagic, -kRoundMagic));
  // -(code - zp) * scale with two scalar mul.rn: ptxas contracts a mul.rn.f32x2 feeding an add.rn.f32x2
  // into one FFMA2 (it never does for scalar mul.rn), which would skip the reference's rounding of the
  // dequantised value.
  const float2 ny = make_float2(__fmul_rn(rr.x, c.ns), __fmul_rn(rr.y, c.ns));
  const float2 d = __fadd2_rn(x, ny);               // x - y: same square as y - x
  return __ffma2_rn(d, d, acc);
}
__device__ __forceinline__ float sweep_one_fast(float x, const SweepCand& c, float acc) {
  const float q0 = __fmul_rn(x, c.r);
  const float e = __fmaf_rn(c.ns, q0, x);
  const float q = __fmaf_rn(e, c.r, q0);
  const float k = min_nan(max_nan(q, c.a), c.b);
  const float rr = (k + kRoundMagic) - kRoundMagic;
  const float d = x + rr * c.ns;
  return __fmaf_rn(d, d, acc);
}

constexpr int kSweepElems = 16;  // elements a thread holds in registers per tile (fp32: four 128-bit loads)

// Per-thread running sums live in shared memory ([candidate][thread], conflict-free): one LDS + STS per
// candidate per tile instead of a 10-instruction warp reduction; the block reduces them once at the end.
template <typename T>
__global__ void __launch_bounds__(kThreads, 2)
sweep_tensor_kernel(const T* __restrict__ x, int64_t n, const float* __restrict__ stats, float qmax, int allow_offset,
                    float* __restrict__ sse, void* ws) {
  using V = Vec<T>;
  using raw = typename V::raw;
  constexpr int NV = kSweepElems / V::N >= 1 ? kSweepElems / V::N : 1;   // vectors per thread per tile
  constexpr int NE = NV * V::N;
  extern __shared__ __align__(16) float w_acc[];                          // [kNC][kThreads]
  __shared__ float c_sc[kNC], c_zp[kNC];
  __shared__ __align__(16) SweepCand c_par[kNC];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int ok = 1;
  if (threadIdx.x < kNC) {
    const float lo = allow_offset ? stats[0] : 0.f;
    sweep_candidate(threadIdx.x, lo, stats[1], qmax, c_sc[threadIdx.x], c_zp[threadIdx.x]);
    SweepCand c;
    ok = sweep_cand_fast(c_sc[threadIdx.x], c_zp[threadIdx.x], qmax, c) ? 1 : 0;
    c_par[threadIdx.x] = c;
  }
  for (int k = threadIdx.x; k < kNC * kThreads; k += kThreads) w_acc[k] = 0.f;
  const bool all_fast = __syncthreads_and(ok) != 0;
  float* my_acc = w_acc + threadIdx.x;

  const bool vec = (reinterpret_cast<uintptr_t>(x) & 15u) == 0;
  const int64_t nvec = vec ? n / V::N : 0;
  const int64_t tiles = nvec / (static_cast<int64_t>(kThreads) * NV);   // full tiles only
  const raw* xv = reinterpret_cast<const raw*>(x);
  for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
    float f[NE];
    raw r[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) r[v] = ld_stream(xv + (t * NV + v) * kThreads + threadIdx.x);
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      float tmp[V::N];
      V::unpack(r[v], tmp);
#pragma unroll
      for (int e = 0; e < V::N; ++e) f[v * V::N + e] = tmp[e];
    }
    float m = 0.f;
#pragma unroll
    for (int e = 0; e < NE; ++e) m = fmaxf(m, fabsf(f[e]));
    if (all_fast && m <= kFastDivMaxX) {         // inf / huge values: literal chain for this thread's tile
#pragma unroll 2
      for (int c = 0; c < kNC; ++c) {
        const SweepCand cp = c_par[c];
        float2 a0 = make_float2(0.f, 0.f), a1 = make_float2(0.f, 0.f);
#pragma unroll
        for (int e = 0; e < NE; e += 4) {
          a0 = sweep_pair_fast(make_float2(f[e], f[e + 1]), cp, a0);
          a1 = sweep_pair_fast(make_float2(f[e + 2], f[e + 3]), cp, a1);
        }
        my_acc[c * kThreads] += (a0.x + a0.y) + (a1.x + a1.y);
      }
    } else {
      for (int c = 0; c < kNC; ++c) {
        const float sc = c_sc[c], zp = c_zp[c];
        float a = 0.f;
#pragma unroll
        for (int e = 0; e < NE; ++e) a += sweep_err2(f[e], sc, zp, qmax);
        my_acc[c * kThreads] += a;
      }
    }
  }
  // remainder (elements past the last full tile, or everything when x is unaligned): block 0
  if (blockIdx.x == 0) {
    const int64_t start = tiles * kThreads * NE;
    for (int64_t j = start + threadIdx.x; j < n; j += kThreads) {
      const float v = to_f32<T>(x[j]);
      for (int c = 0; c < kNC; ++c) my_acc[c * kThreads] += sweep_err2(v, c_sc[c], c_zp[c], qmax);
    }
  }
  __syncthreads();
  // block reduction: warp w sums candidates w, w+8, ... over the 256 per-thread sums in a fixed order
  float* part = ws_partials(ws);
  for (int c = warp; c < kNC; c += kThreads / 32) {
    float a = 0.f;
#pragma unroll
    for (int k = 0; k < kThreads / 32; ++k) a += w_acc[c * kThreads + k * 32 + lane];
    a = warp_sum(a);
    if (lane == 0) part[static_cast<int64_t>(blockIdx.x) * kNC + c] = a;
  }
  // the partials above are stored by lane 0 of ALL warps: every warp must have stored before thread 0 fences and
  // draws the ticket (the barrier + thread 0's cumulative fence order all of this CTA's partials before the ticket)
  __syncthreads();
  if (take_last_ticket(ws_counter(ws), gridDim.x)) {
    if (threadIdx.x < kNC) {
      double a = 0.0;
      for (int b = 0; b < static_cast<int>(gridDim.x); ++b) a += part[static_cast<int64_t>(b) * kNC + threadIdx.x];
      sse[threadIdx.x] = static_cast<float>(a);
    }
    if (threadIdx.x == 0) *ws_counter(ws) = 0u;
  }
}

// ops.py:48-66: loss_i = l2_loss = sse_i / rows_for_mean; first strict minimum below 1000 wins,
// otherwise the fallback (max/qmax, 0) of :49-50 stays.
__global__ void sweep_tensor_finalize_kernel(const float* __restrict__ sse, const float* __restrict__ stats,
                                             float rows_for_mean, float qmax, int allow_offset,
                                             float* __restrict__ scale, float* __restrict__ offset,
                                             int32_t* __restrict__ picked) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const float lo = allow_offset ? stats[0] : 0.f, hi = stats[1];
  float best = 1000.f, s_out = hi / qmax, z_out = 0.f;
  int pick = -1;
  for (int i = 0; i < kNC; ++i) {
    const float loss = sse[i] / rows_for_mean;
    if (loss < best) {
      best = loss;
      pick = i;
      sweep_candidate(i, lo, hi, qmax, s_out, z_out);
    }
  }
  scale[0] = s_out;
  offset[0] = z_out;
  if (picked) picked[0] = pick;
}

// ---------------------------------------------------------------------------------------
// 80-candidate sweep, per channel: `wpr` warps per row (1, 2, 4 or 8 - chosen on the host so that few-row
// tensors still fill the GPU), the row staged ONCE in shared memory by a bulk async copy (TMA 1-D:
// cp.async.bulk + mbarrier, SASS UBLKCP) and swept 80 times on chip.  The reference's accept rule is
// sequential (ops.py:191-194 and its aliasing of min_val with the offset vector), so every candidate's
// sum is reduced across the row's warps before the next candidate's scale is known: warp shuffle ->
// shared memory -> named barrier of the row's warps only, double-buffered by parity.
// ---------------------------------------------------------------------------------------
constexpr int kSweepWarps = 8;                 // warps per CTA
constexpr int kSweepSmemFloats = 50 * 1024;    // 200 KB of row staging per CTA at most

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void group_bar(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

struct SweepRowGroup {
  float* red;      // [2][kSweepWarps] exchange slots of this row's warps
  int wpr, wig, lane, bar_id;
  int parity;
  // all-reduce over the row's warps; every thread of the group returns the same value (fixed order)
  template <typename Op>
  __device__ __forceinline__ float all(float v, Op op) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
    if (wpr == 1) return v;
    float* slot = red + parity * kSweepWarps;
    parity ^= 1;
    if (lane == 0) slot[wig] = v;
    group_bar(bar_id, wpr * 32);
    float t = slot[0];
    for (int w = 1; w < wpr; ++w) t = op(t, slot[w]);
    return t;
  }
};

template <typename T>
__device__ __forceinline__ void sweep_channel_body(const T* __restrict__ x, int64_t channels, int64_t inner, float qmax,
                                                   float signed_div, int is_signed, float* __restrict__ scale,
                                                   float* __restrict__ offset, int wpr, int row_floats, int staged,
                                                   int64_t cta) {
  extern __shared__ __align__(128) unsigned char dyn_smem[];
  __shared__ __align__(8) unsigned long long bars[kSweepWarps];
  __shared__ float red_all[kSweepWarps][2][kSweepWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int group = warp / wpr, wig = warp - group * wpr;
  const int rows_per_cta = kSweepWarps / wpr;
  const int64_t row = cta * rows_per_cta + group;
  if (row >= channels) return;                 // a whole row group exits together; barriers are per group
  const int tg = wig * 32 + lane, gt = wpr * 32;
  SweepRowGroup grp{&red_all[group][0][0], wpr, wig, lane, group + 1, 0};
  float* buf = reinterpret_cast<float*>(dyn_smem) + static_cast<size_t>(group) * row_floats;
  const T* xr = x + row * inner;
  const float* src = nullptr;                  // fp32 view of the row in shared memory (element j at src[j])
  int64_t h = 0, body = 0;                     // [h, h+body) is the 16-byte aligned interior
  if (staged) {
    float* dst = buf + 4;
    if (sizeof(T) == 4) {
      // aligned interior by one bulk async copy issued by the group's first thread; the <=3 head and
      // tail elements by plain loads.  dst + h is 16-byte aligned in shared memory like xr + h in global.
      const uintptr_t a = reinterpret_cast<uintptr_t>(xr);
      const int head = static_cast<int>(((16 - (a & 15u)) & 15u) / 4);
      h = head < inner ? head : inner;
      body = ((inner - h) / 4) * 4;
      dst = buf + 4 - h;
      const uint32_t bar = smem_u32(&bars[group]);
      if (tg == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      }
      if (wpr == 1) __syncwarp(); else group_bar(grp.bar_id, gt);
      if (body > 0 && tg == 0) {
        const uint32_t bytes = static_cast<uint32_t>(body * 4);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(dst + h)), "l"(reinterpret_cast<const float*>(xr) + h), "r"(bytes), "r"(bar)
                     : "memory");
      }
      for (int64_t j = tg; j < h; j += gt) dst[j] = to_f32<T>(xr[j]);
      for (int64_t j = h + body + tg; j < inner; j += gt) dst[j] = to_f32<T>(xr[j]);
      if (body > 0) {
        uint32_t ok = 0;
        while (!ok) {
          asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                       "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(bar), "r"(0u) : "memory");
        }
      }
    } else {
      for (int64_t j = tg; j < inner; j += gt) dst[j] = to_f32<T>(xr[j]);   // bf16: convert while staging
      body = (inner / 4) * 4;
    }
    if (wpr == 1) __syncwarp(); else group_bar(grp.bar_id, gt);
    src = dst;
  }
  auto at = [&](int64_t j) -> float { return staged ? src[j] : to_f32<T>(xr[j]); };
  const int64_t nvec = staged ? body / 4 : 0;
  const float4* sv = reinterpret_cast<const float4*>(src + h);
  const int64_t n_edge = staged ? inner - body : 0;       // head + tail elements, handled one per thread

  // row statistics (ops.py:171 -> quantize_minmax_channel)
  float mn = INFINITY, mx = -INFINITY, am = 0.f, nanf_ = 0.f;
  for (int64_t j = tg; j < inner; j += gt) {
    const float v = at(j);
    nanf_ = (v != v) ? 1.f : nanf_;
    mn = fminf(mn, v); mx = fmaxf(mx, v); am = fmaxf(am, fabsf(v));
  }
  auto fmin_op = [](float a, float b) { return fminf(a, b); };
  auto fmax_op = [](float a, float b) { return fmaxf(a, b); };
  auto add_op = [](float a, float b) { return a + b; };
  mn = grp.all(mn, fmin_op); mx = grp.all(mx, fmax_op); am = grp.all(am, fmax_op);
  const bool nan = grp.all(nanf_, fmax_op) != 0.f;
  const bool row_fast = am <= kFastDivMaxX;      // no inf / huge value in the row
  if (nan) mn = mx = am = NAN;
  float cur_scale, cur_off;
  if (is_signed) { cur_scale = am / signed_div; cur_off = 0.f; }           // ops.py:125-127
  else           { cur_off = mn; cur_scale = (mx - mn) / qmax; }           // ops.py:129-136
  float min_v = cur_off;                                                   // ops.py:172 (alias of offset)
  const float max_v = cur_off + cur_scale * qmax;                          // ops.py:173
  float best = 1000.f;                                                     // ops.py:176
  for (int i = 0; i < kNC; ++i) {
    float sc, zp;
    sweep_candidate(i, min_v, max_v, qmax, sc, zp);                        // ops.py:179-185
    SweepCand cp;
    const bool fast = sweep_cand_fast(sc, zp, qmax, cp) && row_fast;
    float a = 0.f;
    if (fast && staged) {
      float2 a0 = make_float2(0.f, 0.f), a1 = make_float2(0.f, 0.f);
      for (int64_t v = tg; v < nvec; v += gt) {
        const float4 q = sv[v];
        a0 = sweep_pair_fast(make_float2(q.x, q.y), cp, a0);
        a1 = sweep_pair_fast(make_float2(q.z, q.w), cp, a1);
      }
      a = (a0.x + a0.y) + (a1.x + a1.y);
      if (tg < n_edge) a = sweep_one_fast(src[tg < h ? tg : body + tg], cp, a);
    } else if (fast) {
      for (int64_t j = tg; j < inner; j += gt) a = sweep_one_fast(at(j), cp, a);
    } else {
      for (int64_t j = tg; j < inner; j += gt) a += sweep_err2(at(j), sc, zp, qmax);
    }
    a = grp.all(a, add_op);
    if (best > a) {                                                        // ops.py:191-194
      cur_scale = sc;
      cur_off = zp;
      min_v = zp;           // offset[c] = new_offset also rewrites min_val[c] (reference aliasing)
      best = a;
    }
  }
  if (tg == 0) { scale[row] = cur_scale; offset[row] = cur_off; }
}

template <typename T>
__global__ void __launch_bounds__(kSweepWarps * 32)
sweep_channel_kernel(const T* __restrict__ x, int64_t channels, int64_t inner, float qmax, float signed_div,
                     int is_signed, float* __restrict__ scale, float* __restrict__ offset, int wpr, int row_floats,
                     int staged) {
  sweep_channel_body<T>(x, channels, inner, qmax, signed_div, is_signed, scale, offset, wpr, row_floats, staged,
                        blockIdx.x);
}

// All per-channel weight sweeps of a model in ONE launch: a CNN's 23-54 weight tensors are swept in 50-150 us each
// when launched one by one (the 80 dependent candidates set a ~45 us floor per launch however few rows a tensor has).
// CTA b finds its tensor by a binary search over the CTA prefix; every tensor keeps the geometry (warps per row,
// staging) its own launch would use, so the result is bit-identical to the per-tensor call.
template <typename T>
__global__ void __launch_bounds__(kSweepWarps * 32)
sweep_channel_grouped_kernel(const dlmcq_sweep_item* __restrict__ items, const int64_t* __restrict__ cta_prefix,
                             int n_items) {
  int lo = 0, hi = n_items - 1;
  const int64_t b = blockIdx.x;
  while (lo < hi) {                                     // last item whose first CTA is <= b
    const int mid = (lo + hi + 1) >> 1;
    if (cta_prefix[mid] <= b) lo = mid; else hi = mid - 1;
  }
  const dlmcq_sweep_item it = items[lo];
  const float qmax = static_cast<float>((1 << it.n_bits) - 1);
  const float sdiv = static_cast<float>((1 << (it.n_bits - 1)) - 1);
  sweep_channel_body<T>(static_cast<const T*>(it.x), it.channels, it.inner, qmax, sdiv, it.is_signed, it.scale,
                        it.offset, it.wpr, it.row_floats, it.staged, b - cta_prefix[lo]);
}

// ---------------------------------------------------------------------------------------
// l2norm fixed point: one iteration
// ---------------------------------------------------------------------------------------
// Inner product terms of one iteration on the fast path (packed f32x2, 6 issue slots per element):
//   code = clamp(rint(q), lo, hi) == rint(clamp(q, lo, hi)) for integer bounds == (c + 1.5*2^23) - 1.5*2^23;
//   a += x * code ; b += code * code + 1e-7 (code^2 is exact, so fma(code, code, 1e-7) is the reference's
//   rounded sum).  The sign of a zero code is not kept - it cannot change either dot product.
__device__ __forceinline__ void l2norm_pair_fast(float2 x, const ChanParams& p, float lo, float hi, float2& a,
                                                 float2& b) {
  const float2 r2 = make_float2(p.fd.r, p.fd.r), ns2 = make_float2(-p.div, -p.div);
  const float2 num = __fadd2_rn(x, make_float2(-p.off, -p.off));
  const float2 q0 = __fmul2_rn(num, r2);
  const float2 e = __ffma2_rn(ns2, q0, num);
  const float2 q = __ffma2_rn(e, r2, q0);
  float2 k;
  k.x = min_nan(max_nan(q.x, lo), hi);
  k.y = min_nan(max_nan(q.y, lo), hi);
  const float2 t = __fadd2_rn(k, make_float2(kRoundMagic, kRoundMagic));
  const float2 code = __fadd2_rn(t, make_float2(-kRoundMagic, -kRoundMagic));
  a = __ffma2_rn(x, code, a);
  b = __fadd2_rn(b, __ffma2_rn(code, code, make_float2(1e-7f, 1e-7f)));
}

template <typename T>
__global__ void __launch_bounds__(kRowWarps * 32)
l2norm_rows_kernel(const T* __restrict__ x, RowGeom gm, const float* __restrict__ scale,
                   const float* __restrict__ offset, float lo, float hi, const int32_t* __restrict__ done,
                   float* __restrict__ part) {
  using V = Vec<T>;
  using raw = typename V::raw;
  if (*done) return;
  const int lane = threadIdx.x & 31;
  const int64_t item = static_cast<int64_t>(blockIdx.x) * kRowWarps + (threadIdx.x >> 5);
  if (item >= gm.rows * gm.segs) return;
  const int64_t row = item / gm.segs, seg = item - row * gm.segs;
  const ChanParams p = make_params<DLMCQ_FORM_A1>(scale, offset, row % gm.channels, 0.f, lo, hi);
  const int64_t beg = seg * gm.seg;
  const int64_t len = (gm.inner - beg) < gm.seg ? (gm.inner - beg) : gm.seg;
  const T* xr = x + row * gm.inner + beg;
  float a = 0.f, b = 0.f;
  float2 a2 = make_float2(0.f, 0.f), b2 = make_float2(0.f, 0.f);
  const bool fast_p = p.fd.ok && fabsf(p.off) <= 0x1p59f;
  auto add_vec = [&](const float (&f)[V::N]) {
    float m = 0.f;
#pragma unroll
    for (int e = 0; e < V::N; ++e) m = fmaxf(m, fabsf(f[e]));
    if (fast_p && m <= 0x1p59f) {                            // |x - off| <= 2^60: the verified division domain
#pragma unroll
      for (int e = 0; e < V::N; e += 2) l2norm_pair_fast(make_float2(f[e], f[e + 1]), p, lo, hi, a2, b2);
    } else {
      float code[V::N], y[V::N];
      fq_vec<DLMCQ_FORM_A1, V::N>(f, p, lo, hi, code, y);   // ops.py:78,206 quantize()
#pragma unroll
      for (int e = 0; e < V::N; ++e) {
        a += f[e] * code[e];                                 // (tensor * tensor_q).sum()
        b += code[e] * code[e] + 1e-7f;                      // (tensor_q * tensor_q + 1e-7).sum()
      }
    }
  };
  auto add = [&](float v) {
    float code, y;
    fq_elem<DLMCQ_FORM_A1>(v, p, lo, hi, code, y);
    a += v * code;
    b += code * code + 1e-7f;
  };
  int64_t fin = 0;
  if ((reinterpret_cast<uintptr_t>(xr) & 15u) == 0) {
    const int64_t nvec = len / V::N;
    const raw* xv = reinterpret_cast<const raw*>(xr);
    constexpr int U = 4;                                     // 128-bit loads in flight per lane
    int64_t j = lane;
    for (; j + 32 * (U - 1) < nvec; j += 32 * U) {
      raw r[U];
#pragma unroll
      for (int h = 0; h < U; ++h) r[h] = ld_stream(xv + j + 32 * h);
#pragma unroll
      for (int h = 0; h < U; ++h) {
        float f[V::N];
        V::unpack(r[h], f);
        add_vec(f);
      }
    }
    if (j < nvec) {                                          // last, partial block: still all loads first
      raw r[U];
#pragma unroll
      for (int h = 0; h < U; ++h)
        if (j + 32 * h < nvec) r[h] = ld_stream(xv + j + 32 * h);
#pragma unroll
      for (int h = 0; h < U; ++h) {
        if (j + 32 * h < nvec) {
          float f[V::N];
          V::unpack(r[h], f);
          add_vec(f);
        }
      }
    }
    fin = nvec * V::N;
  }
  for (int64_t j = fin + lane; j < len; j += 32) add(to_f32<T>(xr[j]));
  a += a2.x + a2.y;
  b += b2.x + b2.y;
  a = warp_sum(a);
  b = warp_sum(b);
  if (lane == 0) { part[2 * item] = a; part[2 * item + 1] = b; }
}

// Per-tensor (one channel): a single CTA strides over the segments, computes the new scale, the convergence
// measure and the done flag (ops.py:79-81).
__global__ void __launch_bounds__(kThreads)
l2norm_finalize_kernel(const float* __restrict__ part, RowGeom gm, float* __restrict__ scale, float* __restrict__ diff,
                       int32_t* __restrict__ done, int32_t* __restrict__ iters) {
  __shared__ double sh[2][kThreads / 32];
  if (*done) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double a = 0.0, b = 0.0;
  for (int64_t sg = threadIdx.x; sg < gm.segs; sg += blockDim.x) {
    a += part[2 * sg];
    b += part[2 * sg + 1];
  }
  a = warp_sum(a);
  b = warp_sum(b);
  if (lane == 0) { sh[0][warp] = a; sh[1][warp] = b; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double ta = 0.0, tb = 0.0;
    for (int w = 0; w < kThreads / 32; ++w) { ta += sh[0][w]; tb += sh[1][w]; }
    const float s_old = scale[0];
    const float s_new = static_cast<float>(ta) / static_cast<float>(tb);
    scale[0] = s_new;
    const float df = fabsf(s_new - s_old) / s_old;                      // ops.py:80
    diff[0] = df;
    if (iters) iters[0] += 1;
    if (!(df > 1e-5f)) done[0] = 1;                                     // `while diff > epsilon`
  }
}

// Per-channel variant: one thread per channel over ceil(C / 256) CTAs; the CTA that draws the last ticket
// combines the per-CTA (|ds|^2, |s|^2) sums in a fixed order and sets the convergence flag (ops.py:207-210).
__global__ void __launch_bounds__(kThreads)
l2norm_finalize_channels_kernel(const float* __restrict__ part, RowGeom gm, float* __restrict__ scale,
                                float* __restrict__ diff, int32_t* __restrict__ done, int32_t* __restrict__ iters,
                                double* __restrict__ cta_part, unsigned int* __restrict__ counter) {
  __shared__ double sh[2][kThreads / 32];
  if (*done) return;        // only the last CTA of an iteration ever sets it, after every CTA passed this test
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t c = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x;
  double num = 0.0, den = 0.0;
  if (c < gm.channels) {
    double a = 0.0, b = 0.0;
    for (int64_t sg = 0; sg < gm.segs; ++sg) {
      a += part[2 * (c * gm.segs + sg)];
      b += part[2 * (c * gm.segs + sg) + 1];
    }
    const float s_old = scale[c];
    const float s_new = static_cast<float>(a) / static_cast<float>(b);
    scale[c] = s_new;
    const float d = s_new - s_old;
    num = static_cast<double>(d * d);
    den = static_cast<double>(s_old * s_old);
  }
  num = warp_sum(num);
  den = warp_sum(den);
  if (lane == 0) { sh[0][warp] = num; sh[1][warp] = den; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double tn = 0.0, td = 0.0;
    for (int w = 0; w < kThreads / 32; ++w) { tn += sh[0][w]; td += sh[1][w]; }
    cta_part[2 * blockIdx.x] = tn;
    cta_part[2 * blockIdx.x + 1] = td;
  }
  if (take_last_ticket(counter, gridDim.x)) {
    if (threadIdx.x == 0) {
      double tn = 0.0, td = 0.0;
      for (unsigned int b = 0; b < gridDim.x; ++b) { tn += cta_part[2 * b]; td += cta_part[2 * b + 1]; }
      const float df = sqrtf(static_cast<float>(tn)) / sqrtf(static_cast<float>(td));   // ops.py:209
      diff[0] = df;
      if (iters) iters[0] += 1;
      if (!(df > 1e-5f)) done[0] = 1;
      *counter = 0u;
    }
  }
}

// ---------------------------------------------------------------------------------------
// l2norm fixed point, RESIDENT form: the whole loop of ops.py:71-83 / 198-215 in ONE launch.
//
// The step-wise form above re-reads the tensor from HBM on every one of the 50-100 iterations and needs two launches
// plus a host poll per few iterations.  A per-channel weight matrix (<= 9.4 MB for a CNN layer) fits in the GPU's
// shared memory (148 x 200 KB), so: every CTA stages its (row, 2048-element segment) items ONCE, then all CTAs iterate
// on chip - per iteration one warp pass over each staged item (A1 codes, the two dot products), a grid barrier, one
// thread per row forming the new scale and its share of the convergence norm, a second grid barrier, and every CTA
// evaluating the same convergence test from the same G partials in the same order (so no third barrier).  Launched
// cooperatively (all CTAs co-resident); the barrier is a monotonically increasing arrival counter.  Deterministic.
// ---------------------------------------------------------------------------------------
constexpr int kResSeg = 2048;                       // floats per staged item (one warp sweeps it)
constexpr int kResSlots = 24;                       // items per CTA at most: 24 x 8 KB = 192 KB
constexpr int kResWarps = 8;

template <typename T>
__global__ void __launch_bounds__(kResWarps * 32, 1)
l2norm_resident_kernel(const T* __restrict__ x, int64_t channels, int64_t inner, int segs, float* __restrict__ scale,
                       const float* __restrict__ offset, float lo, float hi, int max_iters, float* __restrict__ diff,
                       int32_t* __restrict__ done, int32_t* __restrict__ iters, double* __restrict__ cta_part,
                       unsigned int* __restrict__ counters) {
  extern __shared__ __align__(16) float stage[];                        // [slots][kResSeg]
  __shared__ double sh[2][kResWarps];
  __shared__ float item_a[kResSlots], item_b[kResSlots], s_loc[kResSlots];
  __shared__ int s_stop;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int G = gridDim.x;
  const bool single = channels == 1;
  // local items: single row: items blockIdx.x, +G, ...; otherwise rows blockIdx.x, +G, ... with `segs` slots each
  const int64_t total_items = channels * segs;
  int n_slots = 0;
  if (single) n_slots = static_cast<int>((total_items - blockIdx.x + G - 1) / G);
  else n_slots = static_cast<int>((channels - blockIdx.x + G - 1) / G) * segs;
  if (n_slots < 0) n_slots = 0;
  auto slot_row = [&](int slot) -> int64_t { return single ? 0 : blockIdx.x + static_cast<int64_t>(slot / segs) * G; };
  auto slot_seg = [&](int slot) -> int64_t { return single ? blockIdx.x + static_cast<int64_t>(slot) * G : slot % segs; };
  for (int slot = 0; slot < n_slots; ++slot) {                          // stage once, zero-padded
    const int64_t row = slot_row(slot), beg = slot_seg(slot) * kResSeg;
    const int64_t len = (inner - beg) < kResSeg ? (inner - beg) : kResSeg;
    const T* xr = x + row * inner + beg;
    float* dst = stage + slot * kResSeg;
    for (int j = threadIdx.x; j < kResSeg; j += blockDim.x) dst[j] = j < len ? to_f32<T>(xr[j]) : 0.f;
  }
  const int n_rows_loc = single ? 1 : n_slots / segs;
  if (threadIdx.x < n_rows_loc) s_loc[threadIdx.x] = scale[single ? 0 : blockIdx.x + static_cast<int64_t>(threadIdx.x) * G];
  __syncthreads();
  unsigned int barrier_no = 0;
  int it_count = 0;
  while (true) {
    // ---- one warp per staged item: sum x*code and sum(code*code + 1e-7)
    for (int slot = warp; slot < n_slots; slot += kResWarps) {
      const int64_t row = slot_row(slot), beg = slot_seg(slot) * kResSeg;
      const int len = static_cast<int>((inner - beg) < kResSeg ? (inner - beg) : kResSeg);
      ChanParams p;                                                   // A1 form: divisor s + 1e-7, multiplier s
      {
        const float sc = s_loc[single ? 0 : slot / segs];
        p.off = offset ? __ldg(offset + row) : 0.f;
        p.div = sc + 1e-7f;
        p.mul = sc;
        p.fd = make_fastdiv(p.div);
        p.fd.ok = p.fd.ok && (fabsf(lo) <= 0x1p21f) && (fabsf(hi) <= 0x1p21f) && (fabsf(p.off) <= kFastDivMaxX);
      }
      const float* src = stage + slot * kResSeg;
      const bool fast_p = p.fd.ok && fabsf(p.off) <= 0x1p59f;
      float a = 0.f, b = 0.f;
      float2 a2 = make_float2(0.f, 0.f), b2 = make_float2(0.f, 0.f);
      const int nvec = len / 4;
      for (int v = lane; v < nvec; v += 32) {
        const float4 q = reinterpret_cast<const float4*>(src)[v];
        const float f[4] = {q.x, q.y, q.z, q.w};
        const float m = fmaxf(fmaxf(fabsf(f[0]), fabsf(f[1])), fmaxf(fabsf(f[2]), fabsf(f[3])));
        if (fast_p && m <= 0x1p59f) {
          l2norm_pair_fast(make_float2(f[0], f[1]), p, lo, hi, a2, b2);
          l2norm_pair_fast(make_float2(f[2], f[3]), p, lo, hi, a2, b2);
        } else {
          float code[4], y[4];
          fq_vec<DLMCQ_FORM_A1, 4>(f, p, lo, hi, code, y);
#pragma unroll
          for (int e = 0; e < 4; ++e) { a += f[e] * code[e]; b += code[e] * code[e] + 1e-7f; }
        }
      }
      for (int j = nvec * 4 + lane; j < len; j += 32) {
        float code, y;
        fq_elem<DLMCQ_FORM_A1>(src[j], p, lo, hi, code, y);
        a += src[j] * code;
        b += code * code + 1e-7f;
      }
      a += a2.x + a2.y;
      b += b2.x + b2.y;
      a = warp_sum(a);
      b = warp_sum(b);
      if (lane == 0) { item_a[slot] = a; item_b[slot] = b; }
    }
    __syncthreads();
    // ---- per-row new scale (local) or the CTA's share of the single row's sums; one (num, den) pair per CTA
    double num = 0.0, den = 0.0;
    float s_new_loc = 0.f;
    if (single) {
      if (threadIdx.x == 0) {
        for (int sl = 0; sl < n_slots; ++sl) { num += static_cast<double>(item_a[sl]); den += static_cast<double>(item_b[sl]); }
      }
    } else if (threadIdx.x < n_rows_loc) {
      double a = 0.0, b = 0.0;
      for (int sg = 0; sg < segs; ++sg) {
        a += static_cast<double>(item_a[threadIdx.x * segs + sg]);
        b += static_cast<double>(item_b[threadIdx.x * segs + sg]);
      }
      const float s_old = s_loc[threadIdx.x];
      s_new_loc = static_cast<float>(a) / static_cast<float>(b);       // ops.py:207
      const float d = s_new_loc - s_old;
      num = static_cast<double>(d * d);
      den = static_cast<double>(s_old * s_old);
    }
    num = warp_sum(num);
    den = warp_sum(den);
    if (lane == 0) { sh[0][warp] = num; sh[1][warp] = den; }
    __syncthreads();
    if (!single && threadIdx.x < n_rows_loc) s_loc[threadIdx.x] = s_new_loc;
    if (threadIdx.x == 0) {
      double tn = 0.0, td = 0.0;
      for (int w = 0; w < kResWarps; ++w) { tn += sh[0][w]; td += sh[1][w]; }
      cta_part[2 * blockIdx.x] = tn;
      cta_part[2 * blockIdx.x + 1] = td;
    }
    barrier_no += 1;
    grid_barrier(counters, barrier_no * G);
    // ---- the same decision in every CTA, from the same G pairs in the same order (warp 0: lane-strided partial sums,
    // fixed shuffle tree - identical in every CTA)
    it_count += 1;
    double tn = 0.0, td = 0.0;
    if (warp == 0) {
      for (int b = lane; b < G; b += 32) { tn += __ldcg(cta_part + 2 * b); td += __ldcg(cta_part + 2 * b + 1); }
      tn = warp_sum(tn);
      td = warp_sum(td);
    }
    if (threadIdx.x == 0) {
      float df;
      if (single) {
        const float s_old = s_loc[0];
        const float s_new = static_cast<float>(tn) / static_cast<float>(td);          // ops.py:79
        df = fabsf(s_new - s_old) / s_old;                                            // ops.py:80
        s_loc[0] = s_new;
      } else {
        df = sqrtf(static_cast<float>(tn)) / sqrtf(static_cast<float>(td));           // ops.py:209
      }
      const bool conv = !(df > 1e-5f);                                                // `while diff > epsilon`
      s_stop = (conv || it_count >= max_iters) ? 1 : 0;
      if (blockIdx.x == 0) {
        diff[0] = df;
        iters[0] = it_count;
        done[0] = conv ? 1 : 0;
      }
    }
    __syncthreads();
    if (s_stop) break;
    // the next iteration's exchange reuses cta_part: nobody may overwrite it before every CTA has read this round's
    // values - guaranteed, because a CTA writes cta_part only after its own pass over the items AND the others can
    // only reach their next write after the same barrier count; a slow reader is still protected by parity:
    cta_part += 2 * G * ((it_count & 1) ? 1 : -1);
  }
  if (threadIdx.x < n_rows_loc && (!single || blockIdx.x == 0))
    scale[single ? 0 : blockIdx.x + static_cast<int64_t>(threadIdx.x) * G] = s_loc[threadIdx.x];
  // leave the workspace counters zeroed: the last CTA out resets them
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(counters + 1, 1u) == static_cast<unsigned int>(G) - 1u) {
      counters[0] = 0u;
      counters[1] = 0u;
    }
  }
}

template <typename T, bool ABS>
static int stats_launch(const T* x, float* stats, const dlmcq_layout* l, void* ws, size_t ws_bytes, cudaStream_t st) {
  const int64_t n = l->outer * l->channels * l->inner;
  if (ws_bytes < dlmcq_workspace_bytes(l)) return DLMCQ_EWORKSPACE;
  if (l->channels == 1) {
    const int64_t tiles = (n / Vec<T>::N + kThreads * 4 - 1) / (kThreads * 4);
    stats_flat_kernel<T, ABS><<<stream_grid(tiles, 8), kThreads, 0, st>>>(x, n, stats, ws);
  } else if (slab_ok<T>(l->outer, l->channels, l->inner, x, nullptr, nullptr, nullptr)) {
    const SlabGeom sg = make_slab<T>(l->outer, l->channels, l->inner);
    Stat4* part = reinterpret_cast<Stat4*>(ws_partials(ws));
    stats_slab_kernel<T, ABS><<<static_cast<unsigned>(sg.groups) * sg.chunks, kThreads, 0, st>>>(x, sg, part);
    DLMCQ_LAUNCH_CHECK();
    stats_finalize_kernel<<<static_cast<unsigned>(sg.channels), 128, 0, st>>>(part, sg.chunks, sg.chunks, 0, stats);
  } else if (cmaj_ok(l->outer, l->channels, l->inner)) {
    const bool vec = cmaj_vec_ok<T>(l->inner, x, nullptr, nullptr, nullptr);
    const CmajGeom cg = make_cmaj(l->outer, l->channels, l->inner, vec ? Vec<T>::N : 1);
    const int64_t blocks = (cg.channels * cg.chunks + kRowWarps - 1) / kRowWarps;
    if (blocks > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
    Stat4* part = reinterpret_cast<Stat4*>(ws_partials(ws));
    auto kern = vec ? stats_cmaj_kernel<T, ABS, Vec<T>::N> : stats_cmaj_kernel<T, ABS, 1>;
    kern<<<static_cast<unsigned>(blocks), kRowWarps * 32, 0, st>>>(x, cg, part);
    DLMCQ_LAUNCH_CHECK();
    stats_finalize_kernel<<<static_cast<unsigned>(cg.channels), 128, 0, st>>>(part, cg.chunks, cg.chunks, 0, stats);
  } else {
    const RowGeom gm = make_geom(l->outer, l->channels, l->inner);
    const int64_t items = gm.rows * gm.segs;
    const int64_t blocks = (items + kRowWarps - 1) / kRowWarps;
    if (blocks > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
    const int direct = (l->outer == 1 && gm.segs == 1) ? 1 : 0;
    Stat4* part = reinterpret_cast<Stat4*>(ws_partials(ws));
    stats_rows_kernel<T, ABS><<<static_cast<unsigned>(blocks), kRowWarps * 32, 0, st>>>(x, gm, stats, part, direct);
    if (!direct) {
      DLMCQ_LAUNCH_CHECK();
      stats_finalize_kernel<<<static_cast<unsigned>(gm.channels), 128, 0, st>>>(part, l->outer * gm.segs, gm.segs,
                                                                                 gm.channels * gm.segs, stats);
    }
  }
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

}  // namespace dlmcq

using namespace dlmcq;

extern "C" int dlmcq_obs_stats(const void* x, float* stats, const dlmcq_layout* layout, int flags, void* workspace,
                               size_t workspace_bytes, void* stream) {
  if (!layout || layout->outer < 1 || layout->channels < 1 || layout->inner < 1) return DLMCQ_EINVAL;
  if (!x || !stats || !workspace) return DLMCQ_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool ab = (flags & DLMCQ_STATS_ABS_INPUT) != 0;
  if (layout->dtype == DLMCQ_F32) {
    const float* p = static_cast<const float*>(x);
    return ab ? stats_launch<float, true>(p, stats, layout, workspace, workspace_bytes, st)
              : stats_launch<float, false>(p, stats, layout, workspace, workspace_bytes, st);
  }
  if (layout->dtype == DLMCQ_BF16) {
    const __nv_bfloat16* p = static_cast<const __nv_bfloat16*>(x);
    return ab ? stats_launch<__nv_bfloat16, true>(p, stats, layout, workspace, workspace_bytes, st)
              : stats_launch<__nv_bfloat16, false>(p, stats, layout, workspace, workspace_bytes, st);
  }
  return DLMCQ_EINVAL;
}

extern "C" int dlmcq_obs_minmax_finalize_mode(const float* stats, float* scale, float* offset, int64_t channels,
                                              int n_bits, int is_signed, int allow_offset, int scalar_div_mode,
                                              void* stream) {
  if (!stats || !scale || !offset || channels < 1 || n_bits < 1 || n_bits > 24) return DLMCQ_EINVAL;
  if (scalar_div_mode != DLMCQ_DIV_IEEE && scalar_div_mode != DLMCQ_DIV_CUDA_EAGER) return DLMCQ_EINVAL;
  const float qdiv = is_signed ? static_cast<float>((1 << (n_bits - 1)) - 1) : static_cast<float>((1 << n_bits) - 1);
  const int blocks = static_cast<int>((channels + 127) / 128);
  minmax_finalize_kernel<<<blocks, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      stats, scale, offset, channels, qdiv, is_signed, allow_offset, scalar_div_mode == DLMCQ_DIV_CUDA_EAGER ? 1 : 0);
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

extern "C" int dlmcq_obs_minmax_finalize(const float* stats, float* scale, float* offset, int64_t channels,
                                         int n_bits, int is_signed, int allow_offset, void* stream) {
  return dlmcq_obs_minmax_finalize_mode(stats, scale, offset, channels, n_bits, is_signed, allow_offset, DLMCQ_DIV_IEEE,
                                        stream);
}

extern "C" int dlmcq_obs_absmean_finalize(const float* stats, float* out, int64_t channels, double count,
                                          double mul_a, double mul_b, int mode, void* stream) {
  if (!stats || !out || channels < 1 || count <= 0) return DLMCQ_EINVAL;
  const int blocks = static_cast<int>((channels + 127) / 128);
  absmean_finalize_kernel<<<blocks, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      stats, out, channels, static_cast<float>(count), static_cast<float>(mul_a), static_cast<float>(mul_b), mode);
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

extern "C" int dlmcq_obs_sweep_tensor_sse(const void* x, int64_t numel, int dtype, const float* stats, int n_bits,
                                          int allow_offset, float* sse, void* workspace, size_t workspace_bytes,
                                          void* stream) {
  if (!x || !stats || !sse || !workspace || numel < 1 || n_bits < 1 || n_bits > 24) return DLMCQ_EINVAL;
  if (workspace_bytes < dlmcq_workspace_bytes(nullptr)) return DLMCQ_EWORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const float qmax = static_cast<float>((1 << n_bits) - 1);
  const int64_t tiles = (numel + kThreads * kSweepElems - 1) / (kThreads * kSweepElems);
  const int grid = stream_grid(tiles, 2);
  const size_t smem = static_cast<size_t>(kNC) * kThreads * sizeof(float);   // per-thread running sums
  cudaError_t e;
  if (dtype == DLMCQ_F32) {
    e = cudaFuncSetAttribute(sweep_tensor_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             static_cast<int>(smem));
    if (e != cudaSuccess) return set_cuda_error(e);
    sweep_tensor_kernel<float><<<grid, kThreads, smem, st>>>(static_cast<const float*>(x), numel, stats, qmax,
                                                             allow_offset, sse, workspace);
  } else if (dtype == DLMCQ_BF16) {
    e = cudaFuncSetAttribute(sweep_tensor_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             static_cast<int>(smem));
    if (e != cudaSuccess) return set_cuda_error(e);
    sweep_tensor_kernel<__nv_bfloat16><<<grid, kThreads, smem, st>>>(static_cast<const __nv_bfloat16*>(x), numel,
                                                                     stats, qmax, allow_offset, sse, workspace);
  } else {
    return DLMCQ_EINVAL;
  }
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

extern "C" int dlmcq_obs_sweep_tensor_finalize(const float* sse, const float* stats, double rows_for_mean, int n_bits,
                                               int allow_offset, float* scale, float* offset, int32_t* picked,
                                               void* stream) {
  if (!sse || !stats || !scale || !offset || rows_for_mean <= 0 || n_bits < 1 || n_bits > 24) return DLMCQ_EINVAL;
  sweep_tensor_finalize_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(
      sse, stats, static_cast<float>(rows_for_mean), static_cast<float>((1 << n_bits) - 1), allow_offset, scale,
      offset, picked);
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

extern "C" int dlmcq_obs_sweep_channel(const void* x, int64_t channels, int64_t inner, int dtype, int n_bits,
                                       int is_signed, float* scale, float* offset, void* stream) {
  return dlmcq_obs_sweep_channel_geom(x, channels, inner, dtype, n_bits, is_signed, channels, scale, offset, stream);
}

extern "C" int dlmcq_obs_sweep_channel_plan(dlmcq_sweep_item* item, int64_t geom_channels) {
  if (!item || item->channels < 1 || item->inner < 1) return DLMCQ_EINVAL;
  if (geom_channels < item->channels) geom_channels = item->channels;
  const int64_t inner = item->inner;
  // warps per row: enough warps to fill the GPU (>= 8 per SM) when the tensor has few rows - every warp of
  // a row repeats the per-candidate prologue (candidate scale, zero-point, reciprocal: ~100 instructions),
  // so more warps per row than that only add issue slots - and at least 256-512 elements per warp; fewer rows
  // per CTA when the staged rows would not fit in shared memory
  int wpr = 1;
  const int64_t want_warps = static_cast<int64_t>(num_sms()) * 8;
  // geom_channels (>= channels): the row count of the whole matrix when `x` is one rank's block of it - the
  // warps-per-row choice fixes the summation order, so a row gets the same qparams whoever sweeps it
  const int64_t min_per_warp = geom_channels <= num_sms() ? 256 : 512;   // measured: profiles/README.md
  while (wpr < kSweepWarps && geom_channels * wpr < want_warps && inner >= min_per_warp * wpr) wpr *= 2;
  const int64_t row_floats = ((inner + 8 + 3) / 4) * 4;
  while (wpr < kSweepWarps && (kSweepWarps / wpr) * row_floats > kSweepSmemFloats) wpr *= 2;
  const int staged = (kSweepWarps / wpr) * row_floats <= kSweepSmemFloats ? 1 : 0;
  const int rows_per_cta = kSweepWarps / wpr;
  item->wpr = wpr;
  item->row_floats = static_cast<int32_t>(row_floats);
  item->staged = staged;
  item->smem_bytes = staged ? static_cast<int64_t>(rows_per_cta) * row_floats * static_cast<int64_t>(sizeof(float)) : 0;
  item->ctas = (item->channels + rows_per_cta - 1) / rows_per_cta;
  return DLMCQ_OK;
}

extern "C" int dlmcq_obs_sweep_channel_grouped(const dlmcq_sweep_item* items, const int64_t* cta_prefix, int n_items,
                                               int64_t total_ctas, int dtype, int64_t smem_bytes, void* stream) {
  if (!items || !cta_prefix || n_items < 1 || total_ctas < 1 || smem_bytes < 0) return DLMCQ_EINVAL;
  if (smem_bytes > static_cast<int64_t>(kSweepSmemFloats * sizeof(float)) || total_ctas > 0x7fffffffLL)
    return DLMCQ_EUNSUPPORTED;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaError_t e;
  if (dtype == DLMCQ_F32) {
    e = cudaFuncSetAttribute(sweep_channel_grouped_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             static_cast<int>(kSweepSmemFloats * sizeof(float)));
    if (e != cudaSuccess) return set_cuda_error(e);
    sweep_channel_grouped_kernel<float><<<static_cast<unsigned>(total_ctas), kSweepWarps * 32,
                                          static_cast<size_t>(smem_bytes), st>>>(items, cta_prefix, n_items);
  } else if (dtype == DLMCQ_BF16) {
    e = cudaFuncSetAttribute(sweep_channel_grouped_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             static_cast<int>(kSweepSmemFloats * sizeof(float)));
    if (e != cudaSuccess) return set_cuda_error(e);
    sweep_channel_grouped_kernel<__nv_bfloat16><<<static_cast<unsigned>(total_ctas), kSweepWarps * 32,
                                                  static_cast<size_t>(smem_bytes), st>>>(items, cta_prefix, n_items);
  } else {
    return DLMCQ_EINVAL;
  }
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

extern "C" int dlmcq_obs_sweep_channel_geom(const void* x, int64_t channels, int64_t inner, int dtype, int n_bits,
                                            int is_signed, int64_t geom_channels, float* scale, float* offset,
                                            void* stream) {
  if (!x || !scale || !offset || channels < 1 || inner < 1 || n_bits < 1 || n_bits > 24) return DLMCQ_EINVAL;
  if (geom_channels < channels) return DLMCQ_EINVAL;
  if (dtype != DLMCQ_F32 && dtype != DLMCQ_BF16) return DLMCQ_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const float qmax = static_cast<float>((1 << n_bits) - 1);
  const float sdiv = static_cast<float>((1 << (n_bits - 1)) - 1);
  dlmcq_sweep_item plan = {};
  plan.channels = channels;
  plan.inner = inner;
  if (int e = dlmcq_obs_sweep_channel_plan(&plan, geom_channels)) return e;
  const int wpr = plan.wpr, staged = plan.staged;
  const int64_t row_floats = plan.row_floats;
  const size_t smem = static_cast<size_t>(plan.smem_bytes);
  const int64_t blocks = plan.ctas;
  if (blocks > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
  cudaError_t e;
  if (dtype == DLMCQ_F32) {
    e = cudaFuncSetAttribute(sweep_channel_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             static_cast<int>(kSweepSmemFloats * sizeof(float)));
    if (e != cudaSuccess) return set_cuda_error(e);
    sweep_channel_kernel<float><<<static_cast<unsigned>(blocks), kSweepWarps * 32, smem, st>>>(
        static_cast<const float*>(x), channels, inner, qmax, sdiv, is_signed, scale, offset, wpr,
        static_cast<int>(row_floats), staged);
  } else {
    e = cudaFuncSetAttribute(sweep_channel_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             static_cast<int>(kSweepSmemFloats * sizeof(float)));
    if (e != cudaSuccess) return set_cuda_error(e);
    sweep_channel_kernel<__nv_bfloat16><<<static_cast<unsigned>(blocks), kSweepWarps * 32, smem, st>>>(
        static_cast<const __nv_bfloat16*>(x), channels, inner, qmax, sdiv, is_signed, scale, offset, wpr,
        static_cast<int>(row_floats), staged);
  }
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

extern "C" int dlmcq_obs_l2norm_step(const void* x, int64_t channels, int64_t inner, int dtype, float* scale,
                                     const float* offset, int lo, int hi, float* diff, int32_t* done, int32_t* iters,
                                     void* workspace, size_t workspace_bytes, void* stream) {
  if (!x || !scale || !diff || !done || !workspace || channels < 1 || inner < 1) return DLMCQ_EINVAL;
  dlmcq_layout l = {1, channels, inner, dtype};
  if (workspace_bytes < dlmcq_workspace_bytes(&l)) return DLMCQ_EWORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // few long rows (per-tensor): cap the number of (row, segment) partials the single finalising CTA sums
  int64_t seg_min = kRowSegMin;
  while (channels * ((inner + seg_min - 1) / seg_min) > 8192 && seg_min < (int64_t(1) << 40)) seg_min *= 2;
  const RowGeom gm = make_geom(1, channels, inner, seg_min);
  const int64_t items = gm.rows * gm.segs;
  const int64_t blocks = (items + kRowWarps - 1) / kRowWarps;
  if (blocks > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
  float* part = ws_partials(workspace);
  const float flo = static_cast<float>(lo), fhi = static_cast<float>(hi);
  if (dtype == DLMCQ_F32)
    l2norm_rows_kernel<float><<<static_cast<unsigned>(blocks), kRowWarps * 32, 0, st>>>(
        static_cast<const float*>(x), gm, scale, offset, flo, fhi, done, part);
  else if (dtype == DLMCQ_BF16)
    l2norm_rows_kernel<__nv_bfloat16><<<static_cast<unsigned>(blocks), kRowWarps * 32, 0, st>>>(
        static_cast<const __nv_bfloat16*>(x), gm, scale, offset, flo, fhi, done, part);
  else
    return DLMCQ_EINVAL;
  DLMCQ_LAUNCH_CHECK();
  if (channels == 1) {
    l2norm_finalize_kernel<<<1, kThreads, 0, st>>>(part, gm, scale, diff, done, iters);
  } else {
    // per-CTA partial sums live behind the (row, segment) partials: 2 * items floats are used of the 4 * items
    // the workspace guarantees
    double* cta_part = reinterpret_cast<double*>(part + 2 * items);
    const unsigned fb = static_cast<unsigned>((channels + kThreads - 1) / kThreads);
    l2norm_finalize_channels_kernel<<<fb, kThreads, 0, st>>>(part, gm, scale, diff, done, iters, cta_part,
                                                            ws_counter(workspace, 1));
  }
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

extern "C" int dlmcq_obs_l2norm_resident(const void* x, int64_t channels, int64_t inner, int dtype, float* scale,
                                         const float* offset, int lo, int hi, int max_iters, float* diff,
                                         int32_t* done, int32_t* iters, void* workspace, size_t workspace_bytes,
                                         void* stream) {
  if (!x || !scale || !diff || !done || !iters || !workspace || channels < 1 || inner < 1 || max_iters < 1)
    return DLMCQ_EINVAL;
  if (dtype != DLMCQ_F32 && dtype != DLMCQ_BF16) return DLMCQ_EINVAL;
  const int64_t segs = (inner + kResSeg - 1) / kResSeg;
  const int sms = num_sms();
  int grid;
  int64_t slots;
  if (channels == 1) {                               // one row spread over the CTAs
    if (segs > static_cast<int64_t>(sms) * kResSlots) return DLMCQ_EUNSUPPORTED;
    grid = static_cast<int>(segs < sms ? segs : sms);
    slots = (segs + grid - 1) / grid;
  } else {                                           // whole rows per CTA
    if (segs > kResSlots) return DLMCQ_EUNSUPPORTED;
    grid = static_cast<int>(channels < sms ? channels : sms);
    slots = ((channels + grid - 1) / grid) * segs;
    if (slots > kResSlots) return DLMCQ_EUNSUPPORTED;                   // not resident
  }
  const size_t smem = static_cast<size_t>(slots) * kResSeg * sizeof(float);
  // workspace: [counters][cta_part: 2 parities x 2*grid doubles]
  const size_t need = kWsHeaderBytes + 4 * static_cast<size_t>(grid) * sizeof(double) + 16;
  if (workspace_bytes < need) return DLMCQ_EWORKSPACE;
  double* cta_part = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(ws_partials(workspace)) + 15) & ~uintptr_t(15));
  unsigned int* counters = ws_counter(workspace, 2);                    // [2], [3]: zero between calls
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const float flo = static_cast<float>(lo), fhi = static_cast<float>(hi);
  const int segs_i = static_cast<int>(segs);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kResWarps * 32);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;        // all CTAs co-resident: the grid barrier cannot deadlock
  attr[0].val.cooperative = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e;
  if (dtype == DLMCQ_F32) {
    e = cudaFuncSetAttribute(l2norm_resident_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             static_cast<int>(kResSlots * kResSeg * sizeof(float)));
    if (e != cudaSuccess) return set_cuda_error(e);
    e = cudaLaunchKernelEx(&cfg, l2norm_resident_kernel<float>, static_cast<const float*>(x), channels, inner, segs_i,
                           scale, offset, flo, fhi, max_iters, diff, done, iters, cta_part, counters);
  } else {
    e = cudaFuncSetAttribute(l2norm_resident_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             static_cast<int>(kResSlots * kResSeg * sizeof(float)));
    if (e != cudaSuccess) return set_cuda_error(e);
    e = cudaLaunchKernelEx(&cfg, l2norm_resident_kernel<__nv_bfloat16>, static_cast<const __nv_bfloat16*>(x), channels,
                           inner, segs_i, scale, offset, flo, fhi, max_iters, diff, done, iters, cta_part, counters);
  }
  if (e != cudaSuccess) return set_cuda_error(e);
  return DLMCQ_OK;
}
