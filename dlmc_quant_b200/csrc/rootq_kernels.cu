// rootq_kernels.cu - RootQ activation / weight fake-quant, forward and root-estimator backward.
//
// Reference: dlmc/quantization/scalar/RootQ/base.py:77-156 and RootQ/function.py:5-32,58-67.
// The reference differentiates a ~25-op eager chain with autograd (about 40 launches and many
// saved N-sized tensors per layer); here forward is one pass (read w, write w_q) and backward
// is one pass (read w, dy; write dw) that also block-reduces d(upper), d(lower), d(alpha)
// (weights) or d(in_scale) (activations).  Closed forms: SURVEY.md A.5, re-derived and checked
// against autograd in fp64 (tests/test_closed_forms.py, float64 terms in tests/rootq_terms.py).
//
// The scalar prologue (EMA of the running bounds, gradient mix, delta, clamped alpha) is a
// one-thread "prepare" kernel writing a small state block: no host sync, and the in-place
// update of the running buffers (base.py:101,141-142) cannot race with the streaming kernel.
#include "fq_math.cuh"

namespace dlmcq {

constexpr int kRqUnroll = 4;

// state layout (floats)
enum { RA_SCALE = 0, RA_UPPER = 1, RA_G = 2, RA_M = 3, RA_Q = 4 };
enum { RW_U = 0, RW_L = 1, RW_DELTA = 2, RW_ALPHA = 3, RW_G = 4, RW_M = 5, RW_AMASK = 6, RW_Q = 7 };

__global__ void rootq_act_prepare_kernel(const float* in_scale, float* run_scale, float one_minus_m, float m, float g,
                                         float one_minus_g, float q, int training, float* state) {
  float rs;
  if (training) {
    // base.py:95  run.mul(1-m).add(m * in_scale);  :97  g*rs + (1-g)*rs.detach()
    rs = run_scale[0] * one_minus_m + m * in_scale[0];
    rs = g * rs + one_minus_g * rs;
    run_scale[0] = rs;                               // :101
  } else {
    rs = run_scale[0];                               // :105
  }
  state[RA_SCALE] = rs;
  state[RA_UPPER] = rs * q;                          // :99,106
  state[RA_G] = g;
  state[RA_M] = m;
  state[RA_Q] = q;
}

__global__ void rootq_wt_prepare_kernel(const float* upper, const float* lower, const float* alpha, float* run_upper,
                                        float* run_lower, float one_minus_m, float m, float g, float one_minus_g,
                                        float q, int training, float* state) {
  float U, L;
  if (training) {
    U = run_upper[0] * one_minus_m + m * upper[0];   // base.py:137
    L = run_lower[0] * one_minus_m + m * lower[0];   // :138
    U = g * U + one_minus_g * U;                     // :139
    L = g * L + one_minus_g * L;                     // :140
    run_upper[0] = U;                                // :141
    run_lower[0] = L;                                // :142
  } else {
    U = run_upper[0];
    L = run_lower[0];
  }
  const float a0 = alpha[0];
  // function.py:25-26  alpha + relu(1e-4 - alpha);  alpha - relu(alpha - 1)
  const float r1 = relu_ref(1e-4f - a0);
  const float a1 = a0 + r1;
  const float r2 = relu_ref(a1 - 1.f);
  const float a2 = a1 - r2;
  state[RW_U] = U;
  state[RW_L] = L;
  state[RW_DELTA] = (U - L) / q;                     // base.py:147
  state[RW_ALPHA] = a2;
  state[RW_G] = g;
  state[RW_M] = m;
  state[RW_AMASK] = (!(r1 > 0.f) && !(r2 > 0.f)) ? 1.f : 0.f;   // relu backward masks
  state[RW_Q] = q;
}

// ---- per-element math -------------------------------------------------------------------
// activation: function.py:15-20 clipping(x, upper, 0); base.py:109-111
__device__ __forceinline__ float rq_act_fwd(float x, float rs, float up) {
  const float x1 = x + relu_ref(0.f - x);
  const float xq = x1 - relu_ref(x1 - up);
  return round_pass(xq / rs) * rs;
}
__device__ __forceinline__ float rq_act_bwd(float x, float dy, float rs, float up, float q, float& acc) {
  const float nl = 0.f - x;
  const float x1 = x + relu_ref(nl);
  const float ov = x1 - up;
  const float xq = x1 - relu_ref(ov);
  const float v = xq / rs;
  const float I = round_pass(v);
  const bool clipped_hi = ov > 0.f;
  acc += dy * ((I - v) + (clipped_hi ? q : 0.f));
  // relu's gradient passes wherever its input is not <= 0, NaN included: a NaN x gets dx = 0 like x -> +-inf
  return ((nl <= 0.f) && (ov <= 0.f)) ? dy : 0.f;
}

// Fast path of the activation chain on vectors (same results; see fq_math.cuh for the argument):
// relu as max.NaN (the sign of a zero is erased by the following add), x/s by the hoisted reciprocal with
// residual correction, round_pass(v) == rint(v)+0 for finite v.  Out-of-domain vectors use the literal chain.
template <int N>
__device__ __forceinline__ void rq_act_fwd_vec(const float (&x)[N], float rs, float up, const FastDiv& fd,
                                               float (&y)[N]) {
  if (fd.ok) {
    float xq[N];
    float m = 0.f;
#pragma unroll
    for (int e = 0; e < N; ++e) {
      const float x1 = x[e] + max_nan(0.f - x[e], 0.f);
      xq[e] = x1 - max_nan(x1 - up, 0.f);
      m = fmaxf(m, fabsf(xq[e]));
    }
    if (m <= kFastDivMaxX) {
#pragma unroll
      for (int e = 0; e < N; ++e) y[e] = (rintf(fast_div(xq[e], fd)) + 0.f) * rs;
      return;
    }
  }
#pragma unroll
  for (int e = 0; e < N; ++e) y[e] = rq_act_fwd(x[e], rs, up);
}
template <int N>
__device__ __forceinline__ void rq_act_bwd_vec(const float (&x)[N], const float (&dy)[N], float rs, float up, float q,
                                               const FastDiv& fd, float (&dx)[N], float& acc) {
  if (fd.ok) {
    float xq[N], ov[N], nl[N];
    float m = 0.f;
#pragma unroll
    for (int e = 0; e < N; ++e) {
      nl[e] = 0.f - x[e];
      const float x1 = x[e] + max_nan(nl[e], 0.f);
      ov[e] = x1 - up;
      xq[e] = x1 - max_nan(ov[e], 0.f);
      m = fmaxf(m, fabsf(xq[e]));
    }
    if (m <= kFastDivMaxX) {
#pragma unroll
      for (int e = 0; e < N; ++e) {
        const float v = fast_div(xq[e], fd);
        const float I = rintf(v) + 0.f;
        const bool hi_clip = ov[e] > 0.f;
        acc = __fmaf_rn(dy[e], (I - v) + (hi_clip ? q : 0.f), acc);
        dx[e] = ((nl[e] <= 0.f) && (ov[e] <= 0.f)) ? dy[e] : 0.f;
      }
      return;
    }
  }
#pragma unroll
  for (int e = 0; e < N; ++e) dx[e] = rq_act_bwd(x[e], dy[e], rs, up, q, acc);
}

struct RqW {
  float U, L, delta, alpha, k, q, half_delta;
  FastDiv fd;
};
// (c - L) / delta with the hoisted reciprocal when in the fast domain (uniform divisor delta)
struct RqWDiv { FastDiv fd; };
__device__ __forceinline__ float rq_div_delta(float num, float delta, const FastDiv& fd) {
  return (fd.ok && fabsf(num) <= kFastDivMaxX) ? fast_div(num, fd) : num / delta;
}
__device__ __forceinline__ RqW load_rqw(const float* st) {
  RqW p;
  p.U = st[RW_U]; p.L = st[RW_L]; p.delta = st[RW_DELTA]; p.alpha = st[RW_ALPHA]; p.q = st[RW_Q];
  p.k = 2.f / p.delta;                               // function.py:29
  p.half_delta = p.delta * 0.5f;
  p.fd = make_fastdiv(p.delta);
  return p;
}
// The level sign of function.py:31,58, sgn(pow(b, alpha) * sg) with b = k*|z| + 1e-5, as the reference evaluates it.
// With delta > 0 (k > 0), b >= 1e-5 > 0 and the sign is sign(z), which the callers use without a pow.  With U < L
// (delta < 0) b can be negative: pow gives NaN (sgn 0) for a fractional alpha and b itself for alpha == 1.
__device__ __forceinline__ float rq_sgn(float v) { return (v > 0.f) ? 1.f : ((v < 0.f) ? -1.f : 0.f); }
__device__ __forceinline__ float rq_level_sign_literal(float z, const RqW& p) {
  const float az = fabsf(z);
  return rq_sgn(powf(p.k * az + 1e-5f, p.alpha) * (z / (az + 1e-5f)));
}
// weight forward value: base.py:146-155; torch.sgn(NaN) is 0.
__device__ __forceinline__ float rq_wt_fwd(float w, const RqW& p) {
  const float x1 = w + relu_ref(p.L - w);
  const float c = x1 - relu_ref(x1 - p.U);
  const float t = rq_div_delta(c - p.L, p.delta, p.fd);
  const float fl = floorf(t);
  const float I = (fl - t) + t;                      // floor_pass value, utils.py:34-37
  const float mi = (I + 0.5f) * p.delta + p.L;       // base.py:149
  const float z = c - mi;
  const float sig = (p.k > 0.f) ? rq_sgn(z) : rq_level_sign_literal(z, p);
  return ((sig + 1.f) / 2.f + I) * p.delta + p.L;    // function.py:63-67
}
// weight backward: returns dw, accumulates the three reduced gradients (un-chained).
__device__ __forceinline__ float rq_wt_bwd(float w, float dy, const RqW& p, float& accU, float& accL, float& accA) {
  const float lw = p.L - w;
  const float x1 = w + relu_ref(lw);
  const float ov = x1 - p.U;
  const float c = x1 - relu_ref(ov);
  const bool m_lo = lw > 0.f, m_hi = ov > 0.f;
  const float dcw = (m_lo || m_hi) ? 0.f : 1.f;
  const float cu = m_hi ? 1.f : 0.f;
  const float cl = (m_lo && !m_hi) ? 1.f : 0.f;
  const float t = rq_div_delta(c - p.L, p.delta, p.fd);
  const float fl = floorf(t);
  const float I = (fl - t) + t;
  const float mi = (I + 0.5f) * p.delta + p.L;
  const float z = c - mi;
  const float az = fabsf(z);
  const float den = az + 1e-5f;
  const float sg = z / den;
  const float b = p.k * az + 1e-5f;
  const float lb = logf(b);
  const bool kpos = p.k > 0.f;
  const float pw = kpos ? expf(p.alpha * lb) : powf(b, p.alpha);   // b^alpha (b may be negative when U < L)
  const float sgnz = rq_sgn(z);
  const float sig = kpos ? sgnz : rq_sgn(pw * sg);   // level sign, as in rq_wt_fwd
  const float pw_b = pw / b;                         // b^(alpha-1)
  const float dpdz = p.alpha * pw_b * p.k * sgnz * sg + pw * 1e-5f / (den * den);
  const float dpdd = -(p.alpha * pw_b * p.k * az * sg) / p.delta;
  const float dpda = pw * lb * sg;
  const float lvl = (sig + 1.f) * 0.5f + I;
  const float inv_q = 1.f / p.q;
  accA += dy * (p.half_delta * dpda);
  accU += dy * (p.half_delta * (dpdz * cu + dpdd * inv_q) + (cu - t * inv_q) + lvl * inv_q);
  accL += dy * (p.half_delta * (dpdz * cl - dpdd * inv_q) + (cl - 1.f + t * inv_q) - lvl * inv_q + 1.f);
  return dy * dcw * (1.f + p.half_delta * dpdz);
}

// ---- streaming kernels ----------------------------------------------------------------------
template <typename T, bool WEIGHT>
__global__ void __launch_bounds__(kThreads, 4)
rootq_fwd_kernel(const T* __restrict__ x, T* __restrict__ y, int64_t n, const float* __restrict__ state) {
  using V = Vec<T>;
  using raw = typename V::raw;
  RqW pw = {};
  float rs = 0.f, up = 0.f;
  FastDiv fd = {};
  pdl_wait();
  pdl_trigger();
  if constexpr (WEIGHT) pw = load_rqw(state);
  else { rs = state[RA_SCALE]; up = state[RA_UPPER]; fd = make_fastdiv(rs); }
  const bool vec = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15u) == 0;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  auto f = [&](float v) { return WEIGHT ? rq_wt_fwd(v, pw) : rq_act_fwd(v, rs, up); };
  if (vec) {
    const int64_t nvec = n / V::N;
    const raw* xv = reinterpret_cast<const raw*>(x);
    raw* yv = reinterpret_cast<raw*>(y);
    auto body = [&](const raw& r, int64_t idx) {
      float a[V::N], o[V::N];
      V::unpack(r, a);
      if constexpr (WEIGHT) {
#pragma unroll
        for (int e = 0; e < V::N; ++e) o[e] = f(a[e]);
      } else {
        rq_act_fwd_vec<V::N>(a, rs, up, fd, o);
      }
      st_stream(yv + idx, V::pack(o));
    };
    const int64_t tile_vecs = static_cast<int64_t>(kRqUnroll) * blockDim.x;   // contiguous 16 KB tiles
    const int64_t ntiles = nvec / tile_vecs;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
      const int64_t b = t * tile_vecs + threadIdx.x;
      raw r[kRqUnroll];
#pragma unroll
      for (int k = 0; k < kRqUnroll; ++k) r[k] = ld_stream(xv + b + k * blockDim.x);
#pragma unroll
      for (int k = 0; k < kRqUnroll; ++k) body(r[k], b + k * blockDim.x);
    }
    for (int64_t j = ntiles * tile_vecs + i; j < nvec; j += stride) body(ld_stream(xv + j), j);
    if (blockIdx.x == 0) {
      const int64_t t = nvec * V::N + threadIdx.x;
      if (t < n) y[t] = from_f32<T>(f(to_f32<T>(x[t])));
    }
  } else {
    for (; i < n; i += stride) y[i] = from_f32<T>(f(to_f32<T>(x[i])));
  }
}

template <typename T, bool WEIGHT>
__global__ void __launch_bounds__(kThreads, 3)
rootq_bwd_kernel(const T* __restrict__ x, const T* __restrict__ dy, T* __restrict__ dx, int64_t n,
                 const float* __restrict__ state, float* __restrict__ grads, void* ws) {
  using V = Vec<T>;
  using raw = typename V::raw;
  __shared__ __align__(16) float smem[192];
  RqW pw = {};
  float rs = 0.f, up = 0.f, qa = 0.f;
  FastDiv fd = {};
  pdl_wait();
  pdl_trigger();
  if constexpr (WEIGHT) pw = load_rqw(state);
  else { rs = state[RA_SCALE]; up = state[RA_UPPER]; qa = state[RA_Q]; fd = make_fastdiv(rs); }
  float acc[3] = {0.f, 0.f, 0.f};
  const bool vec = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dy) |
                     reinterpret_cast<uintptr_t>(dx)) & 15u) == 0;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  auto f = [&](float v, float g) {
    return WEIGHT ? rq_wt_bwd(v, g, pw, acc[0], acc[1], acc[2]) : rq_act_bwd(v, g, rs, up, qa, acc[0]);
  };
  if (vec) {
    const int64_t nvec = n / V::N;
    const raw* xv = reinterpret_cast<const raw*>(x);
    const raw* gv = reinterpret_cast<const raw*>(dy);
    raw* ov = reinterpret_cast<raw*>(dx);
    auto body = [&](const raw& rx, const raw& rg, int64_t idx) {
      float a[V::N], b[V::N], o[V::N];
      V::unpack(rx, a);
      V::unpack(rg, b);
      if constexpr (WEIGHT) {
#pragma unroll
        for (int e = 0; e < V::N; ++e) o[e] = f(a[e], b[e]);
      } else {
        rq_act_bwd_vec<V::N>(a, b, rs, up, qa, fd, o, acc[0]);
      }
      st_stream(ov + idx, V::pack(o));
    };
    constexpr int U = WEIGHT ? 2 : kRqUnroll;
    const int64_t tile_vecs = static_cast<int64_t>(U) * blockDim.x;
    const int64_t ntiles = nvec / tile_vecs;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
      const int64_t b = t * tile_vecs + threadIdx.x;
      raw rx[U], rg[U];
#pragma unroll
      for (int k = 0; k < U; ++k) {
        rx[k] = ld_stream(xv + b + k * blockDim.x);
        rg[k] = ld_stream(gv + b + k * blockDim.x);
      }
#pragma unroll
      for (int k = 0; k < U; ++k) body(rx[k], rg[k], b + k * blockDim.x);
    }
    for (int64_t j = ntiles * tile_vecs + i; j < nvec; j += stride) body(ld_stream(xv + j), ld_stream(gv + j), j);
    if (blockIdx.x == 0) {
      const int64_t t = nvec * V::N + threadIdx.x;
      if (t < n) dx[t] = from_f32<T>(f(to_f32<T>(x[t]), to_f32<T>(dy[t])));
    }
  } else {
    for (; i < n; i += stride) dx[i] = from_f32<T>(f(to_f32<T>(x[i]), to_f32<T>(dy[i])));
  }
  block_sum<3>(acc, smem);
  float* partials = ws_partials(ws);
  if (threadIdx.x == 0) {
    partials[3 * blockIdx.x] = acc[0];
    partials[3 * blockIdx.x + 1] = acc[1];
    partials[3 * blockIdx.x + 2] = acc[2];
  }
  if (take_last_ticket(ws_counter(ws), gridDim.x)) {
    double s[3] = {0.0, 0.0, 0.0};
    for (int b = threadIdx.x; b < static_cast<int>(gridDim.x); b += blockDim.x) {
      s[0] += partials[3 * b]; s[1] += partials[3 * b + 1]; s[2] += partials[3 * b + 2];
    }
    double* sm = reinterpret_cast<double*>(smem);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
#pragma unroll
    for (int q = 0; q < 3; ++q) s[q] = warp_sum(s[q]);
    __syncthreads();
    if (lane == 0) { sm[warp] = s[0]; sm[8 + warp] = s[1]; sm[16 + warp] = s[2]; }
    __syncthreads();
    if (threadIdx.x == 0) {
      double t[3] = {0.0, 0.0, 0.0};
      for (int w = 0; w < nwarp; ++w) { t[0] += sm[w]; t[1] += sm[8 + w]; t[2] += sm[16 + w]; }
      if (WEIGHT) {
        const float g = state[RW_G], m = state[RW_M];
        grads[0] = m * (g * static_cast<float>(t[0]));      // base.py:137,139 chain: d wt_upper
        grads[1] = m * (g * static_cast<float>(t[1]));      // d wt_lower
        grads[2] = state[RW_AMASK] * static_cast<float>(t[2]);   // d wt_alpha (function.py:25-26)
      } else {
        const float g = state[RA_G], m = state[RA_M];
        grads[0] = m * (g * static_cast<float>(t[0]));      // base.py:95,97 chain: d in_scale
      }
      *ws_counter(ws) = 0u;
    }
  }
}

// ---- grouped (multi-tensor) launches --------------------------------------------------------------
// The RootQ weight tensors of a CNN are <= 9.4 MB each and every quantizer has a scalar prologue: 21 layers
// of cifar ResNet-18 cost 126 launches per training step when run one by one.  Here ONE launch prepares all
// quantizers (activation and weight), ONE quantises all weight tensors and ONE differentiates them
// (+ a small finalisation): work units of DLMCQ_ROOTQ_UNIT elements, one warp each, located by a binary
// search over the unit prefix.  Same per-element device functions as the single-tensor kernels.
__global__ void rootq_prepare_many_kernel(const dlmcq_rootq_prep* __restrict__ items, int n_items) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_items) return;
  const dlmcq_rootq_prep it = items[k];
  const float m = static_cast<float>(it.momentum), one_minus_m = static_cast<float>(1.0 - it.momentum);
  const float g = static_cast<float>(it.g), one_minus_g = static_cast<float>(1.0 - it.g);
  const float q = static_cast<float>(it.hi - it.lo);
  if (it.is_weight) {
    float U, L;
    if (it.training) {
      U = it.run_a[0] * one_minus_m + m * it.param_a[0];   // base.py:137
      L = it.run_b[0] * one_minus_m + m * it.param_b[0];   // :138
      U = g * U + one_minus_g * U;                         // :139
      L = g * L + one_minus_g * L;                         // :140
      it.run_a[0] = U;                                     // :141
      it.run_b[0] = L;                                     // :142
    } else {
      U = it.run_a[0];
      L = it.run_b[0];
    }
    const float a0 = it.alpha[0];
    const float r1 = relu_ref(1e-4f - a0);                 // function.py:25-26
    const float a1 = a0 + r1;
    const float r2 = relu_ref(a1 - 1.f);
    it.state[RW_U] = U;
    it.state[RW_L] = L;
    it.state[RW_DELTA] = (U - L) / q;                      // base.py:147
    it.state[RW_ALPHA] = a1 - r2;
    it.state[RW_G] = g;
    it.state[RW_M] = m;
    it.state[RW_AMASK] = (!(r1 > 0.f) && !(r2 > 0.f)) ? 1.f : 0.f;
    it.state[RW_Q] = q;
  } else {
    float rs;
    if (it.training) {
      rs = it.run_a[0] * one_minus_m + m * it.param_a[0];  // base.py:95
      rs = g * rs + one_minus_g * rs;                      // :97
      it.run_a[0] = rs;                                    // :101
    } else {
      rs = it.run_a[0];                                    // :105
    }
    it.state[RA_SCALE] = rs;
    it.state[RA_UPPER] = rs * q;                           // :99,106
    it.state[RA_G] = g;
    it.state[RA_M] = m;
    it.state[RA_Q] = q;
  }
}

__device__ __forceinline__ int rq_find(const int64_t* __restrict__ prefix, int n_items, int64_t unit) {
  int lo = 0, hi = n_items;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(prefix + mid) <= unit) lo = mid; else hi = mid;
  }
  return lo;
}

template <typename T, bool WEIGHT, bool BWD>
__global__ void __launch_bounds__(kRowWarps * 32)
rootq_grouped_kernel(const dlmcq_rootq_item* __restrict__ items, const int64_t* __restrict__ prefix, int n_items,
                     int64_t total_units, float* __restrict__ partials) {
  using V = Vec<T>;
  using raw = typename V::raw;
  constexpr int U = WEIGHT ? 2 : 4;                        // 128-bit loads per tensor in flight per lane
  const int lane = threadIdx.x & 31;
  const int64_t unit = static_cast<int64_t>(blockIdx.x) * kRowWarps + (threadIdx.x >> 5);
  if (unit >= total_units) return;
  const int k = rq_find(prefix, n_items, unit);
  const dlmcq_rootq_item it = items[k];
  const int64_t beg = (unit - __ldg(prefix + k)) * DLMCQ_ROOTQ_UNIT;
  const int64_t len = (it.numel - beg) < DLMCQ_ROOTQ_UNIT ? (it.numel - beg) : DLMCQ_ROOTQ_UNIT;
  RqW pw = {};
  float rs = 0.f, up = 0.f, qa = 0.f;
  FastDiv fd = {};
  if constexpr (WEIGHT) pw = load_rqw(it.state);
  else { rs = it.state[RA_SCALE]; up = it.state[RA_UPPER]; qa = it.state[RA_Q]; fd = make_fastdiv(rs); }
  const T* xr = static_cast<const T*>(it.x) + beg;
  const T* gr = BWD ? static_cast<const T*>(it.dy) + beg : nullptr;
  T* yr = static_cast<T*>(it.y) + beg;
  float acc[3] = {0.f, 0.f, 0.f};
  int64_t done = 0;
  const bool vec = ((reinterpret_cast<uintptr_t>(xr) | reinterpret_cast<uintptr_t>(yr) |
                     reinterpret_cast<uintptr_t>(gr)) & 15u) == 0;
  if (vec) {
    const int64_t nvec = len / V::N;
    const raw* xv = reinterpret_cast<const raw*>(xr);
    const raw* gv = reinterpret_cast<const raw*>(gr);
    raw* yv = reinterpret_cast<raw*>(yr);
    for (int64_t j = lane; j < nvec; j += 32 * U) {
      raw xs[U], gs[U];
#pragma unroll
      for (int h = 0; h < U; ++h) {
        const bool in = j + 32 * h < nvec;
        xs[h] = ld_stream(xv + (in ? j + 32 * h : j));
        if (BWD) gs[h] = ld_stream(gv + (in ? j + 32 * h : j));
      }
#pragma unroll
      for (int h = 0; h < U; ++h) {
        if (j + 32 * h >= nvec) break;
        float a[V::N], b[V::N], o[V::N];
        V::unpack(xs[h], a);
        if (BWD) V::unpack(gs[h], b);
        if constexpr (WEIGHT) {
#pragma unroll
          for (int e = 0; e < V::N; ++e)
            o[e] = BWD ? rq_wt_bwd(a[e], b[e], pw, acc[0], acc[1], acc[2]) : rq_wt_fwd(a[e], pw);
        } else if constexpr (BWD) {
          rq_act_bwd_vec<V::N>(a, b, rs, up, qa, fd, o, acc[0]);
        } else {
          rq_act_fwd_vec<V::N>(a, rs, up, fd, o);
        }
        st_stream(yv + j + 32 * h, V::pack(o));
      }
    }
    done = nvec * V::N;
  }
  for (int64_t j = done + lane; j < len; j += 32) {
    const float a = to_f32<T>(xr[j]);
    float o;
    if constexpr (WEIGHT) o = BWD ? rq_wt_bwd(a, to_f32<T>(gr[j]), pw, acc[0], acc[1], acc[2]) : rq_wt_fwd(a, pw);
    else o = BWD ? rq_act_bwd(a, to_f32<T>(gr[j]), rs, up, qa, acc[0]) : rq_act_fwd(a, rs, up);
    yr[j] = from_f32<T>(o);
  }
  if (BWD) {
#pragma unroll
    for (int q = 0; q < (WEIGHT ? 3 : 1); ++q) acc[q] = warp_sum(acc[q]);
    if (lane == 0) {
      partials[3 * unit] = acc[0];
      if (WEIGHT) {
        partials[3 * unit + 1] = acc[1];
        partials[3 * unit + 2] = acc[2];
      }
    }
  }
}

// one warp per tensor: fixed-order sum (double) of its units' partials, then the chain of base.py:137-139 (weights)
// or base.py:95,97 (activations)
template <bool WEIGHT>
__global__ void __launch_bounds__(kRowWarps * 32)
rootq_grouped_finalize(const dlmcq_rootq_item* __restrict__ items, const int64_t* __restrict__ prefix, int n_items,
                       const float* __restrict__ partials) {
  const int lane = threadIdx.x & 31;
  const int k = blockIdx.x * kRowWarps + (threadIdx.x >> 5);
  if (k >= n_items) return;
  const dlmcq_rootq_item it = items[k];
  const int64_t u0 = prefix[k], u1 = prefix[k + 1];
  double t[3] = {0.0, 0.0, 0.0};
  for (int64_t u = u0 + lane; u < u1; u += 32) {
    t[0] += partials[3 * u];
    if (WEIGHT) { t[1] += partials[3 * u + 1]; t[2] += partials[3 * u + 2]; }
  }
#pragma unroll
  for (int q = 0; q < (WEIGHT ? 3 : 1); ++q) t[q] = warp_sum(t[q]);
  if (lane == 0) {
    if (WEIGHT) {
      const float g = it.state[RW_G], m = it.state[RW_M];
      it.grads[0] = m * (g * static_cast<float>(t[0]));
      it.grads[1] = m * (g * static_cast<float>(t[1]));
      it.grads[2] = it.state[RW_AMASK] * static_cast<float>(t[2]);
    } else {
      const float g = it.state[RA_G], m = it.state[RA_M];
      it.grads[0] = m * (g * static_cast<float>(t[0]));      // d in_scale
    }
  }
}

// forward: one tile per CTA; backward: capped (every CTA leaves one partial sum per reduced quantity)
static inline int rq_grid(int64_t n, int per_thread, int blocks_per_sm) {
  const int64_t tiles = (n / per_thread + kThreads * kRqUnroll - 1) / (kThreads * kRqUnroll);
  if (blocks_per_sm >= 8) return stream_grid(tiles, 1024);
  int64_t cap = n < (int64_t(1) << 25) ? 888 : 2048;
  return static_cast<int>(tiles < 1 ? 1 : (tiles < cap ? tiles : cap));
}

}  // namespace dlmcq

using namespace dlmcq;

extern "C" int dlmcq_rootq_act_prepare(const float* in_scale, float* run_scale, double momentum, double g, int lo,
                                       int hi, int training, float* state, void* stream) {
  if (!in_scale || !run_scale || !state) return DLMCQ_EINVAL;
  rootq_act_prepare_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(
      in_scale, run_scale, static_cast<float>(1.0 - momentum), static_cast<float>(momentum), static_cast<float>(g),
      static_cast<float>(1.0 - g), static_cast<float>(hi - lo), training, state);
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

extern "C" int dlmcq_rootq_wt_prepare(const float* upper, const float* lower, const float* alpha, float* run_upper,
                                      float* run_lower, double momentum, double g, int lo, int hi, int training,
                                      float* state, void* stream) {
  if (!upper || !lower || !alpha || !run_upper || !run_lower || !state) return DLMCQ_EINVAL;
  rootq_wt_prepare_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(
      upper, lower, alpha, run_upper, run_lower, static_cast<float>(1.0 - momentum), static_cast<float>(momentum),
      static_cast<float>(g), static_cast<float>(1.0 - g), static_cast<float>(hi - lo), training, state);
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

template <bool WEIGHT>
static int rootq_forward(const void* x, void* y, int64_t n, int dtype, const float* state, void* stream) {
  if (!x || !y || !state || n < 0) return DLMCQ_EINVAL;
  if (n == 0) return DLMCQ_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaError_t e;
  if (dtype == DLMCQ_F32)
    e = launch_pdl(rootq_fwd_kernel<float, WEIGHT>, dim3(rq_grid(n, 4, 8)), dim3(kThreads), 0, st,
                   static_cast<const float*>(x), static_cast<float*>(y), n, state);
  else if (dtype == DLMCQ_BF16)
    e = launch_pdl(rootq_fwd_kernel<__nv_bfloat16, WEIGHT>, dim3(rq_grid(n, 8, 8)), dim3(kThreads), 0, st,
                   static_cast<const __nv_bfloat16*>(x), static_cast<__nv_bfloat16*>(y), n, state);
  else
    return DLMCQ_EINVAL;
  if (e != cudaSuccess) return set_cuda_error(e);
  return DLMCQ_OK;
}

template <bool WEIGHT>
static int rootq_backward(const void* x, const void* dy, void* dx, float* grads, int64_t n, int dtype,
                          const float* state, void* ws, size_t ws_bytes, void* stream) {
  if (!x || !dy || !dx || !grads || !state || !ws || n < 0) return DLMCQ_EINVAL;
  if (ws_bytes < dlmcq_workspace_bytes(nullptr)) return DLMCQ_EWORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaError_t e;
  if (dtype == DLMCQ_F32)
    e = launch_pdl(rootq_bwd_kernel<float, WEIGHT>, dim3(rq_grid(n, 4, 6)), dim3(kThreads), 0, st,
                   static_cast<const float*>(x), static_cast<const float*>(dy), static_cast<float*>(dx), n, state,
                   grads, ws);
  else if (dtype == DLMCQ_BF16)
    e = launch_pdl(rootq_bwd_kernel<__nv_bfloat16, WEIGHT>, dim3(rq_grid(n, 8, 6)), dim3(kThreads), 0, st,
                   static_cast<const __nv_bfloat16*>(x), static_cast<const __nv_bfloat16*>(dy),
                   static_cast<__nv_bfloat16*>(dx), n, state, grads, ws);
  else
    return DLMCQ_EINVAL;
  if (e != cudaSuccess) return set_cuda_error(e);
  return DLMCQ_OK;
}

extern "C" int dlmcq_rootq_act_forward(const void* x, void* y, int64_t numel, int dtype, const float* state,
                                       void* stream) {
  return rootq_forward<false>(x, y, numel, dtype, state, stream);
}
extern "C" int dlmcq_rootq_wt_forward(const void* w, void* y, int64_t numel, int dtype, const float* state,
                                      void* stream) {
  return rootq_forward<true>(w, y, numel, dtype, state, stream);
}
extern "C" int dlmcq_rootq_act_backward(const void* x, const void* dy, void* dx, float* d_in_scale, int64_t numel,
                                        int dtype, const float* state, void* workspace, size_t workspace_bytes,
                                        void* stream) {
  return rootq_backward<false>(x, dy, dx, d_in_scale, numel, dtype, state, workspace, workspace_bytes, stream);
}
extern "C" int dlmcq_rootq_wt_backward(const void* w, const void* dy, void* dw, float* grads, int64_t numel, int dtype,
                                       const float* state, void* workspace, size_t workspace_bytes, void* stream) {
  return rootq_backward<true>(w, dy, dw, grads, numel, dtype, state, workspace, workspace_bytes, stream);
}

extern "C" int dlmcq_rootq_prepare_many(const dlmcq_rootq_prep* items, int n_items, void* stream) {
  if (!items || n_items < 0) return DLMCQ_EINVAL;
  if (n_items == 0) return DLMCQ_OK;
  rootq_prepare_many_kernel<<<(n_items + 63) / 64, 64, 0, static_cast<cudaStream_t>(stream)>>>(items, n_items);
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

template <bool WEIGHT, bool BWD>
static int rootq_grouped_launch(const dlmcq_rootq_item* items, const int64_t* unit_prefix, int n_items,
                                int64_t total_units, int dtype, float* partials, void* stream) {
  if (!items || !unit_prefix || (BWD && !partials) || n_items < 1 || total_units < 0) return DLMCQ_EINVAL;
  if (total_units == 0) return DLMCQ_OK;
  const int64_t blocks = (total_units + kRowWarps - 1) / kRowWarps;
  if (blocks > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == DLMCQ_F32)
    rootq_grouped_kernel<float, WEIGHT, BWD><<<static_cast<unsigned>(blocks), kRowWarps * 32, 0, st>>>(
        items, unit_prefix, n_items, total_units, partials);
  else if (dtype == DLMCQ_BF16)
    rootq_grouped_kernel<__nv_bfloat16, WEIGHT, BWD><<<static_cast<unsigned>(blocks), kRowWarps * 32, 0, st>>>(
        items, unit_prefix, n_items, total_units, partials);
  else
    return DLMCQ_EINVAL;
  DLMCQ_LAUNCH_CHECK();
  if (BWD) {
    rootq_grouped_finalize<WEIGHT><<<(n_items + kRowWarps - 1) / kRowWarps, kRowWarps * 32, 0, st>>>(
        items, unit_prefix, n_items, partials);
    DLMCQ_LAUNCH_CHECK();
  }
  return DLMCQ_OK;
}

extern "C" int dlmcq_rootq_wt_forward_grouped(const dlmcq_rootq_item* items, const int64_t* unit_prefix, int n_items,
                                              int64_t total_units, int dtype, void* stream) {
  return rootq_grouped_launch<true, false>(items, unit_prefix, n_items, total_units, dtype, nullptr, stream);
}

extern "C" int dlmcq_rootq_wt_backward_grouped(const dlmcq_rootq_item* items, const int64_t* unit_prefix, int n_items,
                                               int64_t total_units, int dtype, float* partials, void* stream) {
  return rootq_grouped_launch<true, true>(items, unit_prefix, n_items, total_units, dtype, partials, stream);
}

extern "C" int dlmcq_rootq_act_forward_grouped(const dlmcq_rootq_item* items, const int64_t* unit_prefix, int n_items,
                                               int64_t total_units, int dtype, void* stream) {
  return rootq_grouped_launch<false, false>(items, unit_prefix, n_items, total_units, dtype, nullptr, stream);
}

extern "C" int dlmcq_rootq_act_backward_grouped(const dlmcq_rootq_item* items, const int64_t* unit_prefix, int n_items,
                                                int64_t total_units, int dtype, float* partials, void* stream) {
  return rootq_grouped_launch<false, true>(items, unit_prefix, n_items, total_units, dtype, partials, stream);
}
