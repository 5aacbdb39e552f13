// fq_kernels.cu - fused fake-quant forward / backward kernels and their C-ABI entry points.
//
// Two kernel shapes cover every layout:
//   * flat   (channels == 1): each CTA streams contiguous 16 KB tiles, every thread keeps UNROLL
//            128-bit loads in flight (forward: one tile per CTA; backward: a capped grid because
//            every CTA contributes one partial sum).  Backward block-reduces the scale gradient
//            and either the last CTA to finish combines the partials in a fixed order, or they
//            are left for dlmcq_fq_finalize_many (one launch for all layers of a step).
//   * rows   (per-channel): the tensor is rows = outer*channels of length `inner`; one warp
//            owns one row segment (<= kRowSeg elements), so the channel's qparams are loaded
//            once per warp and the per-channel scale gradient is a warp-shuffle reduction.
// Roofline: HBM.  Algorithmic bytes: forward 2*sizeof(T), backward 3*sizeof(T) per element.
#include <mutex>

#include "fq_rows.cuh"

namespace dlmcq {

constexpr int kUnroll = 4;

// ---------------------------------------------------------------------------------------
// flat forward
// ---------------------------------------------------------------------------------------
// independent: the host proved that the preceding launch writes nothing this one reads (capture_check), so the
// qparams and the first tile are loaded before pdl_wait() and overlap its tail.
template <int FORM, typename T>
__global__ void __launch_bounds__(kThreads, 4)
fq_fwd_flat(const T* __restrict__ x, T* __restrict__ y, T* __restrict__ codes, int64_t n,
            const float* __restrict__ scale, const float* __restrict__ offset, float g, float lo, float hi,
            int independent) {
  using V = Vec<T>;
  using raw = typename V::raw;
  const int64_t nvec = n / V::N;
  const raw* xv = reinterpret_cast<const raw*>(x);
  const int64_t tile_vecs = static_cast<int64_t>(kUnroll) * blockDim.x;
  const int64_t ntiles = nvec / tile_vecs;
  ChanParams p;
  raw r0[kUnroll];
  const bool hoist = independent && blockIdx.x < ntiles;
  if (independent) {
    p = make_params<FORM>(scale, offset, 0, g, lo, hi);
    if (hoist) {
      const int64_t b = static_cast<int64_t>(blockIdx.x) * tile_vecs + threadIdx.x;
#pragma unroll
      for (int k = 0; k < kUnroll; ++k) r0[k] = ld_stream(xv + b + k * blockDim.x);
    }
  }
  pdl_wait();
  pdl_trigger();
  if (!independent) p = make_params<FORM>(scale, offset, 0, g, lo, hi);
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  raw* yv = reinterpret_cast<raw*>(y);
  raw* cv = reinterpret_cast<raw*>(codes);

  auto body = [&](const raw& r, int64_t idx) {
    float f[V::N], fy[V::N], fc[V::N];
    V::unpack(r, f);
    fq_vec<FORM, V::N>(f, p, lo, hi, fc, fy);
    if (y) st_stream(yv + idx, V::pack(fy));
    if (codes) st_stream(cv + idx, V::pack(fc));
  };
  // each CTA iteration covers one contiguous tile of kUnroll*256 vectors (16 KB for fp32)
  int64_t t = blockIdx.x;
  if (hoist) {
    const int64_t b = t * tile_vecs + threadIdx.x;
#pragma unroll
    for (int k = 0; k < kUnroll; ++k) body(r0[k], b + k * blockDim.x);
    t += gridDim.x;
  }
  for (; t < ntiles; t += gridDim.x) {
    const int64_t b = t * tile_vecs + threadIdx.x;
    raw r[kUnroll];
#pragma unroll
    for (int k = 0; k < kUnroll; ++k) r[k] = ld_stream(xv + b + k * blockDim.x);
#pragma unroll
    for (int k = 0; k < kUnroll; ++k) body(r[k], b + k * blockDim.x);
  }
  for (int64_t j = ntiles * tile_vecs + i; j < nvec; j += stride) body(ld_stream(xv + j), j);
  // ragged tail (< one vector)
  if (blockIdx.x == 0) {
    const int64_t t = nvec * V::N + threadIdx.x;
    if (t < n) {
      float c, v;
      fq_elem<FORM>(to_f32<T>(x[t]), p, lo, hi, c, v);
      if (y) y[t] = from_f32<T>(v);
      if (codes) codes[t] = from_f32<T>(c);
    }
  }
}

// scalar-access variant for pointers that are not 16-byte aligned (tensor views)
template <int FORM, typename T>
__global__ void __launch_bounds__(kThreads)
fq_fwd_flat_unaligned(const T* __restrict__ x, T* __restrict__ y, T* __restrict__ codes, int64_t n,
                      const float* __restrict__ scale, const float* __restrict__ offset, float g, float lo, float hi) {
  const ChanParams p = make_params<FORM>(scale, offset, 0, g, lo, hi);
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    float c, v;
    fq_elem<FORM>(to_f32<T>(x[i]), p, lo, hi, c, v);
    if (y) y[i] = from_f32<T>(v);
    if (codes) codes[i] = from_f32<T>(c);
  }
}

// ---------------------------------------------------------------------------------------
// flat backward: dx + reduced dscale (+ doffset)
// ---------------------------------------------------------------------------------------
template <int FORM>
__device__ __forceinline__ void finalize_flat(float* partials, int nblocks, float g, float* dscale, float* doffset,
                                              float* smem) {
  // fixed-order combination of the block partials in double
  double s = 0.0, o = 0.0;
  for (int b = threadIdx.x; b < nblocks; b += blockDim.x) {
    s += static_cast<double>(partials[2 * b]);
    o += static_cast<double>(partials[2 * b + 1]);
  }
  s = warp_sum(s);
  o = warp_sum(o);
  double* sm = reinterpret_cast<double*>(smem);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  __syncthreads();
  if (lane == 0) { sm[warp] = s; sm[32 + warp] = o; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double ts = 0.0, to = 0.0;
    for (int w = 0; w < nwarp; ++w) { ts += sm[w]; to += sm[32 + w]; }
    float r = static_cast<float>(ts);
    // AFFINE: chain through grad_scale (utils.py:24-27) multiplies by g; A1: FunLSQ's "* g"
    if (FORM == DLMCQ_FORM_AFFINE || FORM == DLMCQ_FORM_A1) r = r * g;
    dscale[0] = r;
    if (doffset) doffset[0] = static_cast<float>(to);
  }
}

// DEFER: leave the per-CTA partials in `ws` ([0]=#CTAs, [1]=chain factor, then (ds, doff) pairs) for
// dlmcq_fq_finalize_many instead of finalising in the last CTA - the ticket + serial finalisation costs
// ~3.4 us per launch (measured, profiles/README.md), a once-per-step batched finalisation ~4 us in total.
// independent (VECTOR only): as for fq_fwd_flat, the qparams and the first tile of x and dy are loaded before
// pdl_wait(); the partials, the ticket and every store stay behind it.
template <int FORM, typename T, bool VECTOR, bool WANT_OFF, bool DEFER>
__global__ void __launch_bounds__(kThreads, 4)
fq_bwd_flat(const T* __restrict__ x, const T* __restrict__ dy, T* __restrict__ dx, int64_t n,
            const float* __restrict__ scale, const float* __restrict__ offset, float g, float lo, float hi,
            float* __restrict__ dscale, float* __restrict__ doffset, void* ws, int independent) {
  using V = Vec<T>;
  using raw = typename V::raw;
  __shared__ __align__(16) float smem[128];
  const int64_t nvec = n / V::N;
  const raw* xv = reinterpret_cast<const raw*>(x);
  const raw* gv = reinterpret_cast<const raw*>(dy);
  const int64_t tile_vecs = static_cast<int64_t>(kUnroll) * blockDim.x;
  const int64_t ntiles = nvec / tile_vecs;
  ChanParams p;
  raw rx0[kUnroll], rg0[kUnroll];
  const bool hoist = VECTOR && independent && blockIdx.x < ntiles;
  if (VECTOR && independent) {
    p = make_params<FORM>(scale, offset, 0, g, lo, hi);
    if (hoist) {
      const int64_t b = static_cast<int64_t>(blockIdx.x) * tile_vecs + threadIdx.x;
#pragma unroll
      for (int k = 0; k < kUnroll; ++k) {
        rx0[k] = ld_stream(xv + b + k * blockDim.x);
        rg0[k] = ld_stream(gv + b + k * blockDim.x);
      }
    }
  }
  pdl_wait();
  pdl_trigger();
  if (!(VECTOR && independent)) p = make_params<FORM>(scale, offset, 0, g, lo, hi);
  float acc[2] = {0.f, 0.f};
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (VECTOR) {
    raw* ov = reinterpret_cast<raw*>(dx);
    auto body = [&](const raw& rx, const raw& rg, int64_t idx) {
      float fx[V::N], fg[V::N], fo[V::N];
      V::unpack(rx, fx);
      V::unpack(rg, fg);
      fq_vec_bwd<FORM, WANT_OFF, V::N>(fx, fg, p, lo, hi, fo, acc[0], acc[1]);
      st_stream(ov + idx, V::pack(fo));
    };
    // each CTA iteration covers one contiguous tile of kUnroll*256 vectors of x and of dy
    int64_t t = blockIdx.x;
    if (hoist) {
      const int64_t b = t * tile_vecs + threadIdx.x;
#pragma unroll
      for (int k = 0; k < kUnroll; ++k) body(rx0[k], rg0[k], b + k * blockDim.x);
      t += gridDim.x;
    }
    for (; t < ntiles; t += gridDim.x) {
      const int64_t b = t * tile_vecs + threadIdx.x;
      raw rx[kUnroll], rg[kUnroll];
#pragma unroll
      for (int k = 0; k < kUnroll; ++k) {
        rx[k] = ld_stream(xv + b + k * blockDim.x);
        rg[k] = ld_stream(gv + b + k * blockDim.x);
      }
#pragma unroll
      for (int k = 0; k < kUnroll; ++k) body(rx[k], rg[k], b + k * blockDim.x);
    }
    for (int64_t j = ntiles * tile_vecs + i; j < nvec; j += stride) body(ld_stream(xv + j), ld_stream(gv + j), j);
    if (blockIdx.x == 0) {
      const int64_t t = nvec * V::N + threadIdx.x;
      if (t < n) dx[t] = from_f32<T>(fq_elem_bwd<FORM, WANT_OFF>(to_f32<T>(x[t]), to_f32<T>(dy[t]), p, lo, hi, acc[0], acc[1]));
    }
  } else {
    for (; i < n; i += stride)
      dx[i] = from_f32<T>(fq_elem_bwd<FORM, WANT_OFF>(to_f32<T>(x[i]), to_f32<T>(dy[i]), p, lo, hi, acc[0], acc[1]));
  }
  block_sum<2>(acc, smem);
  if (DEFER) {
    float* out = static_cast<float*>(ws);
    if (threadIdx.x == 0) {
      if (blockIdx.x == 0) {
        out[0] = __int_as_float(static_cast<int>(gridDim.x));
        out[1] = (FORM == DLMCQ_FORM_AFFINE || FORM == DLMCQ_FORM_A1) ? g : 1.f;
      }
      out[2 + 2 * blockIdx.x] = acc[0];
      out[3 + 2 * blockIdx.x] = acc[1];
    }
    return;
  }
  float* partials = ws_partials(ws);
  if (threadIdx.x == 0) {
    partials[2 * blockIdx.x] = acc[0];
    partials[2 * blockIdx.x + 1] = acc[1];
  }
  if (take_last_ticket(ws_counter(ws), gridDim.x)) {
    finalize_flat<FORM>(partials, gridDim.x, g, dscale, doffset, smem);
    if (threadIdx.x == 0) *ws_counter(ws) = 0u;   // leave the workspace reusable
  }
}

// ---------------------------------------------------------------------------------------
// row kernels (per-channel qparams): one warp per row segment
// ---------------------------------------------------------------------------------------
template <int FORM, typename T>
__global__ void __launch_bounds__(kRowWarps * 32, 3)
fq_fwd_rows(const T* __restrict__ x, T* __restrict__ y, T* __restrict__ codes, RowGeom gm,
            const float* __restrict__ scale, const float* __restrict__ offset, float g, float lo, float hi) {
  const int lane = threadIdx.x & 31;
  const int64_t item = static_cast<int64_t>(blockIdx.x) * kRowWarps + (threadIdx.x >> 5);
  if (item >= gm.rows * gm.segs) return;
  const int64_t row = item / gm.segs, seg = item - row * gm.segs;
  const ChanParams p = make_params<FORM>(scale, offset, row % gm.channels, g, lo, hi);
  const int64_t beg = seg * gm.seg;
  const int64_t len = (gm.inner - beg) < gm.seg ? (gm.inner - beg) : gm.seg;
  const int64_t base = row * gm.inner + beg;
  fwd_row_segment<FORM, T, 8>(x + base, y ? y + base : nullptr, codes ? codes + base : nullptr, len, p, lo, hi, lane);
}

// Backward rows: writes dx; per-(row,segment) partials go to `part` (2 floats each) unless the
// geometry has a single partial per channel, in which case dscale is written directly.
template <int FORM, typename T>
__global__ void __launch_bounds__(kRowWarps * 32)
fq_bwd_rows(const T* __restrict__ x, const T* __restrict__ dy, T* __restrict__ dx, RowGeom gm,
            const float* __restrict__ scale, const float* __restrict__ offset, float g, float lo, float hi,
            float* __restrict__ dscale, float* __restrict__ doffset, float* __restrict__ part, int direct) {
  const int lane = threadIdx.x & 31;
  const int64_t item = static_cast<int64_t>(blockIdx.x) * kRowWarps + (threadIdx.x >> 5);
  if (item >= gm.rows * gm.segs) return;
  const int64_t row = item / gm.segs, seg = item - row * gm.segs;
  const int64_t ch = row % gm.channels;
  const ChanParams p = make_params<FORM>(scale, offset, ch, g, lo, hi);
  const int64_t beg = seg * gm.seg;
  const int64_t len = (gm.inner - beg) < gm.seg ? (gm.inner - beg) : gm.seg;
  const int64_t base = row * gm.inner + beg;
  float as = 0.f, ao = 0.f;
  bwd_row_segment<FORM, T>(x + base, dy + base, dx + base, len, p, lo, hi, lane, as, ao);
  if (lane == 0) {
    if (direct) {
      dscale[ch] = (FORM == DLMCQ_FORM_AFFINE || FORM == DLMCQ_FORM_A1) ? as * g : as;
      if (doffset) doffset[ch] = ao;
    } else {
      part[2 * item] = as;
      part[2 * item + 1] = ao;
    }
  }
}

// ---------------------------------------------------------------------------------------
// channel-major kernels: per-channel ACTIVATIONS with short rows ([B, C, HW], HW < 256, e.g. 7x7 planes).
// One warp owns (channel c, a chunk of batch indices): its qparams are resolved once, all lanes stay busy
// on the flattened (b, e) index space of that channel (rows of 49 elements would leave 23 % of a
// warp-per-row kernel idle and pay the per-row setup 1.4 M times), and the per-channel scale gradient
// stays in registers across the whole chunk.
// ---------------------------------------------------------------------------------------
// VEC = 1: scalar accesses (rows of any length / alignment).  VEC = Vec<T>::N: rows are whole, aligned 128-bit
// vectors (14x14, 8x8, 12x12 ... planes): the flattened index runs over vectors, so the index arithmetic is paid
// once per 4 (fp32) / 8 (bf16) elements and the accesses are 128-bit.
template <int FORM, typename T, bool BWD, int VEC>
__global__ void __launch_bounds__(kRowWarps * 32, 4)
fq_cmaj_kernel(const T* __restrict__ x, const T* __restrict__ dy, T* __restrict__ out, T* __restrict__ codes,
               CmajGeom gm, const float* __restrict__ scale, const float* __restrict__ offset, float g, float lo,
               float hi, float* __restrict__ dscale, float* __restrict__ part, int direct) {
  using V = Vec<T>;
  using raw = typename V::raw;
  constexpr int U = VEC == 1 ? kCmajUnroll : 4;
  const int lane = threadIdx.x & 31;
  const int64_t item = static_cast<int64_t>(blockIdx.x) * kRowWarps + (threadIdx.x >> 5);
  if (item >= gm.channels * gm.chunks) return;
  // consecutive warps own consecutive channels of the same batch chunk: the 8 warps of a CTA then read
  // adjacent rows, so the 32-byte sectors that straddle two rows are fetched once
  const int64_t j = item / gm.channels, c = item - j * gm.channels;
  const int64_t b0 = j * gm.bc;
  const int64_t nb = (gm.outer - b0) < gm.bc ? (gm.outer - b0) : gm.bc;
  const uint32_t inner = static_cast<uint32_t>(gm.inner) / VEC;          // units per row
  const uint32_t total = static_cast<uint32_t>(nb) * inner;
  const ChanParams p = make_params<FORM>(scale, offset, c, g, lo, hi);
  const uint32_t plane = static_cast<uint32_t>(gm.channels * gm.inner) / VEC;   // bc * plane < 2^31 (cmaj_ok)
  const int64_t base = (b0 * gm.channels + c) * gm.inner;
  const T* xb = x + base;
  const T* gb = BWD ? dy + base : nullptr;
  T* ob = out ? out + base : nullptr;
  T* cb = codes ? codes + base : nullptr;
  float as = 0.f, ao = 0.f;
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
      float v[U], gq[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        v[u] = ok[u] ? to_f32<T>(xb[off[u]]) : 0.f;
        if (BWD) gq[u] = ok[u] ? to_f32<T>(gb[off[u]]) : 0.f;
      }
      if (BWD) {
        float d[U];
        fq_vec_bwd<FORM, false, U>(v, gq, p, lo, hi, d, as, ao);
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (ok[u]) ob[off[u]] = from_f32<T>(d[u]);
      } else {
        float cd[U], y[U];
        fq_vec<FORM, U>(v, p, lo, hi, cd, y);
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (ok[u]) {
            if (ob) ob[off[u]] = from_f32<T>(y[u]);
            if (cb) cb[off[u]] = from_f32<T>(cd[u]);
          }
        }
      }
    } else {
      const raw* xv = reinterpret_cast<const raw*>(xb);
      const raw* gv = reinterpret_cast<const raw*>(gb);
      raw rx[U], rg[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (ok[u]) {
          rx[u] = ld_stream(xv + off[u]);
          if (BWD) rg[u] = ld_stream(gv + off[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (!ok[u]) continue;
        float f[V::N], o1[V::N], o2[V::N];
        V::unpack(rx[u], f);
        if (BWD) {
          float fg[V::N];
          V::unpack(rg[u], fg);
          fq_vec_bwd<FORM, false, V::N>(f, fg, p, lo, hi, o1, as, ao);
          st_stream(reinterpret_cast<raw*>(ob) + off[u], V::pack(o1));
        } else {
          fq_vec<FORM, V::N>(f, p, lo, hi, o2, o1);
          if (ob) st_stream(reinterpret_cast<raw*>(ob) + off[u], V::pack(o1));
          if (cb) st_stream(reinterpret_cast<raw*>(cb) + off[u], V::pack(o2));
        }
      }
    }
  }
  if (BWD) {
    as = warp_sum(as);
    if (lane == 0) {
      if (direct) dscale[c] = (FORM == DLMCQ_FORM_AFFINE || FORM == DLMCQ_FORM_A1) ? as * g : as;
      else part[c * gm.chunks + j] = as;
    }
  }
}

// ---------------------------------------------------------------------------------------
// slab kernel (forward): per-channel activations whose short rows are not whole 128-bit vectors (SlabGeom,
// common.cuh).  The backward of these layouts stays on fq_cmaj_kernel: its scalar accesses already reach 0.86 of the
// copy rate on 7x7 planes (the backward moves 12 B per element for the same index arithmetic), and a slab backward
// measured slower (per-slot accumulators + a CTA fold per channel).
// ---------------------------------------------------------------------------------------
template <int FORM, typename T>
__global__ void __launch_bounds__(kThreads, 3)
fq_slab_kernel(const T* __restrict__ x, T* __restrict__ out, T* __restrict__ codes, SlabGeom gm,
               const float* __restrict__ scale, const float* __restrict__ offset, float g, float lo, float hi) {
  using V = Vec<T>;
  using raw = typename V::raw;
  constexpr int U = kSlabUnroll;
  const int tid = threadIdx.x;
  const int r = tid / gm.W, v = tid - r * gm.W;
  if (r >= gm.R) return;
  // adjacent CTAs own adjacent channel groups of the same batch chunk: adjacent memory
  const int64_t j = blockIdx.x / gm.groups, grp = blockIdx.x - j * gm.groups;
  const int64_t b0 = j * gm.bc;
  const int64_t b1 = (gm.outer - b0) < gm.bc ? gm.outer : b0 + gm.bc;
  const int64_t col = grp * gm.W + v;                       // vector index inside one batch plane
  const raw* xv = reinterpret_cast<const raw*>(x) + col;
  raw* ov = out ? reinterpret_cast<raw*>(out) + col : nullptr;
  raw* cv = codes ? reinterpret_cast<raw*>(codes) + col : nullptr;
  ChanParams p[V::N];
#pragma unroll
  for (int k = 0; k < V::N; ++k)
    p[k] = make_params<FORM>(scale, offset, grp * gm.G + (V::N * v + k) / static_cast<int>(gm.inner), g, lo, hi);
  for (int64_t b = b0 + r; b < b1; b += static_cast<int64_t>(gm.R) * U) {
    raw rx[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t bb = b + static_cast<int64_t>(u) * gm.R;
      if (bb < b1) rx[u] = ld_stream(xv + bb * gm.plane_vecs);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t bb = b + static_cast<int64_t>(u) * gm.R;
      if (bb >= b1) break;
      float f[V::N], o1[V::N], o2[V::N];
      V::unpack(rx[u], f);
#pragma unroll
      for (int k = 0; k < V::N; ++k) fq_elem<FORM>(f[k], p[k], lo, hi, o2[k], o1[k]);
      if (ov) st_stream(ov + bb * gm.plane_vecs, V::pack(o1));
      if (cv) st_stream(cv + bb * gm.plane_vecs, V::pack(o2));
    }
  }
}

// one CTA per channel: fixed-order sum (in double) of that channel's `per` partials, WIDTH floats each, at
// part[WIDTH * ((k / inner_n) * stride_o + ch * inner_n + k % inner_n)]  (rows: k = (b, seg), inner_n = segs,
// stride_o = C * segs; channel-major: inner_n = chunks, stride_o = 0)
template <int WIDTH>
__global__ void __launch_bounds__(128)
chan_finalize(const float* __restrict__ part, int64_t per, int64_t inner_n, int64_t stride_o, float gmul,
              float* __restrict__ dscale, float* __restrict__ doffset) {
  __shared__ double sh[2][4];
  const int64_t ch = blockIdx.x;
  double s = 0.0, o = 0.0;
  for (int64_t k = threadIdx.x; k < per; k += blockDim.x) {
    const int64_t q = k / inner_n, i = k - q * inner_n;
    const int64_t item = q * stride_o + ch * inner_n + i;
    s += static_cast<double>(part[WIDTH * item]);
    if (WIDTH == 2) o += static_cast<double>(part[WIDTH * item + 1]);
  }
  s = warp_sum(s);
  o = warp_sum(o);
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s; sh[1][threadIdx.x >> 5] = o; }
  __syncthreads();
  if (threadIdx.x == 0) {
    s = (sh[0][0] + sh[0][1]) + (sh[0][2] + sh[0][3]);
    o = (sh[1][0] + sh[1][1]) + (sh[1][2] + sh[1][3]);
    dscale[ch] = static_cast<float>(s) * gmul;
    if (WIDTH == 2 && doffset) doffset[ch] = static_cast<float>(o);
  }
}

// ---------------------------------------------------------------------------------------
// dequantize (utils.py:5-6)
// ---------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kThreads)
dequant_kernel(const T* __restrict__ codes, T* __restrict__ y, int64_t n, int64_t channels, int64_t inner,
               const float* __restrict__ scale, const float* __restrict__ offset) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    const int64_t ch = channels == 1 ? 0 : (i / inner) % channels;
    const float s = __ldg(scale + ch), o = offset ? __ldg(offset + ch) : 0.f;
    y[i] = from_f32<T>(to_f32<T>(codes[i]) * s + o);
  }
}

// ---------------------------------------------------------------------------------------
// tiled per-channel kernels: per-channel ACTIVATIONS [B, C, HW] with planes that are whole, aligned 128-bit vectors
// and at least 64 vectors long.  The tensor is streamed exactly like the flat kernels - one contiguous 16 KB tile
// per CTA, four 128-bit loads in flight per thread, packed arithmetic - and only the qparams lookup differs: the
// <= kTileRows rows a tile touches have their ChanParams resolved once per CTA into shared memory.  Backward: every
// thread adds its vectors' scale-gradient terms into a private shared-memory slot per row, a warp folds each row's
// 256 slots, the per-(tile, row) partials go to the workspace and one CTA per channel combines them in a fixed
// order (deterministic).  Replaces the warp-per-row kernels on this geometry (5.4-6.0 -> 6.3+ TB/s).
// ---------------------------------------------------------------------------------------
constexpr int kTileVecs = kThreads * kUnroll;     // 1024 vectors per tile
constexpr int kTileMinVpr = 64;                   // vectors per row at least
constexpr int kTileRows = kTileVecs / kTileMinVpr + 2;

struct TileGeom {
  int64_t nvec;        // vectors in the tensor
  uint32_t vpr;        // vectors per row (inner / Vec::N)
  uint32_t channels;
  uint32_t step_rows;  // kThreads / vpr
  uint32_t step_rem;   // kThreads % vpr
};

template <typename T>
static inline bool tiled_ok(const dlmcq_layout* l, const void* a, const void* b, const void* c) {
  const int64_t vn = Vec<T>::N;
  return l->outer > 1 && l->channels > 1 && l->inner % vn == 0 && l->inner / vn >= kTileMinVpr &&
         l->inner / vn < (int64_t(1) << 31) && l->channels < (int64_t(1) << 31) && aligned16(a) && aligned16(b) &&
         aligned16(c);
}
template <typename T>
static inline TileGeom make_tile_geom(const dlmcq_layout* l) {
  TileGeom g;
  g.vpr = static_cast<uint32_t>(l->inner / Vec<T>::N);
  g.nvec = l->outer * l->channels * static_cast<int64_t>(g.vpr);
  g.channels = static_cast<uint32_t>(l->channels);
  g.step_rows = kThreads / g.vpr;
  g.step_rem = kThreads % g.vpr;
  return g;
}

template <int FORM, typename T, bool BWD>
__global__ void __launch_bounds__(kThreads, 4)
fq_tiled_chan_kernel(const T* __restrict__ x, const T* __restrict__ dy, T* __restrict__ out, T* __restrict__ codes,
                     TileGeom gm, const float* __restrict__ scale, const float* __restrict__ offset, float g, float lo,
                     float hi, float* __restrict__ part /* [tiles][kTileRows] */) {
  using V = Vec<T>;
  using raw = typename V::raw;
  __shared__ ChanParams sp[kTileRows];
  __shared__ float acc_sm[BWD ? kTileRows * kThreads : 1];
  __shared__ int64_t s_row_first;
  __shared__ uint32_t s_nrows, s_rem_first;
  const int64_t tile = blockIdx.x;
  const int64_t v_first = tile * kTileVecs;
  if (threadIdx.x == 0) {                        // the 64-bit divisions once per CTA, not once per thread
    const int64_t rf = v_first / gm.vpr;
    const int64_t v_last = (v_first + kTileVecs < gm.nvec ? v_first + kTileVecs : gm.nvec) - 1;
    s_row_first = rf;
    s_rem_first = static_cast<uint32_t>(v_first - rf * gm.vpr);
    s_nrows = static_cast<uint32_t>(v_last / gm.vpr - rf) + 1u;             // <= kTileRows
  }
  __syncthreads();
  const int nrows = static_cast<int>(s_nrows);
  if (threadIdx.x < nrows)
    sp[threadIdx.x] = make_params<FORM>(scale, offset, (s_row_first + threadIdx.x) % gm.channels, g, lo, hi);
  if (BWD) {
    for (int r = 0; r < nrows; ++r) acc_sm[r * kThreads + threadIdx.x] = 0.f;
  }
  __syncthreads();
  // local row / remainder of this thread's first vector, then +kThreads vectors per step
  const int64_t v0 = v_first + threadIdx.x;
  const uint32_t t0 = s_rem_first + threadIdx.x;                            // < vpr + kThreads
  uint32_t lr = t0 / gm.vpr;
  uint32_t rem = t0 - lr * gm.vpr;
  const raw* xv = reinterpret_cast<const raw*>(x);
  const raw* gv = reinterpret_cast<const raw*>(dy);
  raw rx[kUnroll], rg[kUnroll];
  uint32_t rows[kUnroll];
  bool ok[kUnroll];
#pragma unroll
  for (int k = 0; k < kUnroll; ++k) {
    const int64_t v = v0 + static_cast<int64_t>(k) * kThreads;
    ok[k] = v < gm.nvec;
    rows[k] = lr;
    if (ok[k]) {
      rx[k] = ld_stream(xv + v);
      if (BWD) rg[k] = ld_stream(gv + v);
    }
    lr += gm.step_rows;
    rem += gm.step_rem;
    if (rem >= gm.vpr) { rem -= gm.vpr; ++lr; }
  }
#pragma unroll
  for (int k = 0; k < kUnroll; ++k) {
    if (!ok[k]) continue;
    const int64_t v = v0 + static_cast<int64_t>(k) * kThreads;
    const ChanParams p = sp[rows[k]];
    float f[V::N], o1[V::N], o2[V::N];
    V::unpack(rx[k], f);
    if (BWD) {
      float fg[V::N], as = 0.f, ao = 0.f;
      V::unpack(rg[k], fg);
      fq_vec_bwd<FORM, false, V::N>(f, fg, p, lo, hi, o1, as, ao);
      st_stream(reinterpret_cast<raw*>(out) + v, V::pack(o1));
      acc_sm[rows[k] * kThreads + threadIdx.x] += as;
    } else {
      fq_vec<FORM, V::N>(f, p, lo, hi, o2, o1);
      if (out) st_stream(reinterpret_cast<raw*>(out) + v, V::pack(o1));
      if (codes) st_stream(reinterpret_cast<raw*>(codes) + v, V::pack(o2));
    }
  }
  if (BWD) {
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int r = warp; r < nrows; r += kThreads / 32) {
      float a = 0.f;
#pragma unroll
      for (int q = 0; q < kThreads / 32; ++q) a += acc_sm[r * kThreads + q * 32 + lane];
      a = warp_sum(a);
      if (lane == 0) part[tile * kTileRows + r] = a;
    }
  }
}

// one CTA per channel: the rows (b, ch) of that channel, each covered by 1..k consecutive tiles
__global__ void __launch_bounds__(128)
tiled_chan_finalize(const float* __restrict__ part, TileGeom gm, int64_t outer, float gmul, float* __restrict__ dscale) {
  __shared__ double sh[4];
  const int64_t ch = blockIdx.x;
  double s = 0.0;
  for (int64_t b = threadIdx.x; b < outer; b += blockDim.x) {
    const int64_t row = b * gm.channels + ch;
    const int64_t t0 = (row * gm.vpr) / kTileVecs, t1 = ((row + 1) * gm.vpr - 1) / kTileVecs;
    for (int64_t t = t0; t <= t1; ++t) {
      const int64_t row_first = (t * kTileVecs) / gm.vpr;
      s += static_cast<double>(part[t * kTileRows + (row - row_first)]);
    }
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) dscale[ch] = static_cast<float>((sh[0] + sh[1]) + (sh[2] + sh[3])) * gmul;
}

// ---------------------------------------------------------------------------------------
// host-side dispatch
// ---------------------------------------------------------------------------------------
static inline int check_layout(const dlmcq_layout* l) {
  if (!l || l->outer < 1 || l->channels < 1 || l->inner < 0) return DLMCQ_EINVAL;
  if (l->dtype != DLMCQ_F32 && l->dtype != DLMCQ_BF16) return DLMCQ_EINVAL;
  return DLMCQ_OK;
}
static inline size_t elem_size(int dtype) { return dtype == DLMCQ_F32 ? 4 : 2; }
static inline bool elem_aligned(const void* p, int dtype) {
  return p == nullptr || (reinterpret_cast<uintptr_t>(p) % elem_size(dtype)) == 0;
}
static inline RowGeom make_geom(const dlmcq_layout* l) { return make_geom(l->outer, l->channels, l->inner); }

// ---------------------------------------------------------------------------------------
// capture-time independence of consecutive flat launches.  Eagerly the host cannot know what the kernel
// before a launch writes, so every kernel waits before its first load.  During a stream capture it can: the
// capture reports the node(s) the next launch will depend on.  When that is exactly one node and it is this
// library's previous flat launch in the same capture sequence, both launches' pointers and lengths are known
// here, and if the new launch reads nothing the previous one writes, its CTAs load their qparams and first tile
// before pdl_wait() (the invariant next to pdl_wait in common.cuh makes the pairwise check sufficient).
// ---------------------------------------------------------------------------------------
struct ByteRange {
  uintptr_t beg, end;   // [beg, end)
};
struct FlatAccess {
  ByteRange rd[5], wr[6];
  int nrd = 0, nwr = 0;
  void read(const void* p, size_t bytes) {
    if (p && bytes) rd[nrd++] = {reinterpret_cast<uintptr_t>(p), reinterpret_cast<uintptr_t>(p) + bytes};
  }
  void write(const void* p, size_t bytes) {
    if (p && bytes) wr[nwr++] = {reinterpret_cast<uintptr_t>(p), reinterpret_cast<uintptr_t>(p) + bytes};
  }
};
struct CaptureLast {          // the last flat launch of one capture sequence
  unsigned long long id;
  cudaGraphNode_t node;       // nullptr: free slot
  FlatAccess acc;
};
constexpr int kCaptureSlots = 16;   // concurrent capture sequences tracked; an evicted one only loses the overlap
static std::mutex g_capture_mu;
static CaptureLast g_capture[kCaptureSlots];
static int g_capture_next = 0;
static thread_local int g_overlap_count = 0;

// the stream's capture id and its single pending dependency; false when not capturing or not exactly one
static bool capture_tip(cudaStream_t st, unsigned long long* id, cudaGraphNode_t* node) {
  cudaStreamCaptureStatus status = cudaStreamCaptureStatusNone;
  const cudaGraphNode_t* deps = nullptr;
  size_t ndeps = 0;
  if (cudaStreamGetCaptureInfo(st, &status, id, nullptr, &deps, &ndeps) != cudaSuccess) {
    (void)cudaGetLastError();   // the launch that follows reports any real problem with the stream
    return false;
  }
  if (status != cudaStreamCaptureStatusActive || ndeps != 1 || deps[0] == nullptr) return false;
  *node = deps[0];
  return true;
}

// before the launch: 1 when it may load ahead of pdl_wait(), 0 (wait first) otherwise
static int capture_check(cudaStream_t st, const FlatAccess& a) {
  unsigned long long id = 0;
  cudaGraphNode_t node = nullptr;
  if (!pdl_enabled() || !capture_tip(st, &id, &node)) return 0;
  std::lock_guard<std::mutex> lock(g_capture_mu);
  for (const CaptureLast& c : g_capture) {
    if (c.node != node || c.id != id) continue;
    for (int r = 0; r < a.nrd; ++r)
      for (int w = 0; w < c.acc.nwr; ++w)
        if (a.rd[r].beg < c.acc.wr[w].end && c.acc.wr[w].beg < a.rd[r].end) return 0;
    return 1;
  }
  return 0;
}

// after a successful launch: it is now the capture's single dependency
static void capture_record(cudaStream_t st, const FlatAccess& a, int independent) {
  unsigned long long id = 0;
  cudaGraphNode_t node = nullptr;
  if (!pdl_enabled() || !capture_tip(st, &id, &node)) return;
  if (independent) ++g_overlap_count;
  std::lock_guard<std::mutex> lock(g_capture_mu);
  CaptureLast* slot = nullptr;
  for (CaptureLast& c : g_capture)
    if (c.node != nullptr && c.id == id) slot = &c;
  if (!slot) slot = &g_capture[g_capture_next++ % kCaptureSlots];
  slot->id = id;
  slot->node = node;
  slot->acc = a;
}

template <int FORM, typename T>
static int launch_fwd(const void* x, void* y, void* codes, const dlmcq_layout* l, const dlmcq_qparams* qp,
                      cudaStream_t st) {
  const int64_t n = l->outer * l->channels * l->inner;
  if (n == 0) return DLMCQ_OK;
  const float lo = static_cast<float>(qp->lo), hi = static_cast<float>(qp->hi);
  if (l->channels == 1) {
    if (aligned16(x) && aligned16(y) && aligned16(codes)) {
      const int64_t tiles = (n / Vec<T>::N + kThreads * kUnroll - 1) / (kThreads * kUnroll);
      // One contiguous 16 KB tile per CTA (grid-stride only beyond 148*1024 CTAs): measured 6.6-6.7 TB/s on
      // 2^26..2^28 elements vs 5.9-6.0 for a persistent grid-stride grid (profiles/README.md).
      auto kern = fq_fwd_flat<FORM, T>;
      const int bps = 1024;
      const size_t bytes = static_cast<size_t>(n) * sizeof(T);
      FlatAccess acc;
      acc.read(x, bytes);
      acc.read(qp->scale, sizeof(float));
      acc.read(qp->offset, sizeof(float));
      acc.write(y, bytes);
      acc.write(codes, bytes);
      const int independent = capture_check(st, acc);
      cudaError_t e = launch_pdl(kern, dim3(stream_grid(tiles, bps)), dim3(kThreads), 0, st,
                                 static_cast<const T*>(x), static_cast<T*>(y), static_cast<T*>(codes), n, qp->scale,
                                 qp->offset, qp->g, lo, hi, independent);
      if (e != cudaSuccess) return set_cuda_error(e);
      capture_record(st, acc, independent);
    } else {
      const int64_t tiles = (n + kThreads - 1) / kThreads;
      fq_fwd_flat_unaligned<FORM, T><<<stream_grid(tiles, 8), kThreads, 0, st>>>(
          static_cast<const T*>(x), static_cast<T*>(y), static_cast<T*>(codes), n, qp->scale, qp->offset, qp->g, lo, hi);
    }
  } else if (tiled_ok<T>(l, x, y, codes)) {
    const TileGeom tg = make_tile_geom<T>(l);
    const int64_t tiles = (tg.nvec + kTileVecs - 1) / kTileVecs;
    if (tiles > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
    fq_tiled_chan_kernel<FORM, T, false><<<static_cast<unsigned>(tiles), kThreads, 0, st>>>(
        static_cast<const T*>(x), nullptr, static_cast<T*>(y), static_cast<T*>(codes), tg, qp->scale, qp->offset,
        qp->g, lo, hi, nullptr);
  } else if (slab_ok<T>(l->outer, l->channels, l->inner, x, y, codes, nullptr)) {
    const SlabGeom sg = make_slab<T>(l->outer, l->channels, l->inner);
    fq_slab_kernel<FORM, T><<<static_cast<unsigned>(sg.groups) * sg.chunks, kThreads, 0, st>>>(
        static_cast<const T*>(x), static_cast<T*>(y), static_cast<T*>(codes), sg, qp->scale, qp->offset, qp->g, lo, hi);
  } else if (cmaj_ok(l->outer, l->channels, l->inner)) {
    const bool vec = cmaj_vec_ok<T>(l->inner, x, y, codes, nullptr);
    const CmajGeom cg = make_cmaj(l->outer, l->channels, l->inner, vec ? Vec<T>::N : 1);
    const int64_t blocks = (cg.channels * cg.chunks + kRowWarps - 1) / kRowWarps;
    if (blocks > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
    auto kern = vec ? fq_cmaj_kernel<FORM, T, false, Vec<T>::N> : fq_cmaj_kernel<FORM, T, false, 1>;
    kern<<<static_cast<unsigned>(blocks), kRowWarps * 32, 0, st>>>(
        static_cast<const T*>(x), nullptr, static_cast<T*>(y), static_cast<T*>(codes), cg, qp->scale, qp->offset,
        qp->g, lo, hi, nullptr, nullptr, 0);
  } else {
    const RowGeom gm = make_geom(l);
    const int64_t items = gm.rows * gm.segs;
    const int64_t blocks = (items + kRowWarps - 1) / kRowWarps;
    if (blocks > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
    fq_fwd_rows<FORM, T><<<static_cast<unsigned>(blocks), kRowWarps * 32, 0, st>>>(
        static_cast<const T*>(x), static_cast<T*>(y), static_cast<T*>(codes), gm, qp->scale, qp->offset, qp->g, lo, hi);
  }
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

template <int FORM, typename T>
static int launch_bwd(const void* x, const void* dy, void* dx, float* dscale, float* doffset, const dlmcq_layout* l,
                      const dlmcq_qparams* qp, void* ws, size_t ws_bytes, cudaStream_t st, bool defer = false) {
  const int64_t n = l->outer * l->channels * l->inner;
  const float lo = static_cast<float>(qp->lo), hi = static_cast<float>(qp->hi);
  if (!defer && ws_bytes < dlmcq_workspace_bytes(l)) return DLMCQ_EWORKSPACE;
  if (defer && l->channels != 1) return DLMCQ_EUNSUPPORTED;
  if (l->channels == 1) {
    const bool vec = aligned16(x) && aligned16(dy) && aligned16(dx);
    const int64_t per = vec ? Vec<T>::N : 1;
    int64_t tiles = (n / per + kThreads * kUnroll - 1) / (kThreads * kUnroll);
    // CTAs = per-launch partial sums, so the grid is capped; larger tensors amortise more of them
    int64_t cap = n < (int64_t(1) << 25) ? 888 : (n < (int64_t(1) << 27) ? 2048 : 4096);
    if (cap > kMaxPartialBlocks) cap = kMaxPartialBlocks;
    const int grid = static_cast<int>(tiles < 1 ? 1 : (tiles < cap ? tiles : cap));
    auto k = vec ? (doffset ? fq_bwd_flat<FORM, T, true, true, false> : fq_bwd_flat<FORM, T, true, false, false>)
                 : (doffset ? fq_bwd_flat<FORM, T, false, true, false> : fq_bwd_flat<FORM, T, false, false, false>);
    if (defer) k = vec ? fq_bwd_flat<FORM, T, true, false, true> : fq_bwd_flat<FORM, T, false, false, true>;
    FlatAccess acc;
    if (vec) {
      const size_t bytes = static_cast<size_t>(n) * sizeof(T);
      acc.read(x, bytes);
      acc.read(dy, bytes);
      acc.read(qp->scale, sizeof(float));
      acc.read(qp->offset, sizeof(float));
      if (!defer) acc.read(ws, ws_bytes);        // ticket counter and partials
      acc.write(dx, bytes);
      acc.write(dscale, sizeof(float));
      acc.write(doffset, sizeof(float));
      acc.write(ws, defer ? (2 + 2 * static_cast<size_t>(grid)) * sizeof(float) : ws_bytes);
    }
    const int independent = vec ? capture_check(st, acc) : 0;
    cudaError_t e = launch_pdl(k, dim3(grid), dim3(kThreads), 0, st, static_cast<const T*>(x),
                               static_cast<const T*>(dy), static_cast<T*>(dx), n, qp->scale, qp->offset, qp->g, lo, hi,
                               dscale, doffset, ws, independent);
    if (e != cudaSuccess) return set_cuda_error(e);
    if (vec) capture_record(st, acc, independent);
  } else if (doffset == nullptr && n > 0 && tiled_ok<T>(l, x, dy, dx)) {
    const TileGeom tg = make_tile_geom<T>(l);
    const int64_t tiles = (tg.nvec + kTileVecs - 1) / kTileVecs;
    if (tiles > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
    fq_tiled_chan_kernel<FORM, T, true><<<static_cast<unsigned>(tiles), kThreads, 0, st>>>(
        static_cast<const T*>(x), static_cast<const T*>(dy), static_cast<T*>(dx), nullptr, tg, qp->scale, qp->offset,
        qp->g, lo, hi, ws_partials(ws));
    DLMCQ_LAUNCH_CHECK();
    const float gmul = (FORM == DLMCQ_FORM_AFFINE || FORM == DLMCQ_FORM_A1) ? qp->g : 1.f;
    tiled_chan_finalize<<<static_cast<unsigned>(l->channels), 128, 0, st>>>(ws_partials(ws), tg, l->outer, gmul, dscale);
  } else if (cmaj_ok(l->outer, l->channels, l->inner) && doffset == nullptr && n > 0) {
    const bool vec = cmaj_vec_ok<T>(l->inner, x, dy, dx, nullptr);
    const CmajGeom cg = make_cmaj(l->outer, l->channels, l->inner, vec ? Vec<T>::N : 1);
    const int64_t blocks = (cg.channels * cg.chunks + kRowWarps - 1) / kRowWarps;
    if (blocks > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
    const int direct = cg.chunks == 1 ? 1 : 0;
    auto kern = vec ? fq_cmaj_kernel<FORM, T, true, Vec<T>::N> : fq_cmaj_kernel<FORM, T, true, 1>;
    kern<<<static_cast<unsigned>(blocks), kRowWarps * 32, 0, st>>>(
        static_cast<const T*>(x), static_cast<const T*>(dy), static_cast<T*>(dx), nullptr, cg, qp->scale, qp->offset,
        qp->g, lo, hi, dscale, ws_partials(ws), direct);
    if (!direct) {
      DLMCQ_LAUNCH_CHECK();
      const float gmul = (FORM == DLMCQ_FORM_AFFINE || FORM == DLMCQ_FORM_A1) ? qp->g : 1.f;
      chan_finalize<1><<<static_cast<unsigned>(cg.channels), 128, 0, st>>>(ws_partials(ws), cg.chunks, cg.chunks, 0,
                                                                           gmul, dscale, nullptr);
    }
  } else {
    const RowGeom gm = make_geom(l);
    const int64_t items = gm.rows * gm.segs;
    const int64_t blocks = (items + kRowWarps - 1) / kRowWarps;
    if (blocks > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
    const int direct = (l->outer == 1 && gm.segs == 1) ? 1 : 0;
    if (n == 0) return DLMCQ_OK;
    fq_bwd_rows<FORM, T><<<static_cast<unsigned>(blocks), kRowWarps * 32, 0, st>>>(
        static_cast<const T*>(x), static_cast<const T*>(dy), static_cast<T*>(dx), gm, qp->scale, qp->offset, qp->g,
        lo, hi, dscale, doffset, ws_partials(ws), direct);
    if (!direct) {
      DLMCQ_LAUNCH_CHECK();
      const float gmul = (FORM == DLMCQ_FORM_AFFINE || FORM == DLMCQ_FORM_A1) ? qp->g : 1.f;
      chan_finalize<2><<<static_cast<unsigned>(gm.channels), 128, 0, st>>>(
          ws_partials(ws), l->outer * gm.segs, gm.segs, gm.channels * gm.segs, gmul, dscale, doffset);
    }
  }
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

template <typename T>
static int dispatch_fwd(const void* x, void* y, void* codes, const dlmcq_layout* l, const dlmcq_qparams* qp,
                        cudaStream_t st) {
  switch (qp->form) {
    case DLMCQ_FORM_A1: return launch_fwd<DLMCQ_FORM_A1, T>(x, y, codes, l, qp, st);
    case DLMCQ_FORM_AFFINE: return launch_fwd<DLMCQ_FORM_AFFINE, T>(x, y, codes, l, qp, st);
    case DLMCQ_FORM_ZP: return launch_fwd<DLMCQ_FORM_ZP, T>(x, y, codes, l, qp, st);
    case DLMCQ_FORM_SYM: return launch_fwd<DLMCQ_FORM_SYM, T>(x, y, codes, l, qp, st);
  }
  return DLMCQ_EINVAL;
}
template <typename T>
static int dispatch_bwd(const void* x, const void* dy, void* dx, float* ds, float* doff, const dlmcq_layout* l,
                        const dlmcq_qparams* qp, void* ws, size_t wsb, cudaStream_t st, bool defer = false) {
  switch (qp->form) {
    case DLMCQ_FORM_A1: return launch_bwd<DLMCQ_FORM_A1, T>(x, dy, dx, ds, doff, l, qp, ws, wsb, st, defer);
    case DLMCQ_FORM_AFFINE: return launch_bwd<DLMCQ_FORM_AFFINE, T>(x, dy, dx, ds, doff, l, qp, ws, wsb, st, defer);
    case DLMCQ_FORM_ZP: return launch_bwd<DLMCQ_FORM_ZP, T>(x, dy, dx, ds, doff, l, qp, ws, wsb, st, defer);
    case DLMCQ_FORM_SYM: return launch_bwd<DLMCQ_FORM_SYM, T>(x, dy, dx, ds, doff, l, qp, ws, wsb, st, defer);
  }
  return DLMCQ_EINVAL;
}

// one CTA per deferred backward call: fixed-order reduction of its per-CTA partials in double
__global__ void __launch_bounds__(kThreads)
finalize_many_kernel(const dlmcq_finalize_item* __restrict__ items, int n_items) {
  __shared__ double sm[2][kThreads / 32];
  pdl_wait();          // the partials come from the backward launches before it
  pdl_trigger();
  const dlmcq_finalize_item it = items[blockIdx.x];
  const float* p = it.partials;
  const int nblocks = __float_as_int(p[0]);
  const float gmul = p[1];
  double s = 0.0, o = 0.0;
  for (int b = threadIdx.x; b < nblocks; b += blockDim.x) {
    s += static_cast<double>(p[2 + 2 * b]);
    o += static_cast<double>(p[3 + 2 * b]);
  }
  s = warp_sum(s);
  o = warp_sum(o);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { sm[0][warp] = s; sm[1][warp] = o; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double ts = 0.0, to = 0.0;
    for (int w = 0; w < kThreads / 32; ++w) { ts += sm[0][w]; to += sm[1][w]; }
    it.dscale[0] = static_cast<float>(ts) * gmul;
    (void)to;
  }
}

}  // namespace dlmcq

using namespace dlmcq;

extern "C" size_t dlmcq_workspace_bytes(const dlmcq_layout* l) {
  // header + flat partials (always; also covers the 80-candidate sweep) + per-(row,segment) partials
  size_t bytes = kWsHeaderBytes + static_cast<size_t>(kMaxPartialBlocks) * 96 * sizeof(float);
  if (l && l->outer >= 1 && l->channels >= 1 && l->inner >= 0) {
    const RowGeom gm = make_geom(l->outer, l->channels, l->inner);
    const size_t rows_bytes = static_cast<size_t>(gm.rows * gm.segs) * 4 * sizeof(float);
    if (kWsHeaderBytes + rows_bytes > bytes) bytes = kWsHeaderBytes + rows_bytes;
    // tiled per-channel backward: one float per (16 KB tile, row of the tile); bound with the bf16 vector width
    const size_t tiles = static_cast<size_t>(l->outer * l->channels * l->inner) / (kTileVecs * 4) + 1;
    const size_t tiled_bytes = tiles * kTileRows * sizeof(float);
    if (kWsHeaderBytes + tiled_bytes > bytes) bytes = kWsHeaderBytes + tiled_bytes;
  }
  return bytes;
}

extern "C" int dlmcq_fq_forward(const void* x, void* y, void* codes, const dlmcq_layout* layout,
                                const dlmcq_qparams* qp, void* stream) {
  if (int e = check_layout(layout)) return e;
  if (layout->outer * layout->channels * layout->inner == 0) return DLMCQ_OK;   // empty tensor: nothing to do
  if (!qp || !qp->scale || !x || (!y && !codes)) return DLMCQ_EINVAL;
  if (!elem_aligned(x, layout->dtype) || !elem_aligned(y, layout->dtype) || !elem_aligned(codes, layout->dtype))
    return DLMCQ_EALIGN;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return layout->dtype == DLMCQ_F32 ? dispatch_fwd<float>(x, y, codes, layout, qp, st)
                                    : dispatch_fwd<__nv_bfloat16>(x, y, codes, layout, qp, st);
}

extern "C" int dlmcq_fq_backward(const void* x, const void* dy, void* dx, float* dscale, float* doffset,
                                 const dlmcq_layout* layout, const dlmcq_qparams* qp, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  if (int e = check_layout(layout)) return e;
  const bool empty = layout->outer * layout->channels * layout->inner == 0;
  if (!qp || !qp->scale || !dscale || !workspace || (!empty && (!x || !dy || !dx))) return DLMCQ_EINVAL;
  if (!elem_aligned(x, layout->dtype) || !elem_aligned(dy, layout->dtype) || !elem_aligned(dx, layout->dtype))
    return DLMCQ_EALIGN;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return layout->dtype == DLMCQ_F32
             ? dispatch_bwd<float>(x, dy, dx, dscale, doffset, layout, qp, workspace, workspace_bytes, st)
             : dispatch_bwd<__nv_bfloat16>(x, dy, dx, dscale, doffset, layout, qp, workspace, workspace_bytes, st);
}

extern "C" int dlmcq_dequantize(const void* codes, void* y, const dlmcq_layout* layout, const float* scale,
                                const float* offset, void* stream) {
  if (int e = check_layout(layout)) return e;
  if (!codes || !y || !scale) return DLMCQ_EINVAL;
  const int64_t n = layout->outer * layout->channels * layout->inner;
  if (n == 0) return DLMCQ_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = stream_grid((n + kThreads - 1) / kThreads, 8);
  if (layout->dtype == DLMCQ_F32)
    dequant_kernel<float><<<grid, kThreads, 0, st>>>(static_cast<const float*>(codes), static_cast<float*>(y), n,
                                                     layout->channels, layout->inner, scale, offset);
  else
    dequant_kernel<__nv_bfloat16><<<grid, kThreads, 0, st>>>(static_cast<const __nv_bfloat16*>(codes),
                                                             static_cast<__nv_bfloat16*>(y), n, layout->channels,
                                                             layout->inner, scale, offset);
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

extern "C" size_t dlmcq_fq_partials_floats(void) { return 2 + 2 * static_cast<size_t>(kMaxPartialBlocks); }

extern "C" int dlmcq_fq_backward_partials(const void* x, const void* dy, void* dx, const dlmcq_layout* layout,
                                          const dlmcq_qparams* qp, float* partials, void* stream) {
  if (int e = check_layout(layout)) return e;
  if (layout->channels != 1) return DLMCQ_EUNSUPPORTED;
  if (!qp || !qp->scale || !partials || !x || !dy || !dx) return DLMCQ_EINVAL;
  if (!elem_aligned(x, layout->dtype) || !elem_aligned(dy, layout->dtype) || !elem_aligned(dx, layout->dtype))
    return DLMCQ_EALIGN;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return layout->dtype == DLMCQ_F32
             ? dispatch_bwd<float>(x, dy, dx, nullptr, nullptr, layout, qp, partials, 0, st, true)
             : dispatch_bwd<__nv_bfloat16>(x, dy, dx, nullptr, nullptr, layout, qp, partials, 0, st, true);
}

extern "C" int dlmcq_capture_overlap_count(void) {
  const int n = g_overlap_count;
  g_overlap_count = 0;
  return n;
}

extern "C" int dlmcq_fq_finalize_many(const dlmcq_finalize_item* items, int n_items, void* stream) {
  if (!items || n_items < 0) return DLMCQ_EINVAL;
  if (n_items == 0) return DLMCQ_OK;
  cudaError_t e = launch_pdl(finalize_many_kernel, dim3(n_items), dim3(kThreads), 0, static_cast<cudaStream_t>(stream),
                             items, n_items);
  if (e != cudaSuccess) return set_cuda_error(e);
  return DLMCQ_OK;
}
