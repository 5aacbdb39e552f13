// adaround_kernels.cu - AdaRound soft/hard rounding of per-channel weights.
//
// Reference: dlmc/quantization/scalar/FSPTQuant/base.py:69-79 (init_alpha, get_soft_targets),
// :136-141 (floor + soft target / hard target), :151-152 (clamp, * scale).  torch.floor has no
// straight-through here, so the weight gradient is identically zero; the scale gradient comes
// only through the final `* scale`, and alpha receives dy * scale * in * h'(alpha).
// Weight tensors are small (<= 2.4 M elements): one warp per row segment, scalar accesses.
#include "fq_math.cuh"

namespace dlmcq {

constexpr float kZetaMinusGamma = 1.2f;   // zeta - gamma = 1.1 - (-0.1), as fp32
constexpr float kGamma = -0.1f;

__device__ __forceinline__ float sigmoid_ref(float a) { return 1.f / (1.f + expf(-a)); }
__device__ __forceinline__ float soft_target(float a, float& pre) {
  pre = sigmoid_ref(a) * kZetaMinusGamma + kGamma;        // base.py:79
  return clamp_ref(pre, 0.f, 1.f);
}

template <typename T>
__global__ void __launch_bounds__(kRowWarps * 32)
adaround_fwd_kernel(const T* __restrict__ w, const T* __restrict__ alpha, T* __restrict__ y, RowGeom gm,
                    const float* __restrict__ scale, float lo, float hi, int soft) {
  const int lane = threadIdx.x & 31;
  const int64_t item = static_cast<int64_t>(blockIdx.x) * kRowWarps + (threadIdx.x >> 5);
  if (item >= gm.rows * gm.segs) return;
  const int64_t row = item / gm.segs, seg = item - row * gm.segs;
  const float s = __ldg(scale + row % gm.channels);
  const int64_t beg = row * gm.inner + seg * gm.seg;
  const int64_t len = (gm.inner - seg * gm.seg) < gm.seg ? (gm.inner - seg * gm.seg) : gm.seg;
  for (int64_t j = lane; j < len; j += 32) {
    const float a = to_f32<T>(alpha[beg + j]);
    float pre;
    const float h = soft ? soft_target(a, pre) : ((a >= 0.f) ? 1.f : 0.f);   // base.py:139,141
    const float q = floorf(to_f32<T>(w[beg + j]) / s) + h;                   // base.py:137
    y[beg + j] = from_f32<T>(clamp_ref(q, lo, hi) * s);                      // base.py:151-152
  }
}

template <typename T>
__global__ void __launch_bounds__(kRowWarps * 32)
adaround_bwd_kernel(const T* __restrict__ w, const T* __restrict__ alpha, const T* __restrict__ dy,
                    T* __restrict__ dalpha, RowGeom gm, const float* __restrict__ scale, float lo, float hi,
                    float* __restrict__ dscale, float* __restrict__ part, int direct) {
  const int lane = threadIdx.x & 31;
  const int64_t item = static_cast<int64_t>(blockIdx.x) * kRowWarps + (threadIdx.x >> 5);
  if (item >= gm.rows * gm.segs) return;
  const int64_t row = item / gm.segs, seg = item - row * gm.segs;
  const int64_t ch = row % gm.channels;
  const float s = __ldg(scale + ch);
  const int64_t beg = row * gm.inner + seg * gm.seg;
  const int64_t len = (gm.inner - seg * gm.seg) < gm.seg ? (gm.inner - seg * gm.seg) : gm.seg;
  float acc = 0.f;
  for (int64_t j = lane; j < len; j += 32) {
    const float a = to_f32<T>(alpha[beg + j]);
    const float g = to_f32<T>(dy[beg + j]);
    float pre;
    const float h = soft_target(a, pre);
    const float q = floorf(to_f32<T>(w[beg + j]) / s) + h;
    const float qc = clamp_ref(q, lo, hi);
    acc += g * qc;                                              // d/ds of (qc * s)
    const bool in_q = (q >= lo) && (q <= hi);                   // clamp backward, inclusive
    const bool in_h = (pre >= 0.f) && (pre <= 1.f);
    const float sg = sigmoid_ref(a);
    // the masks zero the incoming gradient, not the result: sigmoid's backward still multiplies it by
    // (1 - sg) * sg, so a NaN alpha gives a NaN d alpha, as autograd of the reference chain does
    const float gm = (in_q && in_h) ? (g * s) * kZetaMinusGamma : 0.f;
    const float d = gm * ((1.f - sg) * sg);
    dalpha[beg + j] = from_f32<T>(d);
  }
  acc = warp_sum(acc);
  if (lane == 0) {
    if (direct) dscale[ch] = acc;
    else { part[2 * item] = acc; part[2 * item + 1] = 0.f; }
  }
}

__global__ void __launch_bounds__(kRowWarps * 32)
adaround_finalize(const float* __restrict__ part, RowGeom gm, int64_t outer, float* __restrict__ dscale) {
  const int lane = threadIdx.x & 31;
  const int64_t ch = static_cast<int64_t>(blockIdx.x) * kRowWarps + (threadIdx.x >> 5);
  if (ch >= gm.channels) return;
  double s = 0.0;
  const int64_t per = outer * gm.segs;
  for (int64_t k = lane; k < per; k += 32) {
    const int64_t b = k / gm.segs, sg = k - b * gm.segs;
    s += static_cast<double>(part[2 * ((b * gm.channels + ch) * gm.segs + sg)]);
  }
  s = warp_sum(s);
  if (lane == 0) dscale[ch] = static_cast<float>(s);
}

// base.py:73-76: alpha = -log((zeta-gamma)/(rest-gamma) - 1), rest = w/s - floor(w/s)
template <typename T>
__global__ void __launch_bounds__(kThreads)
adaround_init_kernel(const T* __restrict__ w, T* __restrict__ alpha, int64_t n, int64_t channels, int64_t inner,
                     const float* __restrict__ scale) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float s = __ldg(scale + (channels == 1 ? 0 : (i / inner) % channels));
    const float v = to_f32<T>(w[i]) / s;
    const float rest = v - floorf(v);
    alpha[i] = from_f32<T>(-logf(kZetaMinusGamma / (rest - kGamma) - 1.f));
  }
}

template <typename T>
static int ada_fwd(const void* w, const void* alpha, void* y, const dlmcq_layout* l, const float* scale, int lo, int hi,
                   int soft, cudaStream_t st) {
  const RowGeom gm = make_geom(l->outer, l->channels, l->inner);
  const int64_t blocks = (gm.rows * gm.segs + kRowWarps - 1) / kRowWarps;
  if (blocks > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
  adaround_fwd_kernel<T><<<static_cast<unsigned>(blocks), kRowWarps * 32, 0, st>>>(
      static_cast<const T*>(w), static_cast<const T*>(alpha), static_cast<T*>(y), gm, scale, static_cast<float>(lo),
      static_cast<float>(hi), soft);
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

template <typename T>
static int ada_bwd(const void* w, const void* alpha, const void* dy, void* dalpha, float* dscale, const dlmcq_layout* l,
                   const float* scale, int lo, int hi, void* ws, cudaStream_t st) {
  const RowGeom gm = make_geom(l->outer, l->channels, l->inner);
  const int64_t blocks = (gm.rows * gm.segs + kRowWarps - 1) / kRowWarps;
  if (blocks > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
  const int direct = (l->outer == 1 && gm.segs == 1) ? 1 : 0;
  adaround_bwd_kernel<T><<<static_cast<unsigned>(blocks), kRowWarps * 32, 0, st>>>(
      static_cast<const T*>(w), static_cast<const T*>(alpha), static_cast<const T*>(dy), static_cast<T*>(dalpha), gm,
      scale, static_cast<float>(lo), static_cast<float>(hi), dscale, ws_partials(ws), direct);
  DLMCQ_LAUNCH_CHECK();
  if (!direct) {
    const int64_t fb = (gm.channels + kRowWarps - 1) / kRowWarps;
    adaround_finalize<<<static_cast<unsigned>(fb), kRowWarps * 32, 0, st>>>(ws_partials(ws), gm, l->outer, dscale);
    DLMCQ_LAUNCH_CHECK();
  }
  return DLMCQ_OK;
}

}  // namespace dlmcq

using namespace dlmcq;

static inline bool ada_layout_ok(const dlmcq_layout* l) {
  return l && l->outer >= 1 && l->channels >= 1 && l->inner >= 1 && (l->dtype == DLMCQ_F32 || l->dtype == DLMCQ_BF16);
}

extern "C" int dlmcq_adaround_forward(const void* w, const void* alpha, void* y, const dlmcq_layout* layout,
                                      const float* scale, int lo, int hi, int soft, void* stream) {
  if (!ada_layout_ok(layout) || !w || !alpha || !y || !scale) return DLMCQ_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return layout->dtype == DLMCQ_F32 ? ada_fwd<float>(w, alpha, y, layout, scale, lo, hi, soft, st)
                                    : ada_fwd<__nv_bfloat16>(w, alpha, y, layout, scale, lo, hi, soft, st);
}

extern "C" int dlmcq_adaround_backward(const void* w, const void* alpha, const void* dy, void* dalpha, float* dscale,
                                       const dlmcq_layout* layout, const float* scale, int lo, int hi, void* workspace,
                                       size_t workspace_bytes, void* stream) {
  if (!ada_layout_ok(layout) || !w || !alpha || !dy || !dalpha || !dscale || !scale || !workspace) return DLMCQ_EINVAL;
  if (workspace_bytes < dlmcq_workspace_bytes(layout)) return DLMCQ_EWORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return layout->dtype == DLMCQ_F32
             ? ada_bwd<float>(w, alpha, dy, dalpha, dscale, layout, scale, lo, hi, workspace, st)
             : ada_bwd<__nv_bfloat16>(w, alpha, dy, dalpha, dscale, layout, scale, lo, hi, workspace, st);
}

extern "C" int dlmcq_adaround_init_alpha(const void* w, void* alpha, const dlmcq_layout* layout, const float* scale,
                                         void* stream) {
  if (!ada_layout_ok(layout) || !w || !alpha || !scale) return DLMCQ_EINVAL;
  const int64_t n = layout->outer * layout->channels * layout->inner;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = stream_grid((n + kThreads - 1) / kThreads, 8);
  if (layout->dtype == DLMCQ_F32)
    adaround_init_kernel<float><<<grid, kThreads, 0, st>>>(static_cast<const float*>(w), static_cast<float*>(alpha), n,
                                                           layout->channels, layout->inner, scale);
  else
    adaround_init_kernel<__nv_bfloat16><<<grid, kThreads, 0, st>>>(static_cast<const __nv_bfloat16*>(w),
                                                                   static_cast<__nv_bfloat16*>(alpha), n,
                                                                   layout->channels, layout->inner, scale);
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}
