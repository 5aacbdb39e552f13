// bnq_math.cuh - per-element arithmetic of the eval / training BatchNorm (+ identity) (+ ReLU) -> AFFINE quantizer
// chain, shared by the fused BatchNorm kernels (bnq_kernels.cu) and the code GEMM epilogue that writes the next
// layer's codes (qgemm_kernels.cu), so that both make the same rounding decisions.
#pragma once
#include "fq_math.cuh"

namespace dlmcq {

// Eval BatchNorm constants of one channel from the running buffers: invstd = RN(1 / RN(sqrt(var + eps))) (IEEE
// division and square root), the scale gamma * invstd rounded once (gamma = 1 when the layer has no weight).
__device__ __forceinline__ float bn_eval_invstd(float running_var, float eps) { return 1.0f / sqrtf(running_var + eps); }
__device__ __forceinline__ float bn_scale(float gamma, float invstd) { return gamma * invstd; }

// per-thread channel constants: VN consecutive channels
template <int VN>
struct BnCh {
  float mean[VN], a[VN], b[VN], istd[VN];
};
template <int VN>
__device__ __forceinline__ void load_bnch(BnCh<VN>& c, const float* __restrict__ gamma, const float* __restrict__ beta,
                                          const float* __restrict__ mean, const float* __restrict__ invstd, int ch0) {
#pragma unroll
  for (int e = 0; e < VN; ++e) {
    const float gm = gamma ? __ldg(gamma + ch0 + e) : 1.f;
    c.mean[e] = __ldg(mean + ch0 + e);
    c.istd[e] = __ldg(invstd + ch0 + e);
    c.a[e] = bn_scale(gm, c.istd[e]);
    c.b[e] = beta ? __ldg(beta + ch0 + e) : 0.f;
  }
}
// z = (x - mean) * (gamma * invstd) + beta  (+ identity);  act = relu(z) or z
template <int VN>
__device__ __forceinline__ void bn_act_vec(const float (&x)[VN], const BnCh<VN>& c, const float* idn, bool relu,
                                           float (&act)[VN]) {
#pragma unroll
  for (int e = 0; e < VN; ++e) {
    float z = __fmaf_rn(x[e] - c.mean[e], c.a[e], c.b[e]);
    if (idn) z = z + idn[e];
    act[e] = relu ? relu_ref(z) : z;
  }
}

// ---------------------------------------------------------------------------------------
// packed fast path shared by the apply / reduce / dx kernels.
//
// All arithmetic is issued as f32x2 instructions (FADD2 / FMUL2 / FFMA2: two IEEE-RN results per issue slot): with
// scalar code these kernels are issue-bound, not HBM-bound (measured: 30 - 57 thread-instructions per element, 0.50 -
// 0.81 of the HBM roofline; ncu summary in profiles/).  The quantizer stage is, operation for operation, the packed
// branch of fq_vec / fq_vec_bwd<FORM_AFFINE> (fq_math.cuh), so a_q stays bit-identical to the stand-alone kernel's.
// Domain: that branch needs |a - offset| <= 2^60.  The test here is on the RAW inputs and per thread iteration (one
// FMNMX per element, one branch per 16-32 elements): all |x|, |identity| <= 2^20 together with per-channel constants
// of magnitude <= 2^20 bound |a - offset| by 2^43.  Anything else (huge activations, NaN-free or not) takes the
// generic per-vector code, which carries the same guards as the stand-alone kernels.
// ---------------------------------------------------------------------------------------
constexpr float kBnqSafe = 0x1p20f;

template <int VN>
struct BnCh2 {
  float2 nmean[VN / 2], a[VN / 2], b[VN / 2], istd[VN / 2];
  bool safe;
};
template <int VN>
__device__ __forceinline__ void load_bnch2(BnCh2<VN>& c2, const BnCh<VN>& c) {
  float m = 0.f;
#pragma unroll
  for (int e = 0; e < VN; e += 2) {
    c2.nmean[e / 2] = make_float2(-c.mean[e], -c.mean[e + 1]);
    c2.a[e / 2] = make_float2(c.a[e], c.a[e + 1]);
    c2.b[e / 2] = make_float2(c.b[e], c.b[e + 1]);
    c2.istd[e / 2] = make_float2(c.istd[e], c.istd[e + 1]);
    m = fmaxf(m, fmaxf(fmaxf(fabsf(c.mean[e]), fabsf(c.mean[e + 1])), fmaxf(fabsf(c.a[e]), fabsf(c.a[e + 1]))));
    m = fmaxf(m, fmaxf(fabsf(c.b[e]), fabsf(c.b[e + 1])));
  }
  // NaN constants are ignored by fmaxf and simply flow through the fast path (as NaN data does)
  c2.safe = m <= kBnqSafe;
}

struct QuantK {
  ChanParams p;
  float2 r2, ns2, off2, noff2;
  float lo, hi;
  bool fast;
};
__device__ __forceinline__ QuantK make_quantk(const float* scale, const float* offset, float g, float lo, float hi) {
  QuantK k;
  k.p = make_params<DLMCQ_FORM_AFFINE>(scale, offset, 0, g, lo, hi);
  k.r2 = make_float2(k.p.fd.r, k.p.fd.r);
  k.ns2 = make_float2(-k.p.fd.s, -k.p.fd.s);
  k.off2 = make_float2(k.p.off, k.p.off);
  k.noff2 = make_float2(-k.p.off, -k.p.off);
  k.lo = lo;
  k.hi = hi;
  k.fast = k.p.fd.ok && fabsf(k.p.off) <= kBnqSafe;
  return k;
}

// relu as max.NaN against `floor` (0, or -inf for "no ReLU"): one instruction, NaN propagates like torch.relu
__device__ __forceinline__ float2 act_pair(float2 z, float floor) {
  return make_float2(max_nan(z.x, floor), max_nan(z.y, floor));
}
template <typename T>
__device__ __forceinline__ float2 round_to_storage(float2 v) {
  if (sizeof(T) == 2) return make_float2(to_f32<T>(from_f32<T>(v.x)), to_f32<T>(from_f32<T>(v.y)));
  return v;
}
// q = RN((act - off) / s'), c = clamp(q), cd = rint(c)   (the packed AFFINE branch of fq_vec)
__device__ __forceinline__ void quant_pair(float2 act, const QuantK& k, float2& q, float2& c, float2& cd) {
  const float2 num = __fadd2_rn(act, k.noff2);
  const float2 q0 = __fmul2_rn(num, k.r2);
  const float2 er = __ffma2_rn(k.ns2, q0, num);
  q = __ffma2_rn(er, k.r2, q0);
  c = make_float2(clamp_fast(q.x, k.lo, k.hi), clamp_fast(q.y, k.lo, k.hi));
  cd = __fadd2_rn(__fadd2_rn(c, make_float2(kRoundMagic, kRoundMagic)), make_float2(-kRoundMagic, -kRoundMagic));
}
__device__ __forceinline__ float2 dequant_pair(float2 cd, const QuantK& k) {
  // scalar mul.rn: ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into one FFMA2 (see fq_math.cuh)
  const float2 t = make_float2(__fmul_rn(cd.x, k.p.mul), __fmul_rn(cd.y, k.p.mul));
  return __fadd2_rn(t, k.off2);
}
template <int VN>
__device__ __forceinline__ float absmax_vec(const float (&f)[VN], float m) {
#pragma unroll
  for (int e = 0; e < VN; ++e) m = fmaxf(m, fabsf(f[e]));
  return m;
}

template <int VN>
__device__ __forceinline__ BnCh<VN> unpack_bnch(const BnCh2<VN>& c2) {
  BnCh<VN> c;
#pragma unroll
  for (int e = 0; e < VN; e += 2) {
    c.mean[e] = -c2.nmean[e / 2].x; c.mean[e + 1] = -c2.nmean[e / 2].y;
    c.a[e] = c2.a[e / 2].x; c.a[e + 1] = c2.a[e / 2].y;
    c.b[e] = c2.b[e / 2].x; c.b[e + 1] = c2.b[e / 2].y;
    c.istd[e] = c2.istd[e / 2].x; c.istd[e + 1] = c2.istd[e / 2].y;
  }
  return c;
}
template <int VN>
__device__ __forceinline__ void load_bnch2(BnCh2<VN>& c2, const float* __restrict__ gamma, const float* __restrict__ beta,
                                           const float* __restrict__ mean, const float* __restrict__ invstd, int ch0) {
  BnCh<VN> c;
  load_bnch<VN>(c, gamma, beta, mean, invstd, ch0);
  load_bnch2<VN>(c2, c);
}

template <typename T, int VN, bool QUANT>
__device__ __forceinline__ void apply_generic_vec(const float (&fx)[VN], const float* fi, const BnCh<VN>& c, bool relu,
                                                  const ChanParams& p, float lo, float hi, float (&act)[VN],
                                                  float (&y)[VN], float (&code)[VN]) {
  bn_act_vec<VN>(fx, c, fi, relu, act);
  if (QUANT) {
    float src[VN];
#pragma unroll
    for (int e = 0; e < VN; ++e) src[e] = sizeof(T) == 2 ? to_f32<T>(from_f32<T>(act[e])) : act[e];
    fq_vec<DLMCQ_FORM_AFFINE, VN>(src, p, lo, hi, code, y);
  }
}

}  // namespace dlmcq
