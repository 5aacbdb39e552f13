// codes.cuh - the one-byte operand encoding of the integer-code GEMM (include/dlmcq.h, DLMCQ_QGEMM_*), shared by the
// stand-alone code pass (qgemm_kernels.cu) and the fused BatchNorm producer that writes codes (bnq_kernels.cu), so
// that both emit the same byte for the same code.
#pragma once
#include <cuda_fp8.h>

#include "common.cuh"

namespace dlmcq {

// code (an integer-valued float from the quantizer, or NaN) -> its byte in the low 8 bits
template <int ENC>
__device__ __forceinline__ uint32_t code_byte(float code) {
  if (ENC == DLMCQ_QGEMM_E4M3)                                   // exact: the caller guarantees |code| <= 16
    return static_cast<uint32_t>(__nv_cvt_float_to_fp8(code == code ? code : 0.f, __NV_SATFINITE, __NV_E4M3));
  const int c = (code == code) ? static_cast<int>(code) : 0;     // NaN code -> 0 (as dlmcq_export_codes)
  return static_cast<uint32_t>(c) & 0xFFu;
}

// the same byte, the encoding chosen at run time (the code GEMM epilogue: one kernel serves both consumer encodings)
__device__ __forceinline__ uint32_t code_byte_rt(float code, int encoding) {
  return encoding == DLMCQ_QGEMM_E4M3 ? code_byte<DLMCQ_QGEMM_E4M3>(code) : code_byte<DLMCQ_QGEMM_I8>(code);
}

// Can `encoding` hold every code of [qp->lo, qp->hi]?  DLMCQ_EINVAL for an unknown encoding.
inline int code_range_ok(const dlmcq_qparams* qp, int encoding) {
  if (encoding == DLMCQ_QGEMM_E4M3) return (qp->lo >= -16 && qp->hi <= 16) ? DLMCQ_OK : DLMCQ_EUNSUPPORTED;
  if (encoding != DLMCQ_QGEMM_I8) return DLMCQ_EINVAL;
  if (qp->lo < -128 || qp->hi > 255 || (qp->lo < 0 && qp->hi > 127)) return DLMCQ_EUNSUPPORTED;
  return DLMCQ_OK;
}

}  // namespace dlmcq
