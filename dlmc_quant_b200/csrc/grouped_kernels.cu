// grouped_kernels.cu - multi-tensor fake-quant: every weight tensor of a model in ONE launch.
//
// The weight tensors of a CNN are 0.1 KB ... 9.4 MB each; quantised one by one (54 tensors for
// ResNet-50, forward and backward) the work is pure launch latency on a B200.  Here a device
// table describes all tensors; work units (row segments of <= DLMCQ_GROUP_SEG elements) are laid
// out back to back and each warp finds its tensor with a binary search over the unit prefix.
// Reference loop being replaced: one QBase/FSPTQBase.forward weight branch per layer
// (modules/base.py:131-133, FSPTQuant/base.py:149-152) and its autograd.
#include "fq_rows.cuh"

namespace dlmcq {

__device__ __forceinline__ int find_item(const int64_t* __restrict__ prefix, int n_items, int64_t unit) {
  int lo = 0, hi = n_items;          // prefix[lo] <= unit < prefix[hi]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(prefix + mid) <= unit) lo = mid; else hi = mid;
  }
  return lo;
}

template <int FORM>
__device__ __forceinline__ ChanParams item_params(const dlmcq_group_item& it, int64_t ch) {
  return make_params<FORM>(it.scale, it.offset, ch, it.g, static_cast<float>(it.lo), static_cast<float>(it.hi));
}

template <typename T>
__global__ void __launch_bounds__(kRowWarps * 32)
grouped_fwd_kernel(const dlmcq_group_item* __restrict__ items, const int64_t* __restrict__ prefix, int n_items,
                   int64_t total_units) {
  pdl_wait();          // the inputs and the device table: written by earlier work the host cannot see
  pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int64_t unit = static_cast<int64_t>(blockIdx.x) * kRowWarps + (threadIdx.x >> 5);
  if (unit >= total_units) return;
  const int k = find_item(prefix, n_items, unit);
  const dlmcq_group_item it = items[k];
  const int64_t local = unit - __ldg(prefix + k);
  const int64_t segs = (it.inner + DLMCQ_GROUP_SEG - 1) / DLMCQ_GROUP_SEG;
  const int64_t row = local / segs, seg = local - row * segs;
  const int64_t beg = seg * DLMCQ_GROUP_SEG;
  const int64_t len = (it.inner - beg) < DLMCQ_GROUP_SEG ? (it.inner - beg) : DLMCQ_GROUP_SEG;
  const T* xr = static_cast<const T*>(it.x) + row * it.inner + beg;
  T* yr = static_cast<T*>(it.y) + row * it.inner + beg;
  const float lo = static_cast<float>(it.lo), hi = static_cast<float>(it.hi);
  switch (it.form) {
    case DLMCQ_FORM_A1: fwd_row_segment<DLMCQ_FORM_A1, T>(xr, yr, nullptr, len, item_params<DLMCQ_FORM_A1>(it, row), lo, hi, lane); break;
    case DLMCQ_FORM_AFFINE: fwd_row_segment<DLMCQ_FORM_AFFINE, T>(xr, yr, nullptr, len, item_params<DLMCQ_FORM_AFFINE>(it, row), lo, hi, lane); break;
    case DLMCQ_FORM_ZP: fwd_row_segment<DLMCQ_FORM_ZP, T>(xr, yr, nullptr, len, item_params<DLMCQ_FORM_ZP>(it, row), lo, hi, lane); break;
    default: fwd_row_segment<DLMCQ_FORM_SYM, T>(xr, yr, nullptr, len, item_params<DLMCQ_FORM_SYM>(it, row), lo, hi, lane); break;
  }
}

template <typename T>
__global__ void __launch_bounds__(kRowWarps * 32)
grouped_bwd_kernel(const dlmcq_group_item* __restrict__ items, const int64_t* __restrict__ prefix, int n_items,
                   int64_t total_units, float* __restrict__ partials) {
  pdl_wait();
  pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int64_t unit = static_cast<int64_t>(blockIdx.x) * kRowWarps + (threadIdx.x >> 5);
  if (unit >= total_units) return;
  const int k = find_item(prefix, n_items, unit);
  const dlmcq_group_item it = items[k];
  const int64_t local = unit - __ldg(prefix + k);
  const int64_t segs = (it.inner + DLMCQ_GROUP_SEG - 1) / DLMCQ_GROUP_SEG;
  const int64_t row = local / segs, seg = local - row * segs;
  const int64_t beg = seg * DLMCQ_GROUP_SEG;
  const int64_t len = (it.inner - beg) < DLMCQ_GROUP_SEG ? (it.inner - beg) : DLMCQ_GROUP_SEG;
  const int64_t base = row * it.inner + beg;
  const T* xr = static_cast<const T*>(it.x) + base;
  const T* gr = static_cast<const T*>(it.dy) + base;
  T* dr = static_cast<T*>(it.y) + base;
  const float lo = static_cast<float>(it.lo), hi = static_cast<float>(it.hi);
  float as = 0.f, ao = 0.f;
  switch (it.form) {
    case DLMCQ_FORM_A1: bwd_row_segment<DLMCQ_FORM_A1, T>(xr, gr, dr, len, item_params<DLMCQ_FORM_A1>(it, row), lo, hi, lane, as, ao); break;
    case DLMCQ_FORM_AFFINE: bwd_row_segment<DLMCQ_FORM_AFFINE, T>(xr, gr, dr, len, item_params<DLMCQ_FORM_AFFINE>(it, row), lo, hi, lane, as, ao); break;
    case DLMCQ_FORM_ZP: bwd_row_segment<DLMCQ_FORM_ZP, T>(xr, gr, dr, len, item_params<DLMCQ_FORM_ZP>(it, row), lo, hi, lane, as, ao); break;
    default: bwd_row_segment<DLMCQ_FORM_SYM, T>(xr, gr, dr, len, item_params<DLMCQ_FORM_SYM>(it, row), lo, hi, lane, as, ao); break;
  }
  if (lane == 0) partials[unit] = as;
}

// one warp per (tensor, channel): add the segment partials of that row in a fixed order
__global__ void __launch_bounds__(kRowWarps * 32)
grouped_finalize_kernel(const dlmcq_group_item* __restrict__ items, const int64_t* __restrict__ prefix,
                        const int64_t* __restrict__ chan_prefix, int n_items, int64_t total_channels,
                        const float* __restrict__ partials) {
  pdl_wait();          // the partials come from grouped_bwd_kernel launched just before
  pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int64_t gch = static_cast<int64_t>(blockIdx.x) * kRowWarps + (threadIdx.x >> 5);
  if (gch >= total_channels) return;
  const int k = find_item(chan_prefix, n_items, gch);
  const dlmcq_group_item it = items[k];
  const int64_t ch = gch - __ldg(chan_prefix + k);
  const int64_t segs = (it.inner + DLMCQ_GROUP_SEG - 1) / DLMCQ_GROUP_SEG;
  const float* p = partials + __ldg(prefix + k) + ch * segs;
  double s = 0.0;
  for (int64_t j = lane; j < segs; j += 32) s += static_cast<double>(p[j]);
  s = warp_sum(s);
  if (lane == 0) {
    float r = static_cast<float>(s);
    if (it.form == DLMCQ_FORM_AFFINE || it.form == DLMCQ_FORM_A1) r = r * it.g;
    it.dscale[ch] = r;
  }
}

}  // namespace dlmcq

using namespace dlmcq;

extern "C" int dlmcq_fq_forward_grouped(const dlmcq_group_item* items, const int64_t* unit_prefix, int n_items,
                                        int64_t total_units, int dtype, void* stream) {
  if (!items || !unit_prefix || n_items < 1 || total_units < 0) return DLMCQ_EINVAL;
  if (total_units == 0) return DLMCQ_OK;
  const int64_t blocks = (total_units + kRowWarps - 1) / kRowWarps;
  if (blocks > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype != DLMCQ_F32 && dtype != DLMCQ_BF16) return DLMCQ_EINVAL;
  cudaError_t e = launch_pdl(dtype == DLMCQ_F32 ? grouped_fwd_kernel<float> : grouped_fwd_kernel<__nv_bfloat16>,
                             dim3(static_cast<unsigned>(blocks)), dim3(kRowWarps * 32), 0, st, items, unit_prefix,
                             n_items, total_units);
  if (e != cudaSuccess) return set_cuda_error(e);
  return DLMCQ_OK;
}

extern "C" int dlmcq_fq_backward_grouped(const dlmcq_group_item* items, const int64_t* unit_prefix,
                                         const int64_t* chan_prefix, int n_items, int64_t total_units,
                                         int64_t total_channels, int dtype, float* partials, void* stream) {
  if (!items || !unit_prefix || !chan_prefix || !partials || n_items < 1 || total_units < 0) return DLMCQ_EINVAL;
  if (total_units == 0) return DLMCQ_OK;
  const int64_t blocks = (total_units + kRowWarps - 1) / kRowWarps;
  const int64_t fblocks = (total_channels + kRowWarps - 1) / kRowWarps;
  if (blocks > 0x7fffffffLL || fblocks > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype != DLMCQ_F32 && dtype != DLMCQ_BF16) return DLMCQ_EINVAL;
  cudaError_t e = launch_pdl(dtype == DLMCQ_F32 ? grouped_bwd_kernel<float> : grouped_bwd_kernel<__nv_bfloat16>,
                             dim3(static_cast<unsigned>(blocks)), dim3(kRowWarps * 32), 0, st, items, unit_prefix,
                             n_items, total_units, partials);
  if (e != cudaSuccess) return set_cuda_error(e);
  e = launch_pdl(grouped_finalize_kernel, dim3(static_cast<unsigned>(fblocks)), dim3(kRowWarps * 32), 0, st, items,
                 unit_prefix, chan_prefix, n_items, total_channels, partials);
  if (e != cudaSuccess) return set_cuda_error(e);
  return DLMCQ_OK;
}
