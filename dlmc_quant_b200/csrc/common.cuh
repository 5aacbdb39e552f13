// common.cuh - shared device helpers for libdlmcq (sm_100a only).
//
// Everything on this path is HBM-bound element-wise / reduction work: the helpers here are
// 128-bit vector access, dtype conversion, warp/block reductions and the "last block
// finalises" pattern that keeps scale-gradient reductions deterministic without a second
// launch.  Compiled with -fmad=false: the reference's chains are sequences of separately
// rounded fp32 ops, so no multiply-add may be contracted unless written as fmaf() explicitly.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/dlmcq.h"

namespace dlmcq {

constexpr int kThreads = 256;          // threads per CTA for the streaming kernels
constexpr int kNumSmFallback = 148;    // B200
constexpr int kMaxPartialBlocks = 8192;
constexpr int kRowWarps = 8;           // warps per CTA in the warp-per-row kernels

int num_sms();
int set_cuda_error(cudaError_t e);
#define DLMCQ_LAUNCH_CHECK()                                   \
  do {                                                         \
    cudaError_t e__ = cudaGetLastError();                      \
    if (e__ != cudaSuccess) return ::dlmcq::set_cuda_error(e__); \
  } while (0)

// ---- dtype traits: 16-byte vectors -----------------------------------------------------
template <typename T>
struct Vec;
template <>
struct Vec<float> {
  static constexpr int N = 4;
  using raw = float4;
  __device__ static __forceinline__ void unpack(const raw& r, float (&f)[4]) {
    f[0] = r.x; f[1] = r.y; f[2] = r.z; f[3] = r.w;
  }
  __device__ static __forceinline__ raw pack(const float (&f)[4]) { return make_float4(f[0], f[1], f[2], f[3]); }
};
template <>
struct Vec<__nv_bfloat16> {
  static constexpr int N = 8;
  using raw = uint4;
  __device__ static __forceinline__ void unpack(const raw& r, float (&f)[8]) {
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {   // bf16 -> fp32 is a 16-bit shift, exact
      f[2 * i] = __uint_as_float(w[i] << 16);
      f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
  __device__ static __forceinline__ raw pack(const float (&f)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 p = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);   // RNE, one rounding
      w[i] = *reinterpret_cast<uint32_t*>(&p);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
  }
};

template <typename T>
__device__ __forceinline__ float to_f32(T v);
template <>
__device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T>
__device__ __forceinline__ T from_f32(float v);
template <>
__device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// Streaming 128-bit access.  Inputs are read exactly once (no reuse inside the kernel):
// bypass L1 allocation; outputs are written once: no-allocate in L1 as well.  L2 policy is
// left at default so that a consumer kernel (the conv) can still hit the fake-quantised
// tensor in the 126 MB L2.
template <typename R>
__device__ __forceinline__ R ld_stream(const R* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return *reinterpret_cast<R*>(&v);
}
template <typename R>
__device__ __forceinline__ void st_stream(R* p, const R& r) {
  const uint4 v = *reinterpret_cast<const uint4*>(&r);
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// ---- reductions ------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Block-wide sum of NQ quantities; result valid in thread 0.  Fixed order -> deterministic.
template <int NQ>
__device__ __forceinline__ void block_sum(float (&v)[NQ], float* smem /* >= NQ*32 floats */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int q = 0; q < NQ; ++q) v[q] = warp_sum(v[q]);
  __syncthreads();   // protect smem reuse across calls
  if (lane == 0) {
#pragma unroll
    for (int q = 0; q < NQ; ++q) smem[q * 32 + warp] = v[q];
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      float t = lane < nwarp ? smem[q * 32 + lane] : 0.f;
      v[q] = warp_sum(t);
    }
  }
}

// "Last block finalises": every block publishes its partials, takes a ticket, and the block
// that draws the last ticket reduces all partials in a fixed order.  The ticket counter is
// reset by that block, so a workspace that was zeroed once stays reusable.
__device__ __forceinline__ bool take_last_ticket(unsigned int* counter, unsigned int nblocks) {
  // Call after thread 0 has written this block's partials.  Only thread 0 fences: the fence orders ITS
  // partial-sum stores before the ticket; making all 256 threads fence would stall the whole block until
  // every streaming store of the block has been acknowledged.
  __shared__ bool is_last;
  if (threadIdx.x == 0) {
    __threadfence();
    unsigned int t = atomicAdd(counter, 1u);
    is_last = (t == nblocks - 1);
  }
  __syncthreads();
  if (is_last) __threadfence();   // acquire side: the other blocks' partials are visible below
  return is_last;
}

// Grid-wide barrier for cooperatively launched kernels (all CTAs co-resident): a monotonically increasing arrival
// counter; barrier number b (1-based) completes when it reaches b * gridDim.x.  The counter must be zero at launch.
__device__ __forceinline__ void grid_barrier(unsigned int* counter, unsigned int target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(counter, 1u);
    unsigned int seen;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(counter) : "memory");
    } while (seen < target);
  }
  __syncthreads();
}

// Workspace layout: [0,256) bytes = ticket counters, then float partials.
constexpr size_t kWsHeaderBytes = 256;
__host__ __device__ inline float* ws_partials(void* ws) {
  return reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + kWsHeaderBytes);
}
__host__ __device__ inline unsigned int* ws_counter(void* ws, int i = 0) {
  return reinterpret_cast<unsigned int*>(ws) + i;
}

// Per-channel layouts are processed as rows = outer*channels of length `inner`, each row cut
// into `segs` segments of `seg` elements; one warp owns one (row, segment) work item.
struct RowGeom {
  int64_t rows;
  int64_t channels;
  int64_t inner;
  int64_t segs;   // segments per row
  int64_t seg;    // elements per segment (multiple of 512 -> 16-byte aligned cuts)
};
constexpr int64_t kRowSegMin = 2048;          // ~8 KB (fp32) per warp item: small enough for an even last wave
constexpr int64_t kRowItemsTarget = 1 << 20;
inline RowGeom make_geom(int64_t outer, int64_t channels, int64_t inner, int64_t seg_min = kRowSegMin) {
  RowGeom gm;
  gm.rows = outer * channels;
  gm.channels = channels;
  gm.inner = inner;
  int64_t segs = (inner + seg_min - 1) / seg_min;
  int64_t cap = kRowItemsTarget / (gm.rows > 0 ? gm.rows : 1);
  if (cap < 1) cap = 1;
  if (segs > cap) segs = cap;
  if (segs < 1) segs = 1;
  int64_t seg = (inner + segs - 1) / segs;
  seg = (seg + 511) / 512 * 512;
  if (seg < 512) seg = 512;
  gm.seg = seg;
  gm.segs = (inner + seg - 1) / seg;
  if (gm.segs < 1) gm.segs = 1;
  return gm;
}

// Channel-major geometry for per-channel ACTIVATIONS with short rows ([B, C, HW], HW < 256): one warp owns
// (channel, a chunk of batch indices) and walks the flattened (b, e) index space of that channel.
struct CmajGeom {
  int64_t outer, channels, inner;
  int32_t bc;        // batch indices per work item
  int32_t chunks;    // work items per channel
  uint32_t magic;    // floor(2^24 / inner) + 1: (t * magic) >> 24 == t / inner for t * inner < 2^24
};
constexpr int kCmajUnroll = 8;
constexpr int64_t kCmajMaxInner = 256;

// short rows, more than one batch index, and 32-bit element offsets inside one work item
inline bool cmaj_ok(int64_t outer, int64_t channels, int64_t inner) {
  return outer > 1 && inner >= 1 && inner < kCmajMaxInner && channels * 8192 < (int64_t(1) << 31);
}
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// vec: elements per access unit (1, or the 128-bit vector width when rows are whole vectors): the kernels index
// units, so `magic` divides by inner / vec
inline CmajGeom make_cmaj(int64_t outer, int64_t channels, int64_t inner, int vec = 1) {
  CmajGeom g;
  g.outer = outer; g.channels = channels; g.inner = inner;
  int64_t bc = 8192 / (inner > 0 ? inner : 1);
  if (bc < 1) bc = 1;
  if (bc > outer) bc = outer;
  g.bc = static_cast<int32_t>(bc);
  g.chunks = static_cast<int32_t>((outer + bc - 1) / bc);
  const uint32_t units = static_cast<uint32_t>(inner > 0 ? inner / vec : 1);
  g.magic = static_cast<uint32_t>((1u << 24) / (units > 0 ? units : 1)) + 1u;
  return g;
}
// rows are whole 128-bit vectors and every row start is 16-byte aligned
template <typename T>
inline bool cmaj_vec_ok(int64_t inner, const void* a, const void* b, const void* c, const void* d) {
  return inner % Vec<T>::N == 0 && aligned16(a) && aligned16(b) && aligned16(c) && aligned16(d);
}

// Slab geometry: per-channel ACTIVATIONS [B, C, inner] whose short rows are NOT whole 128-bit vectors (7x7, 5x5, 3x3
// planes, inner == 1).  G = VEC / gcd(inner, VEC) adjacent channels form a contiguous, 16-byte-aligned run of
// W = G * inner / VEC vectors per batch index.  Thread (r, v) of a CTA owns vector v of one run for the batch indices
// r, r + R, ...: the channel of each of its VEC elements is the same for the whole kernel, so the per-channel constants
// are resolved once into registers, every access is a coalesced 128-bit one, and no lane idles on a row remainder
// (the scalar channel-major kernels spend 22 - 41 instructions per element on 7x7 planes and are issue-bound).
struct SlabGeom {
  int64_t outer, channels, inner;
  int64_t plane_vecs;   // C * inner / VEC: vectors between consecutive batch indices
  int32_t G, W, R;      // channels per group, vectors per group row, batch rows per CTA pass (R * W <= kThreads)
  int32_t bc, chunks;   // batch indices per CTA, CTAs per channel group
  int32_t groups;       // C / G
};
constexpr int kSlabUnroll = 4;
template <typename T>
inline bool slab_ok(int64_t outer, int64_t channels, int64_t inner, const void* a, const void* b, const void* c,
                    const void* d) {
  constexpr int VEC = Vec<T>::N;
  if (!cmaj_ok(outer, channels, inner) || inner % VEC == 0) return false;
  int g = 1;
  while ((inner * g) % VEC != 0) g <<= 1;                  // VEC / gcd(inner, VEC): a power of two <= VEC
  return channels % g == 0 && aligned16(a) && aligned16(b) && aligned16(c) && aligned16(d) &&
         channels / g * outer < (int64_t(1) << 31);      // grid = groups * chunks, chunks <= outer
}
template <typename T>
inline SlabGeom make_slab(int64_t outer, int64_t channels, int64_t inner) {
  constexpr int VEC = Vec<T>::N;
  SlabGeom s;
  s.outer = outer; s.channels = channels; s.inner = inner;
  int g = 1;
  while ((inner * g) % VEC != 0) g <<= 1;
  s.G = g;
  s.W = static_cast<int32_t>(inner * g / VEC);
  s.R = kThreads / s.W;
  s.groups = static_cast<int32_t>(channels / g);
  s.plane_vecs = channels * inner / VEC;
  // CTAs live long (the per-thread constants and the CTA fold are paid once per CTA): as few batch chunks as still
  // give ~8 CTAs per SM, each a whole number of (R * unroll)-row passes
  const int64_t pass_rows = static_cast<int64_t>(s.R) * kSlabUnroll * 2;
  int64_t chunks = (148 * 8 + s.groups - 1) / s.groups;
  if (chunks < 1) chunks = 1;
  int64_t bc = (outer + chunks - 1) / chunks;
  bc = (bc + pass_rows - 1) / pass_rows * pass_rows;
  if (bc > outer) bc = outer;
  s.bc = static_cast<int32_t>(bc);
  s.chunks = static_cast<int32_t>((outer + bc - 1) / bc);
  return s;
}

// Programmatic dependent launch: consecutive kernels of one stream (the per-layer quantizer launches of a
// training step) hide their launch latency behind the predecessor's tail.  Every kernel launched this way
// executes pdl_wait() before its first global-memory access - it then sees all of the predecessor's
// writes - and pdl_trigger() right away so that its own successor can be staged early.  The exceptions load
// data that the host or the call sequence proves the predecessor does not write (bnq_apply_kernel, and the flat
// fake-quant kernels when capture_check reports an independent launch) before pdl_wait().
// Invariant: every CTA of every kernel launched through launch_pdl executes pdl_wait() before it triggers, stores
// or exits.  So launch N+2 cannot start before every CTA of launch N+1 has passed its wait, i.e. before launch N
// has completed and flushed: loads hoisted above the wait of N+2 can only race with N+1, and checking N+2's reads
// against N+1's writes alone is enough.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;"); }
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}


// Persistent grid for a streaming kernel over `work_items` block-tiles.
inline int stream_grid(int64_t tiles, int blocks_per_sm) {
  int64_t cap = static_cast<int64_t>(num_sms()) * blocks_per_sm;
  if (cap > kMaxPartialBlocks && blocks_per_sm <= 16) cap = kMaxPartialBlocks;   // reductions size their partials by this
  int64_t g = tiles < cap ? tiles : cap;
  return g < 1 ? 1 : static_cast<int>(g);
}

}  // namespace dlmcq
