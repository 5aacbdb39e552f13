// qgemm_kernels.cu - the layer's matrix product on the INTEGER CODES (SURVEY.md section 8f row f2, consumer side).
//
// Reference: dlmc/quantization/scalar/modules/linear.py / conv.py `_forward_func(q_input, q_weight)` called from
// modules/base.py:140 - F.linear / F.conv2d on the two fake-quantised fp32 tensors.  For a per-tensor activation
// quantizer and a per-output-channel (or per-tensor) weight quantizer without a weight offset the product factors:
//
//     y_a[m,k] = (ca[m,k] - z_a) * m_a + o_a          (z_a: FORM_ZP zero-point, o_a: FORM_A1 / AFFINE offset)
//     y_w[n,k] =  cw[n,k] * m_w[n]
//     sum_k y_a*y_w = m_a*m_w[n] * sum_k ca*cw  +  (o_a - z_a*m_a) * m_w[n] * sum_k cw[n,k]
//                   = alpha[n] * acc[m,n] + beta[n]
//
// acc is an exact integer dot product of the codes.  It runs on the 5th-generation tensor cores:
//   * operands: one BYTE per code (1/4 of the fp32 activation traffic the fake-quantised tensor costs cuDNN),
//     K-major, staged by TMA (cp.async.bulk.tensor.2d, 128-byte swizzle) through a 4-stage mbarrier pipeline;
//   * tcgen05.mma cta_group::1 issued by ONE thread, M=128 x N=128 x K=32 per instruction, accumulators in TMEM
//     (128 lanes x 128 columns); kind::i8 (u8|s8 x s8 -> s32, exact for every code width up to 8 bits; sm_100a has
//     it) or kind::f8f6f4 on codes stored as e4m3 bytes (exact for |code| <= 16, fp32 accumulators);
//   * epilogue: tcgen05.ld (32x32b.x32) -> registers -> a padded smem transpose -> coalesced 128-byte row stores of
//     out = RN(RN(acc * alpha[n]) + beta[n]) (+ ReLU), fp32 or bf16.
// Warp roles (576 threads): warp 0 = TMA producer, warp 1 = TMEM allocation + MMA issue, warps 2-17 = epilogue in
// two groups of 8 (warp w may only touch TMEM lanes 32*(w%4) .. +31: two warps per lane quarter and group, 64 of the
// tile's 128 columns each).  Persistent, one CTA per SM (206 KB of smem, 256 TMEM columns = two accumulator
// buffers, one per epilogue group): while one group streams its tile out, the other reads the next accumulator and
// the loads and MMAs of the tiles after that are already running.  This path is bound by the bytes it moves (codes in, y out), not by the
// tensor pipe - the point of doing the product on codes is the 4x smaller operand.
//
// Also here: dlmcq_codes_forward (x -> one byte per code, the same arithmetic as dlmcq_fq_forward, streaming) and
// dlmcq_qgemm_prepare (alpha / beta from the DEVICE-resident qparams: no host sync, learnable scales stay put).
#include <cuda.h>       // CUtensorMap + enums only; the encoder is fetched through cudaGetDriverEntryPoint
#include <cuda_fp8.h>

#include <type_traits>

#include "bnq_math.cuh"
#include "codes.cuh"

namespace dlmcq {
namespace {

constexpr int kBM = 128, kBN = 128, kBK = 128;                // tile; kBK bytes = codes (one byte each)
constexpr int kStages = 4;
constexpr int kABytes = kBM * kBK, kBBytes = kBN * kBK, kStageBytes = kABytes + kBBytes;
constexpr int kUmmaK = 32;                                    // codes one tcgen05.mma of an 8-bit kind consumes
constexpr int kEpiWarps = 16;                                 // two groups of 8 (two per TMEM lane quarter, 64 columns each)
constexpr int kEpiGroupWarps = kEpiWarps / 2;                 // group g drains accumulator buffer g: even / odd tiles
constexpr int kGemmThreads = 64 + 32 * kEpiWarps;
constexpr int kTmemCols = 2 * kBN;                            // double-buffered accumulator, one 32-bit column per output column
constexpr int kStgPitch = 36;                                 // floats per row of the epilogue's transpose buffer
constexpr int kStgBytes = kEpiWarps * 32 * kStgPitch * 4;
constexpr int kBarBytes = 128;
constexpr size_t kGemmSmem = 1024 + static_cast<size_t>(kStages) * kStageBytes + kStgBytes + kBarBytes;
constexpr long long kWatchdogCycles = 30000000000LL;          // ~15 s in ONE barrier wait: a wedged pipeline traps instead of hanging the GPU

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  long long t0 = 0;
  for (uint32_t spin = 0; !done; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (!done && (spin & 1023u) == 1023u) {
      const long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > kWatchdogCycles) __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// im2col mode: 128 consecutive output pixels (N*Ho*Wo order, wrapping rows and images inside the map's bounding box)
// of one filter tap: {c0, w, h, img} is the window corner of the first pixel, {off_w, off_h} the tap's offset in input
// pixels (s*dil_w, r*dil_h).  Pixels outside the image arrive as zero bytes.
__device__ __forceinline__ void tma_load_im2col(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int w, int h,
                                                int img, uint16_t off_w, uint16_t off_h) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2], {%7, %8};"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(w), "r"(h), "r"(img), "h"(off_w),
        "h"(off_h)
      : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// tcgen05.commit: the mbarrier receives one arrival when every tcgen05.mma this thread issued so far has completed
// (it implies tcgen05.fence::before_thread_sync)
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// Shared-memory matrix descriptor of a K-major operand tile laid out by TMA with the 128-byte swizzle: rows of 128
// bytes, 8-row groups 1024 bytes apart (stride byte offset), descriptor version 1 (sm_100), layout type 2
// (SWIZZLE_128B); the leading byte offset is not used by swizzled K-major layouts (canonical value 1).  The tile
// base is 1024-byte aligned, so a K step of 32 bytes inside the swizzle atom is a plain advance of the start address.
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
  return static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (static_cast<uint64_t>(1024 >> 4) << 32) |
         (1ull << 46) | (2ull << 61);
}
// The same for 64-byte rows (SWIZZLE_64B, layout type 4): 8-row groups 512 bytes apart.
__device__ __forceinline__ uint64_t umma_desc_sw64(uint32_t smem_addr) {
  return static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (static_cast<uint64_t>(512 >> 4) << 32) |
         (1ull << 46) | (4ull << 61);
}
template <int KIND>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  if (KIND == DLMCQ_QGEMM_I8) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n\t"
      "tcgen05.wait::ld.sync.aligned;"          // same statement: the registers may not be read before the wait
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}

// ---------------------------------------------------------------------------------------------------------------
// out[m, n] = RN(RN(float(sum_k A[m,k] * B[n,k]) * alpha[n]) + beta[n])   (optionally max(., 0))
//
// Persistent: one CTA per SM walks the 128x128 output tiles (N tiles fastest, so the CTAs that share an A tile run
// at the same time and the second read comes from L2).  Three decoupled pipelines:
//   TMA producer  --full[s]/empty[s]-->  MMA thread  --acc_full[b]/acc_empty[b]-->  8 epilogue warps
// The accumulator is double-buffered in TMEM (2 x 128 columns), so the epilogue of tile i overlaps the loads and
// MMAs of tile i+1, and the operand ring keeps running across tile boundaries.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

template <bool IS_INT>
__device__ __forceinline__ float acc_value(uint32_t v) {
  return IS_INT ? static_cast<float>(static_cast<int>(v)) : __uint_as_float(v);
}

// Implicit-GEMM geometry of a convolution (qconv_kernel): output row m of the [B*Ho*Wo, n] product is pixel
// (m / HoWo, oh, ow) of a channels-last output; the A operand is the im2col view of the [B, H, W, Cin] codes.
struct ConvArgs {
  int H, W, Ho, Wo, HoWo, kh, kw, sh, sw, ph, pw, dh, dw, cchunks;   // cchunks = Cin / CHUNK
};

// Taps t in [0, k) with 0 <= top + t*d < size form one contiguous range [lo, hi1) (empty when lo >= hi1); both ends
// lie in [0, k], so (lo, hi1) indexes a (k+1) x (k+1) table.
__device__ __forceinline__ void tap_range(int top, int size, int d, int k, int& lo, int& hi1) {
  lo = top >= 0 ? 0 : min(k, (d - 1 - top) / d);
  const int last = size - 1 - top;
  hi1 = last < 0 ? 0 : min(k, last / d + 1);
}

// Offset of output row m's beta vector in the border-class table [(kh+1)^2 (kw+1)^2][N] (dlmcq_qconv_prepare).
__device__ __forceinline__ int conv_beta_offset(const ConvArgs& c, int m, int N) {
  const int img = m / c.HoWo, pix = m - img * c.HoWo;
  const int oh = pix / c.Wo, ow = pix - oh * c.Wo;
  int rl, rh, sl, sh;
  tap_range(oh * c.sh - c.ph, c.H, c.dh, c.kh, rl, rh);
  tap_range(ow * c.sw - c.pw, c.W, c.dw, c.kw, sl, sh);
  return (((rl * (c.kh + 1) + rh) * (c.kw + 1) + sl) * (c.kw + 1) + sh) * N;
}

// Per-column epilogue constants of one 32-column piece, fetched BEFORE the warp waits for the accumulator (their
// latency hides behind the wait).  MODE 0: one column per lane; 1: four (fp32 line stores); 2: eight (bf16).
// BE = false (convolutions): beta depends on the row as well and is read per row from the border-class table.
template <int MODE, bool BE = true>
struct EpiConst {
  static constexpr int W = MODE == 0 ? 1 : (MODE == 1 ? 4 : 8);
  float al[W], be[W];
  __device__ __forceinline__ void load(const float* __restrict__ alpha, const float* __restrict__ beta, int col0, int lane,
                                       int N) {
    const int col = col0 + (MODE == 0 ? lane : (MODE == 1 ? (lane & 7) * 4 : (lane & 3) * 8));
#pragma unroll
    for (int e = 0; e < W; ++e) {
      const bool ok = col + e < N;
      al[e] = ok ? __ldg(alpha + col + e) : 0.f;
      if (BE) be[e] = ok ? __ldg(beta + col + e) : 0.f;
    }
  }
};

// One 32-row x 32-column piece of the tile: this lane holds row `lane` (32 accumulators); the piece is transposed
// through a padded smem buffer (pitch 36 floats: 128-bit writes and reads are both conflict-free) so that global
// stores are whole 128-byte lines.  MODE 0: scalar stores (any N, any alignment); 1: fp32, 16-byte stores
// (N % 4 == 0); 2: bf16, 16-byte stores of 8 values (N % 8 == 0).  All smem reads are issued before the first
// store; `floor` is 0 for a fused ReLU and -inf otherwise (max.NaN: NaN propagates, -0 -> +0, like torch.relu).
// CONV: beta is the row's border-class vector, beta + boff(row); each lane parks its row's offset in the transpose
// buffer's padding column 32 so that every lane can read the offsets of the rows it stores.
template <bool IS_INT, int MODE, bool CONV>
__device__ __forceinline__ void epilogue_piece(const uint32_t (&v)[32], float* stg, int lane, int row0, int col0, int M,
                                               int N, const EpiConst<MODE, !CONV>& k, void* __restrict__ out, float floor,
                                               int out_bf16, const float* __restrict__ beta, int boff) {
#pragma unroll
  for (int j = 0; j < 8; ++j)
    *reinterpret_cast<float4*>(stg + lane * kStgPitch + 4 * j) =
        make_float4(acc_value<IS_INT>(v[4 * j]), acc_value<IS_INT>(v[4 * j + 1]), acc_value<IS_INT>(v[4 * j + 2]),
                    acc_value<IS_INT>(v[4 * j + 3]));
  if (CONV) reinterpret_cast<int*>(stg)[lane * kStgPitch + 32] = boff;
  __syncwarp();
  const int* const boffs = reinterpret_cast<const int*>(stg) + 32;   // row r's offset: boffs[r * kStgPitch]
  const int rows = M - row0;                                    // >= 1; the common case is a full piece (>= 32)
  if (MODE == 1) {
    const int rsub = lane >> 3, c4 = (lane & 7) * 4, col = col0 + c4;
    if (col < N) {
      float* p = static_cast<float*>(out) + static_cast<size_t>(row0 + rsub) * N + col;
      const size_t step = static_cast<size_t>(4) * N;
#pragma unroll
      for (int h = 0; h < 2; ++h) {                             // two batches of four rows: 4 smem reads in flight, 16 live registers
        float4 t[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) t[i] = *reinterpret_cast<const float4*>(stg + ((h * 4 + i) * 4 + rsub) * kStgPitch + c4);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int r = (h * 4 + i) * 4 + rsub;
          float4 be;
          if (CONV) be = __ldg(reinterpret_cast<const float4*>(beta + boffs[r * kStgPitch] + col));
          else be = make_float4(k.be[0], k.be[1], k.be[2], k.be[3]);
          float4 o;
          o.x = max_nan(__fadd_rn(__fmul_rn(t[i].x, k.al[0]), be.x), floor);
          o.y = max_nan(__fadd_rn(__fmul_rn(t[i].y, k.al[1]), be.y), floor);
          o.z = max_nan(__fadd_rn(__fmul_rn(t[i].z, k.al[2]), be.z), floor);
          o.w = max_nan(__fadd_rn(__fmul_rn(t[i].w, k.al[3]), be.w), floor);
          if (r < rows) st_stream(reinterpret_cast<float4*>(p + (h * 4 + i) * step), o);
        }
      }
    }
    __syncwarp();
  } else if (MODE == 2) {
    const int rsub = lane >> 2, c8 = (lane & 3) * 8, col = col0 + c8;
    if (col < N) {
      __nv_bfloat16* p = static_cast<__nv_bfloat16*>(out) + static_cast<size_t>(row0 + rsub) * N + col;
      const size_t step = static_cast<size_t>(8) * N;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        float4 t[2][2];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          t[i][0] = *reinterpret_cast<const float4*>(stg + ((h * 2 + i) * 8 + rsub) * kStgPitch + c8);
          t[i][1] = *reinterpret_cast<const float4*>(stg + ((h * 2 + i) * 8 + rsub) * kStgPitch + c8 + 4);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int r = (h * 2 + i) * 8 + rsub;
          float o[8] = {t[i][0].x, t[i][0].y, t[i][0].z, t[i][0].w, t[i][1].x, t[i][1].y, t[i][1].z, t[i][1].w};
          float be[8];
          if (CONV) {
            const float4* bp = reinterpret_cast<const float4*>(beta + boffs[r * kStgPitch] + col);
            const float4 b0 = __ldg(bp), b1 = __ldg(bp + 1);
            be[0] = b0.x; be[1] = b0.y; be[2] = b0.z; be[3] = b0.w; be[4] = b1.x; be[5] = b1.y; be[6] = b1.z; be[7] = b1.w;
          } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) be[e] = k.be[e];
          }
#pragma unroll
          for (int e = 0; e < 8; ++e) o[e] = max_nan(__fadd_rn(__fmul_rn(o[e], k.al[e]), be[e]), floor);
          if (r < rows) st_stream(reinterpret_cast<uint4*>(p + (h * 2 + i) * step), Vec<__nv_bfloat16>::pack(o));
        }
      }
    }
    __syncwarp();
  } else {
    const int col = col0 + lane;
    if (col < N) {
      const int nr = rows < 32 ? rows : 32;
      for (int r = 0; r < nr; ++r) {
        const float be = CONV ? __ldg(beta + boffs[r * kStgPitch] + col) : k.be[0];
        const float o = max_nan(__fadd_rn(__fmul_rn(stg[r * kStgPitch + lane], k.al[0]), be), floor);
        const size_t idx = static_cast<size_t>(row0 + r) * static_cast<size_t>(N) + static_cast<size_t>(col);
        if (out_bf16) static_cast<__nv_bfloat16*>(out)[idx] = __float2bfloat16_rn(o);
        else static_cast<float*>(out)[idx] = o;
      }
    }
    __syncwarp();
  }
}

// The tile loop of one epilogue warp.  The 16 epilogue warps form two groups: group g owns accumulator buffer g,
// i.e. the CTA's even / odd tiles, so while one group streams its tile to global memory the other one is already
// waiting for / reading the next accumulator - the store pipe never idles behind a barrier round trip (timeline:
// profiles/r02_qgemm_timeline_probe.log).  Inside a group a warp owns TMEM lane quarter q and 64 columns (two
// 32-column pieces, read one at a time: 32 live accumulator registers).  The buffer is handed back to the MMA thread
// by ONE arrival per warp, right after the warp's last TMEM read.
template <bool IS_INT, int MODE, bool CONV>
__device__ __forceinline__ void epilogue_loop(uint32_t tmem, uint32_t bar_acc_full, uint32_t bar_acc_empty, float* stg,
                                              int lane, int q, int grp, int chalf, int num_tiles, int tiles_n, int M,
                                              int N, const float* __restrict__ alpha, const float* __restrict__ beta,
                                              void* __restrict__ out, float floor, int out_bf16, const ConvArgs& cv) {
  const uint32_t full = bar_acc_full + 8 * grp, empty = bar_acc_empty + 8 * grp;
  const uint32_t tbase = tmem + grp * kBN + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(chalf * 64);
  uint32_t ti = grp;
  for (int tile = blockIdx.x + grp * gridDim.x; tile < num_tiles; tile += 2 * gridDim.x, ti += 2) {
    const int m0 = (tile / tiles_n) * kBM, n0 = (tile % tiles_n) * kBN;
    const int col0 = n0 + chalf * 64, row0 = m0 + q * 32;
    const bool has0 = col0 < N, has1 = col0 + 32 < N;            // warp-uniform
    EpiConst<MODE, !CONV> k0;
    k0.load(alpha, beta, col0, lane, N);
    const int boff = CONV ? conv_beta_offset(cv, row0 + lane, N) : 0;   // this lane's row (the table covers rows >= M too)
    mbar_wait(full, (ti >> 1) & 1);
    tc_fence_after();
    uint32_t v[32];
    if (has0) tmem_ld32(tbase, v);
    if (!has1) {                                                // nothing more to read from this buffer
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(empty);
    }
    if (has0 && row0 < M)
      epilogue_piece<IS_INT, MODE, CONV>(v, stg, lane, row0, col0, M, N, k0, out, floor, out_bf16, beta, boff);
    if (has1) {
      EpiConst<MODE, !CONV> k1;                                 // L1-resident by now; fetched here to keep registers free
      k1.load(alpha, beta, col0 + 32, lane, N);
      tmem_ld32(tbase + 32, v);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(empty);
      if (row0 < M)
        epilogue_piece<IS_INT, MODE, CONV>(v, stg, lane, row0, col0 + 32, M, N, k1, out, floor, out_bf16, beta, boff);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Code-output epilogue (dlmcq_qgemm_codes / dlmcq_qconv_codes).  The layer output v = RN(RN(acc * alpha[n]) + beta),
// rounded to T (what the unchained layer stores), goes on through the consumer's eval BatchNorm, the optional ReLU
// and the consumer's AFFINE input quantizer, and only the code byte is stored: element for element the arithmetic of
// bnq_apply_kernel<T, false, true, ENC> (bnq_math.cuh) - the packed fast path under the same domain guard, the
// literal chain for vectors outside it.  BatchNorm is NOT folded into alpha / beta: that would change the roundings.
// Layout: a lane owns one output row of a 32-column piece (the layout tcgen05.ld delivers), so its 32 code bytes are
// one 32-byte sector and no transpose is needed.  The warp's transpose buffer holds the per-column constants instead,
// staged once per tile and read as warp-wide broadcasts.
// ---------------------------------------------------------------------------------------------------------------
struct CodeTail {
  const float* gamma;
  const float* beta;
  const float* mean;       // running_mean
  const float* var;        // running_var
  const float* scale;      // consumer's quantizer
  const float* offset;
  float eps, g, lo, hi;
  int relu, enc;
};
constexpr int kCstBeta = 4 * 64;          // floats: 64 x float4 {alpha, mean, gamma*invstd, bn beta}, then 64 x beta

// The 64 columns col0 .. col0+63 of this warp's tile; returns whether their BatchNorm constants lie in the fast-path
// domain (c2.safe of bnq_apply_kernel).
template <bool CONV>
__device__ __forceinline__ bool stage_code_consts(float* stg, const float* __restrict__ alpha,
                                                  const float* __restrict__ beta, const CodeTail& t, int col0,
                                                  int lane, int N) {
  __syncwarp();                                                 // every lane is done with the previous tile's
  float m = 0.f;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int j = lane + 32 * h, col = col0 + j;
    float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
    float be = 0.f;
    if (col < N) {
      c.x = __ldg(alpha + col);
      c.y = __ldg(t.mean + col);
      c.z = bn_scale(t.gamma ? __ldg(t.gamma + col) : 1.f, bn_eval_invstd(__ldg(t.var + col), t.eps));
      c.w = t.beta ? __ldg(t.beta + col) : 0.f;
      if (!CONV) be = __ldg(beta + col);
      m = fmaxf(m, fmaxf(fmaxf(fabsf(c.y), fabsf(c.z)), fabsf(c.w)));   // NaN constants flow through, as there
    }
    reinterpret_cast<float4*>(stg)[j] = c;
    if (!CONV) stg[kCstBeta + j] = be;
  }
  const bool safe = __all_sync(0xffffffffu, m <= kBnqSafe);
  __syncwarp();
  return safe;
}

// One 32-column piece of row `row` (this lane): columns col .. col+31 (col + 16 >= N: only the first 16 exist, N % 16
// == 0), constants at cbase .. cbase+31 of the staging buffer; CONV: brow = the row's border-class beta row + col.
template <bool IS_INT, bool CONV, typename T>
__device__ __forceinline__ void code_piece(const uint32_t (&v)[32], const float* stg, int cbase, int row, int col, int M,
                                           int N, const float* __restrict__ brow, const QuantK& k, bool fast_ok,
                                           float floor, const CodeTail& t, uint8_t* __restrict__ out) {
  uint32_t w[8];
#pragma unroll
  for (int j = 0; j < 32; j += 4) {
    float4 c[4];
    float x[4], code[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      c[e] = reinterpret_cast<const float4*>(stg)[cbase + j + e];
      const float be = CONV ? (col + j + e < N ? __ldg(brow + j + e) : 0.f) : stg[kCstBeta + cbase + j + e];
      x[e] = to_f32<T>(from_f32<T>(__fadd_rn(__fmul_rn(acc_value<IS_INT>(v[j + e]), c[e].x), be)));
    }
    if (fast_ok && absmax_vec<4>(x, 0.f) <= kBnqSafe) {
#pragma unroll
      for (int e = 0; e < 4; e += 2) {
        const float2 tt = __fadd2_rn(make_float2(x[e], x[e + 1]), make_float2(-c[e].y, -c[e + 1].y));
        const float2 z = __ffma2_rn(tt, make_float2(c[e].z, c[e + 1].z), make_float2(c[e].w, c[e + 1].w));
        float2 q, cc, cd;
        quant_pair(round_to_storage<T>(act_pair(z, floor)), k, q, cc, cd);
        code[e] = cd.x;
        code[e + 1] = cd.y;
      }
    } else {
      BnCh<4> bc;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        bc.mean[e] = c[e].y;
        bc.a[e] = c[e].z;
        bc.b[e] = c[e].w;
        bc.istd[e] = 0.f;                                       // not read by the forward
      }
      float act[4], y[4];
      apply_generic_vec<T, 4, true>(x, nullptr, bc, t.relu != 0, k.p, k.lo, k.hi, act, y, code);
    }
    w[j / 4] = code_byte_rt(code[0], t.enc) | (code_byte_rt(code[1], t.enc) << 8) |
               (code_byte_rt(code[2], t.enc) << 16) | (code_byte_rt(code[3], t.enc) << 24);
  }
  if (row < M) {
    uint8_t* p = out + static_cast<size_t>(row) * N + col;
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(w[0]), "r"(w[1]), "r"(w[2]),
                 "r"(w[3])
                 : "memory");
    if (col + 16 < N)
      asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p + 16), "r"(w[4]), "r"(w[5]),
                   "r"(w[6]), "r"(w[7])
                   : "memory");
  }
  __syncwarp();
}

// The tile loop of one epilogue warp for the code output: the same groups, TMEM reads and buffer hand-back as
// epilogue_loop.
template <bool IS_INT, bool CONV, typename T>
__device__ __forceinline__ void code_epilogue_loop(uint32_t tmem, uint32_t bar_acc_full, uint32_t bar_acc_empty,
                                                   float* stg, int lane, int q, int grp, int chalf, int num_tiles,
                                                   int tiles_n, int M, int N, const float* __restrict__ alpha,
                                                   const float* __restrict__ beta, uint8_t* __restrict__ out,
                                                   const ConvArgs& cv, const CodeTail& t) {
  const uint32_t full = bar_acc_full + 8 * grp, empty = bar_acc_empty + 8 * grp;
  const uint32_t tbase = tmem + grp * kBN + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(chalf * 64);
  const QuantK k = make_quantk(t.scale, t.offset, t.g, t.lo, t.hi);
  const float floor = t.relu ? 0.f : -INFINITY;
  uint32_t ti = grp;
  for (int tile = blockIdx.x + grp * gridDim.x; tile < num_tiles; tile += 2 * gridDim.x, ti += 2) {
    const int m0 = (tile / tiles_n) * kBM, n0 = (tile % tiles_n) * kBN;
    const int col0 = n0 + chalf * 64, row0 = m0 + q * 32, row = row0 + lane;
    const bool has0 = col0 < N, has1 = col0 + 32 < N;            // warp-uniform
    const bool fast_ok = stage_code_consts<CONV>(stg, alpha, beta, t, col0, lane, N) && k.fast;
    const float* brow = CONV ? beta + conv_beta_offset(cv, row, N) + col0 : nullptr;
    mbar_wait(full, (ti >> 1) & 1);
    tc_fence_after();
    uint32_t v[32];
    if (has0) tmem_ld32(tbase, v);
    if (!has1) {
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(empty);
    }
    if (has0 && row0 < M) code_piece<IS_INT, CONV, T>(v, stg, 0, row, col0, M, N, brow, k, fast_ok, floor, t, out);
    if (has1) {
      tmem_ld32(tbase + 32, v);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(empty);
      if (row0 < M)
        code_piece<IS_INT, CONV, T>(v, stg, 32, row, col0 + 32, M, N, CONV ? brow + 32 : nullptr, k, fast_ok, floor, t,
                                    out);
    }
  }
}

// The kernel body, shared by the GEMM (CHUNK = 0: A is a [M, K] matrix, 128-byte K blocks) and the implicit-GEMM
// convolution (CHUNK = 128 / 64: A is the im2col view of channels-last codes; one K block = one filter tap x CHUNK
// channels, K = kh*kw*Cin in (r, s, c) order, so B is the [n, K] matrix of channels-last weight codes and a K block
// never straddles a tap).  Only the A producer, the K-block width and the epilogue's beta differ.
// CT = void: out is the layer output (fp32 / bf16); CT = float / __nv_bfloat16: out is the consumer's code bytes
// (code_epilogue_loop with *tail), CT being the dtype of the layer output the codes are computed from.
template <int KIND, int CHUNK, typename CT = void>
__device__ __forceinline__ void gemm_pipeline(const CUtensorMap* map_a, const CUtensorMap* map_b,
                                              const float* __restrict__ alpha, const float* __restrict__ beta,
                                              void* __restrict__ out, int M, int N, int K, uint32_t idesc, int relu,
                                              int out_bf16, int vec_ok, const ConvArgs& cv,
                                              const CodeTail* tail = nullptr) {
  constexpr int kKb = CHUNK == 0 ? kBK : CHUNK;                 // K bytes per block
  constexpr uint32_t kTx = CHUNK == 0 ? kStageBytes : 2 * kBM * CHUNK;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;                 // the swizzle atoms need 1024-byte alignment
  uint8_t* const tiles = smem_raw + (base - raw);
  float* const stg_all = reinterpret_cast<float*>(tiles + kStages * kStageBytes);
  const uint32_t bars = base + kStages * kStageBytes + kStgBytes;
  const uint32_t bar_full = bars, bar_empty = bars + 8 * kStages, bar_acc_full = bars + 16 * kStages,
                 bar_acc_empty = bar_acc_full + 16;
  uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(tiles + kStages * kStageBytes + kStgBytes + 16 * kStages + 32);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles_n = (N + kBN - 1) / kBN, tiles_m = (M + kBM - 1) / kBM;
  const int num_tiles = tiles_m * tiles_n;
  const int num_kb = (K + kKb - 1) / kKb;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(bar_full + 8 * s, 1);                           // one arrive.expect_tx by the producer
      mbar_init(bar_empty + 8 * s, 1);                          // one tcgen05.commit by the MMA thread
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(bar_acc_full + 8 * b, 1);                       // one tcgen05.commit per tile
      mbar_init(bar_acc_empty + 8 * b, kEpiGroupWarps);         // one arrival per warp of the group that drains buffer b
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {                                              // the allocating warp also frees (whole warp, aligned)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(static_cast<uint32_t>(kTmemCols))
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(tmem_slot);

  if (warp == 0) {
    if (lane == 0) {
      // ===== TMA producer =====
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m0 = (tile / tiles_n) * kBM, n0 = (tile % tiles_n) * kBN;
        if constexpr (CHUNK == 0) {
          for (int kb = 0; kb < num_kb; ++kb, ++it) {
            const uint32_t s = it % kStages, ph = (it / kStages) & 1;
            mbar_wait(bar_empty + 8 * s, ph ^ 1);               // slot free (passes at once in the first round)
            mbar_expect_tx(bar_full + 8 * s, kTx);              // a box always delivers its full byte count (OOB = 0)
            const uint32_t dst = base + s * kStageBytes;
            tma_load_2d(dst, map_a, bar_full + 8 * s, kb * kBK, m0);
            tma_load_2d(dst + kABytes, map_b, bar_full + 8 * s, kb * kBK, n0);
          }
        } else {
          // window corner of the tile's first output pixel; the im2col box walks the next 127 by itself
          const int img = m0 / cv.HoWo, pix = m0 - img * cv.HoWo, oh = pix / cv.Wo, ow = pix - oh * cv.Wo;
          const int hb = oh * cv.sh - cv.ph, wb = ow * cv.sw - cv.pw;
          int kb = 0;
          for (int r = 0; r < cv.kh; ++r)
            for (int t = 0; t < cv.kw; ++t)
              for (int cc = 0; cc < cv.cchunks; ++cc, ++kb, ++it) {
                const uint32_t s = it % kStages, ph = (it / kStages) & 1;
                mbar_wait(bar_empty + 8 * s, ph ^ 1);
                mbar_expect_tx(bar_full + 8 * s, kTx);
                const uint32_t dst = base + s * kStageBytes;
                tma_load_im2col(dst, map_a, bar_full + 8 * s, cc * CHUNK, wb, hb, img, static_cast<uint16_t>(t * cv.dw),
                                static_cast<uint16_t>(r * cv.dh));
                tma_load_2d(dst + kABytes, map_b, bar_full + 8 * s, kb * CHUNK, n0);
              }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===== MMA issuer: one thread drives the tensor core for the whole CTA =====
      uint32_t it = 0, ti = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++ti) {
        const uint32_t ab = ti & 1, aph = (ti >> 1) & 1;
        mbar_wait(bar_acc_empty + 8 * ab, aph ^ 1);             // the epilogue has drained this accumulator buffer
        tc_fence_after();
        const uint32_t d = tmem + ab * kBN;
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const uint32_t s = it % kStages, ph = (it / kStages) & 1;
          mbar_wait(bar_full + 8 * s, ph);
          tc_fence_after();
          const uint32_t a = base + s * kStageBytes, b = a + kABytes;
          if constexpr (CHUNK == 0) {
            const int left = K - kb * kBK;                      // bytes of K beyond this block are zero-filled: skip them
            const int steps = left >= kBK ? kBK / kUmmaK : (left + kUmmaK - 1) / kUmmaK;
            for (int k = 0; k < steps; ++k)
              umma<KIND>(d, umma_desc(a + k * kUmmaK), umma_desc(b + k * kUmmaK), idesc, (kb | k) != 0 ? 1u : 0u);
          } else {                                              // a tap's channel chunk: never a K tail
#pragma unroll
            for (int k = 0; k < CHUNK / kUmmaK; ++k) {
              const uint64_t da = CHUNK == 128 ? umma_desc(a + k * kUmmaK) : umma_desc_sw64(a + k * kUmmaK);
              const uint64_t db = CHUNK == 128 ? umma_desc(b + k * kUmmaK) : umma_desc_sw64(b + k * kUmmaK);
              umma<KIND>(d, da, db, idesc, (kb | k) != 0 ? 1u : 0u);
            }
          }
          tc_commit(bar_empty + 8 * s);                         // the slot returns to the producer when these complete
        }
        tc_commit(bar_acc_full + 8 * ab);                       // ... and this tile's accumulators are final
      }
    }
  } else {
    // ===== epilogue: TMEM -> registers -> smem transpose -> 128-byte line stores =====
    constexpr bool IS_INT = KIND == DLMCQ_QGEMM_I8;
    const int ew = warp - 2;
    const int q = warp & 3;                                     // TMEM lane quarter this warp may read
    const int grp = ew >> 3;                                    // accumulator buffer / tile parity this warp serves
    const int chalf = (ew >> 2) & 1;                            // which 64 of the tile's 128 columns
    float* const stg = stg_all + ew * (32 * kStgPitch);
    if constexpr (!std::is_void<CT>::value) {
      code_epilogue_loop<IS_INT, CHUNK != 0, CT>(tmem, bar_acc_full, bar_acc_empty, stg, lane, q, grp, chalf, num_tiles,
                                                 tiles_n, M, N, alpha, beta, static_cast<uint8_t*>(out), cv, *tail);
    } else {
    const float floor = relu ? 0.f : __int_as_float(0xff800000);
    if (vec_ok && !out_bf16)
      epilogue_loop<IS_INT, 1, CHUNK != 0>(tmem, bar_acc_full, bar_acc_empty, stg, lane, q, grp, chalf, num_tiles, tiles_n, M, N,
                               alpha, beta, out, floor, out_bf16, cv);
    else if (vec_ok)
      epilogue_loop<IS_INT, 2, CHUNK != 0>(tmem, bar_acc_full, bar_acc_empty, stg, lane, q, grp, chalf, num_tiles, tiles_n, M, N,
                               alpha, beta, out, floor, out_bf16, cv);
    else
      epilogue_loop<IS_INT, 0, CHUNK != 0>(tmem, bar_acc_full, bar_acc_empty, stg, lane, q, grp, chalf, num_tiles, tiles_n, M, N,
                               alpha, beta, out, floor, out_bf16, cv);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem),
                 "r"(static_cast<uint32_t>(kTmemCols))
                 : "memory");
  }
}

template <int KIND>
__global__ void __launch_bounds__(kGemmThreads, 1)   // 576 threads: ptxas caps the kernel at 96 registers
qgemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
             const float* __restrict__ alpha, const float* __restrict__ beta, void* __restrict__ out, int M, int N,
             int K, uint32_t idesc, int relu, int out_bf16, int vec_ok) {
  gemm_pipeline<KIND, 0>(&map_a, &map_b, alpha, beta, out, M, N, K, idesc, relu, out_bf16, vec_ok, ConvArgs{});
}

// Implicit-GEMM convolution: map_a is an im2col map of the [B, H, W, Cin] codes, map_b the [n, kh*kw*Cin] weight
// codes; beta is the border-class table; out [B*Ho*Wo, n] (channels-last).
template <int KIND, int CHUNK>
__global__ void __launch_bounds__(kGemmThreads, 1)
qconv_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
             const float* __restrict__ alpha, const float* __restrict__ beta, void* __restrict__ out, int M, int N,
             int K, uint32_t idesc, int relu, int out_bf16, int vec_ok, const ConvArgs cv) {
  gemm_pipeline<KIND, CHUNK>(&map_a, &map_b, alpha, beta, out, M, N, K, idesc, relu, out_bf16, vec_ok, cv);
}

// Code output: out is the [M, N] byte matrix of the consumer's codes (code_epilogue_loop); CHUNK = 0 for the GEMM,
// 128 / 64 for the convolution (map_a, beta and cv as in qconv_kernel); T = the dtype of the unchained layer output.
template <int KIND, int CHUNK, typename T>
__global__ void __launch_bounds__(kGemmThreads, 1)
qchain_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
              const float* __restrict__ alpha, const float* __restrict__ beta, uint8_t* __restrict__ out, int M, int N,
              int K, uint32_t idesc, const ConvArgs cv, const __grid_constant__ CodeTail tail) {
  gemm_pipeline<KIND, CHUNK, T>(&map_a, &map_b, alpha, beta, out, M, N, K, idesc, 0, 0, 0, cv, &tail);
}

// ---------------------------------------------------------------------------------------------------------------
// x -> one byte per code (code_byte: codes.cuh)
// ---------------------------------------------------------------------------------------------------------------
// per-tensor, 16-byte aligned: every thread turns 16 elements into one 16-byte store (the arithmetic is fq_vec,
// i.e. bit-identical codes to dlmcq_fq_forward)
template <int FORM, typename T, int ENC>
__global__ void __launch_bounds__(kThreads, 4)
codes_flat_kernel(const T* __restrict__ x, uint8_t* __restrict__ out, int64_t n, const float* __restrict__ scale,
                  const float* __restrict__ offset, float g, float lo, float hi) {
  using V = Vec<T>;
  using raw = typename V::raw;
  constexpr int L = 16 / V::N;                                    // loads per 16 output bytes
  const ChanParams p = make_params<FORM>(scale, offset, 0, g, lo, hi);
  const int64_t groups = n / 16;
  const raw* xv = reinterpret_cast<const raw*>(x);
  uint4* ov = reinterpret_cast<uint4*>(out);
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t gi = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; gi < groups; gi += stride) {
    raw r[L];
#pragma unroll
    for (int k = 0; k < L; ++k) r[k] = ld_stream(xv + gi * L + k);
    uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int k = 0; k < L; ++k) {
      float f[V::N], fy[V::N], fc[V::N];
      V::unpack(r[k], f);
      fq_vec<FORM, V::N>(f, p, lo, hi, fc, fy);
#pragma unroll
      for (int e = 0; e < V::N; ++e) {
        const int b = k * V::N + e;
        w[b >> 2] |= code_byte<ENC>(fc[e]) << (8 * (b & 3));
      }
    }
    ov[gi] = make_uint4(w[0], w[1], w[2], w[3]);
  }
  if (blockIdx.x == 0) {                                          // ragged tail (< 16 elements)
    const int64_t t = groups * 16 + threadIdx.x;
    if (threadIdx.x < 16 && t < n) {
      float c, v;
      fq_elem_ref<FORM>(to_f32<T>(x[t]), p, lo, hi, c, v);
      out[t] = static_cast<uint8_t>(code_byte<ENC>(c));
    }
  }
}

// any layout / alignment (per-channel weights: a one-off per weight update)
template <int FORM, typename T, int ENC>
__global__ void __launch_bounds__(kThreads)
codes_any_kernel(const T* __restrict__ x, uint8_t* __restrict__ out, int64_t n, int64_t channels, int64_t inner,
                 const float* __restrict__ scale, const float* __restrict__ offset, float g, float lo, float hi) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    const int64_t ch = channels == 1 ? 0 : (i / inner) % channels;
    const ChanParams p = make_params<FORM>(scale, offset, ch, g, lo, hi);
    float c, v;
    fq_elem_ref<FORM>(to_f32<T>(x[i]), p, lo, hi, c, v);
    out[i] = static_cast<uint8_t>(code_byte<ENC>(c));
  }
}

template <int FORM, typename T, int ENC>
int codes_launch(const void* x, void* out, const dlmcq_layout* l, const dlmcq_qparams* qp, cudaStream_t st) {
  const int64_t n = l->outer * l->channels * l->inner;
  const float lo = static_cast<float>(qp->lo), hi = static_cast<float>(qp->hi);
  if (l->channels == 1 && aligned16(x) && aligned16(out)) {
    const int64_t tiles = (n / 16 + kThreads - 1) / kThreads;
    codes_flat_kernel<FORM, T, ENC><<<stream_grid(tiles, 16), kThreads, 0, st>>>(
        static_cast<const T*>(x), static_cast<uint8_t*>(out), n, qp->scale, qp->offset, qp->g, lo, hi);
  } else {
    const int64_t tiles = (n + kThreads - 1) / kThreads;
    codes_any_kernel<FORM, T, ENC><<<stream_grid(tiles, 8), kThreads, 0, st>>>(
        static_cast<const T*>(x), static_cast<uint8_t*>(out), n, l->channels, l->inner, qp->scale, qp->offset, qp->g,
        lo, hi);
  }
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

template <typename T, int ENC>
int codes_form(const void* x, void* out, const dlmcq_layout* l, const dlmcq_qparams* qp, cudaStream_t st) {
  switch (qp->form) {
    case DLMCQ_FORM_A1: return codes_launch<DLMCQ_FORM_A1, T, ENC>(x, out, l, qp, st);
    case DLMCQ_FORM_AFFINE: return codes_launch<DLMCQ_FORM_AFFINE, T, ENC>(x, out, l, qp, st);
    case DLMCQ_FORM_ZP: return codes_launch<DLMCQ_FORM_ZP, T, ENC>(x, out, l, qp, st);
    case DLMCQ_FORM_SYM: return codes_launch<DLMCQ_FORM_SYM, T, ENC>(x, out, l, qp, st);
  }
  return DLMCQ_EINVAL;
}

// Exactness of the accumulation: every partial sum of k products is at most k * max|a| * max|w|.  The fp32
// accumulators of kind::f8f6f4 hold every integer up to 2^24, the s32 accumulators of kind::i8 up to 2^31 - 1.
// Call after code_range_ok (|code| <= 255).
int accumulator_ok(int64_t k, const dlmcq_qparams* act_qp, const dlmcq_qparams* wt_qp, int encoding) {
  const int64_t ma = act_qp->hi > -act_qp->lo ? act_qp->hi : -act_qp->lo;
  const int64_t mw = wt_qp->hi > -wt_qp->lo ? wt_qp->hi : -wt_qp->lo;
  const int64_t bound = encoding == DLMCQ_QGEMM_E4M3 ? (1LL << 24) : 0x7fffffffLL;
  return (ma * mw == 0 || k <= bound / (ma * mw)) ? DLMCQ_OK : DLMCQ_EUNSUPPORTED;
}

// ---------------------------------------------------------------------------------------------------------------
// alpha[n], beta[n] from the device-resident quantizer parameters; one warp per output channel
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ ChanParams params_of(int form, const float* scale, const float* offset, int64_t ch, float g,
                                                float lo, float hi) {
  switch (form) {
    case DLMCQ_FORM_A1: return make_params<DLMCQ_FORM_A1>(scale, offset, ch, g, lo, hi);
    case DLMCQ_FORM_AFFINE: return make_params<DLMCQ_FORM_AFFINE>(scale, offset, ch, g, lo, hi);
    case DLMCQ_FORM_ZP: return make_params<DLMCQ_FORM_ZP>(scale, offset, ch, g, lo, hi);
    default: return make_params<DLMCQ_FORM_SYM>(scale, offset, ch, g, lo, hi);
  }
}

__device__ __forceinline__ int decode_code(uint8_t b, int encoding, int is_signed) {
  if (encoding == DLMCQ_QGEMM_E4M3) {
    // small integers only: sign | exponent(4, bias 7) | mantissa(3)
    const int e = (b >> 3) & 0xF, m = b & 7;
    const float mag = e == 0 ? static_cast<float>(m) * 0.001953125f : ldexpf(1.f + static_cast<float>(m) * 0.125f, e - 7);
    const int v = static_cast<int>(mag);
    return (b & 0x80) ? -v : v;
  }
  return is_signed ? static_cast<int>(static_cast<int8_t>(b)) : static_cast<int>(b);
}

__global__ void __launch_bounds__(kRowWarps * 32)
qgemm_prepare_kernel(const uint8_t* __restrict__ w_codes, int64_t n, int64_t k, int encoding, int act_form,
                     const float* __restrict__ act_scale, const float* __restrict__ act_offset, float act_g,
                     float act_lo, float act_hi, int wt_form, const float* __restrict__ wt_scale, float wt_g,
                     float wt_lo, float wt_hi, int64_t wt_channels, const float* __restrict__ bias,
                     float* __restrict__ alpha, float* __restrict__ beta) {
  const int lane = threadIdx.x & 31;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * kRowWarps + (threadIdx.x >> 5);
  if (row >= n) return;
  int sum = 0;
  const uint8_t* wr = w_codes + row * k;
  for (int64_t i = lane; i < k; i += 32) sum += decode_code(wr[i], encoding, wt_lo < 0.f);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if (lane == 0) {
    const ChanParams pa = params_of(act_form, act_scale, act_offset, 0, act_g, act_lo, act_hi);
    const ChanParams pw = params_of(wt_form, wt_scale, nullptr, wt_channels == 1 ? 0 : row, wt_g, wt_lo, wt_hi);
    const float z_a = act_form == DLMCQ_FORM_ZP ? pa.off : 0.f;
    const float o_a = (act_form == DLMCQ_FORM_A1 || act_form == DLMCQ_FORM_AFFINE) ? pa.off : 0.f;
    const float t = __fsub_rn(o_a, __fmul_rn(z_a, pa.mul));
    alpha[row] = __fmul_rn(pa.mul, pw.mul);
    float b = __fmul_rn(__fmul_rn(t, pw.mul), static_cast<float>(sum));
    if (bias) b = __fadd_rn(b, __ldg(bias + row));
    beta[row] = b;
  }
}

// Convolution: alpha[n] as above; beta for every border class of output pixel.  One block per output channel: the
// per-tap code sums S[r][s] = sum_c cw[n, r, s, c] go to smem, then every class (r_lo, r_hi1, s_lo, s_hi1) - the
// taps of the window that lie inside the image, each range in [0, k] - gets
//     beta[class][n] = RN(RN(t * m_w[n]) * float(sum_{r_lo <= r < r_hi1, s_lo <= s < s_hi1} S[r][s]))  (+ bias[n])
// class = ((r_lo*(kh+1) + r_hi1)*(kw+1) + s_lo)*(kw+1) + s_hi1: the epilogue's conv_beta_offset.
constexpr int kConvPrepThreads = 128;

__global__ void __launch_bounds__(kConvPrepThreads)
qconv_prepare_kernel(const uint8_t* __restrict__ w_codes, int64_t n, int cin, int kh, int kw, int encoding, int act_form,
                     const float* __restrict__ act_scale, const float* __restrict__ act_offset, float act_g,
                     float act_lo, float act_hi, int wt_form, const float* __restrict__ wt_scale, float wt_g,
                     float wt_lo, float wt_hi, int64_t wt_channels, const float* __restrict__ bias,
                     float* __restrict__ alpha, float* __restrict__ beta) {
  extern __shared__ int tap_sum[];
  const int64_t row = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, taps = kh * kw;
  const uint8_t* wr = w_codes + row * static_cast<int64_t>(taps) * cin;
  for (int tap = warp; tap < taps; tap += kConvPrepThreads / 32) {
    int sum = 0;
    for (int c = lane; c < cin; c += 32) sum += decode_code(wr[static_cast<int64_t>(tap) * cin + c], encoding, wt_lo < 0.f);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) tap_sum[tap] = sum;
  }
  __syncthreads();
  const ChanParams pa = params_of(act_form, act_scale, act_offset, 0, act_g, act_lo, act_hi);
  const ChanParams pw = params_of(wt_form, wt_scale, nullptr, wt_channels == 1 ? 0 : row, wt_g, wt_lo, wt_hi);
  const float z_a = act_form == DLMCQ_FORM_ZP ? pa.off : 0.f;
  const float o_a = (act_form == DLMCQ_FORM_A1 || act_form == DLMCQ_FORM_AFFINE) ? pa.off : 0.f;
  const float tm = __fmul_rn(__fsub_rn(o_a, __fmul_rn(z_a, pa.mul)), pw.mul);
  const float bn = bias ? __ldg(bias + row) : 0.f;
  if (threadIdx.x == 0) alpha[row] = __fmul_rn(pa.mul, pw.mul);
  const int classes = (kh + 1) * (kh + 1) * (kw + 1) * (kw + 1);
  for (int cls = threadIdx.x; cls < classes; cls += kConvPrepThreads) {
    const int sh1 = cls % (kw + 1), sl = (cls / (kw + 1)) % (kw + 1);
    const int rh1 = (cls / ((kw + 1) * (kw + 1))) % (kh + 1), rl = cls / ((kw + 1) * (kw + 1) * (kh + 1));
    int sum = 0;
    for (int r = rl; r < rh1; ++r)
      for (int t = sl; t < sh1; ++t) sum += tap_sum[r * kw + t];
    float b = __fmul_rn(tm, static_cast<float>(sum));
    if (bias) b = __fadd_rn(b, bn);
    beta[static_cast<int64_t>(cls) * n + row] = b;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// host side: tensor maps
// ---------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled() {
  static const EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

// [rows, k] bytes, row-major (K-major): box = box_k (128 or 64) bytes of K x 128 rows, swizzle of the same width,
// out-of-bounds = 0
bool make_map(CUtensorMap* m, const void* ptr, int64_t rows, int64_t k, int box_rows, int box_k = kBK) {
  EncodeTiledFn enc = encode_tiled();
  if (!enc) return false;
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(k), static_cast<cuuint64_t>(rows)};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(k)};
  const cuuint32_t box[2] = {static_cast<cuuint32_t>(box_k), static_cast<cuuint32_t>(box_rows)};
  const cuuint32_t estr[2] = {1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(ptr), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, box_k == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*,
                                   CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                   CUtensorMapFloatOOBfill);

EncodeIm2colFn encode_im2col() {
  static const EncodeIm2colFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return reinterpret_cast<EncodeIm2colFn>(p);
  }();
  return fn;
}

// Channels-last codes [B, H, W, Cin] as an im2col map: 128 pixels x `chunk` channels per box.  The bounding box of
// window corners is [-pad, size - 1 + pad - dil*(k-1)] per spatial axis, walked with the convolution's stride, so the
// box's pixels are exactly the output pixels in N*Ho*Wo order.  Arrays are innermost first (C, W, H, N).
bool make_im2col_map(CUtensorMap* m, const void* ptr, const dlmcq_conv_geom* g, int chunk) {
  EncodeIm2colFn enc = encode_im2col();
  if (!enc) return false;
  const cuuint64_t dims[4] = {static_cast<cuuint64_t>(g->cin), static_cast<cuuint64_t>(g->w),
                              static_cast<cuuint64_t>(g->h), static_cast<cuuint64_t>(g->batch)};
  const cuuint64_t strides[3] = {static_cast<cuuint64_t>(g->cin), static_cast<cuuint64_t>(g->cin * g->w),
                                 static_cast<cuuint64_t>(g->cin * g->w * g->h)};
  const int lower[2] = {-g->pad_w, -g->pad_h};
  const int upper[2] = {g->pad_w - g->dil_w * (g->kw - 1), g->pad_h - g->dil_h * (g->kh - 1)};
  const cuuint32_t estr[4] = {1, static_cast<cuuint32_t>(g->stride_w), static_cast<cuuint32_t>(g->stride_h), 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, const_cast<void*>(ptr), dims, strides, lower, upper,
             static_cast<cuuint32_t>(chunk), static_cast<cuuint32_t>(kBM), estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             chunk == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// tcgen05 instruction descriptor: D format [4,6), A format [7,10), B format [10,13), A/B K-major (bits 15, 16 = 0),
// N >> 3 at [17,23), M >> 4 at [24,29)
uint32_t make_idesc(int encoding, int a_signed) {
  uint32_t d = 0;
  if (encoding == DLMCQ_QGEMM_I8) {
    d |= 2u << 4;                              // D = s32
    d |= (a_signed ? 1u : 0u) << 7;            // A = s8 | u8
    d |= 1u << 10;                             // B = s8
  } else {
    d |= 1u << 4;                              // D = f32; A = B = e4m3 (format 0)
  }
  d |= static_cast<uint32_t>(kBN >> 3) << 17;
  d |= static_cast<uint32_t>(kBM >> 4) << 24;
  return d;
}

template <int KIND>
int gemm_launch(const CUtensorMap& ma, const CUtensorMap& mb, const float* alpha, const float* beta, void* out, int m,
                int n, int k, int a_signed, int relu, int out_bf16, cudaStream_t st) {
  static bool opted_in[64] = {};                               // the attribute is per device
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
  if (dev < 0 || dev >= 64 || !opted_in[dev]) {
    const cudaError_t e = cudaFuncSetAttribute(qgemm_kernel<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               static_cast<int>(kGemmSmem));
    if (e != cudaSuccess) return set_cuda_error(e);
    if (dev >= 0 && dev < 64) opted_in[dev] = true;
  }
  const int64_t tiles = static_cast<int64_t>((n + kBN - 1) / kBN) * ((m + kBM - 1) / kBM);
  const int sms = num_sms();
  const unsigned grid = static_cast<unsigned>(tiles < sms ? tiles : sms);      // persistent: one CTA per SM
  // 16-byte row stores need every row start aligned: N a multiple of 4 (fp32) / 8 (bf16) and an aligned base
  const int vec_ok = aligned16(out) && (n % (out_bf16 ? 8 : 4) == 0);
  qgemm_kernel<KIND><<<grid, kGemmThreads, kGemmSmem, st>>>(ma, mb, alpha, beta, out, m, n, k,
                                                            make_idesc(KIND, a_signed), relu, out_bf16, vec_ok);
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

template <int KIND, int CHUNK>
int conv_launch(const CUtensorMap& ma, const CUtensorMap& mb, const float* alpha, const float* beta, void* out, int m,
                int n, int k, const ConvArgs& cv, int a_signed, int relu, int out_bf16, cudaStream_t st) {
  static bool opted_in[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
  if (dev < 0 || dev >= 64 || !opted_in[dev]) {
    const cudaError_t e = cudaFuncSetAttribute(qconv_kernel<KIND, CHUNK>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               static_cast<int>(kGemmSmem));
    if (e != cudaSuccess) return set_cuda_error(e);
    if (dev >= 0 && dev < 64) opted_in[dev] = true;
  }
  const int64_t tiles = static_cast<int64_t>((n + kBN - 1) / kBN) * ((m + kBM - 1) / kBM);
  const int sms = num_sms();
  const unsigned grid = static_cast<unsigned>(tiles < sms ? tiles : sms);
  // the beta table is read with 16-byte loads in the vector epilogues: its rows start at multiples of n
  const int vec_ok = aligned16(out) && aligned16(beta) && (n % (out_bf16 ? 8 : 4) == 0);
  qconv_kernel<KIND, CHUNK><<<grid, kGemmThreads, kGemmSmem, st>>>(ma, mb, alpha, beta, out, m, n, k,
                                                                   make_idesc(KIND, a_signed), relu, out_bf16, vec_ok, cv);
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

template <int KIND, int CHUNK, typename T>
int chain_launch(const CUtensorMap& ma, const CUtensorMap& mb, const float* alpha, const float* beta, void* out, int m,
                 int n, int k, const ConvArgs& cv, int a_signed, const CodeTail& t, cudaStream_t st) {
  static bool opted_in[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
  if (dev < 0 || dev >= 64 || !opted_in[dev]) {
    const cudaError_t e = cudaFuncSetAttribute(qchain_kernel<KIND, CHUNK, T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               static_cast<int>(kGemmSmem));
    if (e != cudaSuccess) return set_cuda_error(e);
    if (dev >= 0 && dev < 64) opted_in[dev] = true;
  }
  const int64_t tiles = static_cast<int64_t>((n + kBN - 1) / kBN) * ((m + kBM - 1) / kBM);
  const int sms = num_sms();
  const unsigned grid = static_cast<unsigned>(tiles < sms ? tiles : sms);
  qchain_kernel<KIND, CHUNK, T><<<grid, kGemmThreads, kGemmSmem, st>>>(ma, mb, alpha, beta, static_cast<uint8_t*>(out), m, n,
                                                                      k, make_idesc(KIND, a_signed), cv, t);
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

template <int CHUNK>
int chain_dispatch(int encoding, int inter_bf16, const CUtensorMap& ma, const CUtensorMap& mb, const float* alpha,
                   const float* beta, void* out, int m, int n, int k, const ConvArgs& cv, int a_signed,
                   const CodeTail& t, cudaStream_t st) {
  if (encoding == DLMCQ_QGEMM_I8)
    return inter_bf16 ? chain_launch<DLMCQ_QGEMM_I8, CHUNK, __nv_bfloat16>(ma, mb, alpha, beta, out, m, n, k, cv, a_signed, t, st)
                      : chain_launch<DLMCQ_QGEMM_I8, CHUNK, float>(ma, mb, alpha, beta, out, m, n, k, cv, a_signed, t, st);
  return inter_bf16 ? chain_launch<DLMCQ_QGEMM_E4M3, CHUNK, __nv_bfloat16>(ma, mb, alpha, beta, out, m, n, k, cv, a_signed, t, st)
                    : chain_launch<DLMCQ_QGEMM_E4M3, CHUNK, float>(ma, mb, alpha, beta, out, m, n, k, cv, a_signed, t, st);
}

// The tail's own refusals (dlmcq_qgemm_codes / dlmcq_qconv_codes), before any CUDA call.
int tail_check(const dlmcq_bnq_tail* t) {
  if (!t || !t->running_mean || !t->running_var || !t->qp) return DLMCQ_EINVAL;
  if (!t->qp->scale || t->qp->form != DLMCQ_FORM_AFFINE) return DLMCQ_EINVAL;
  if (t->inter_dtype != DLMCQ_F32 && t->inter_dtype != DLMCQ_BF16) return DLMCQ_EINVAL;
  return code_range_ok(t->qp, t->encoding);                   // unknown encoding: DLMCQ_EINVAL
}

CodeTail make_tail(const dlmcq_bnq_tail* t) {
  CodeTail c;
  c.gamma = t->gamma;
  c.beta = t->beta;
  c.mean = t->running_mean;
  c.var = t->running_var;
  c.scale = t->qp->scale;
  c.offset = t->qp->offset;
  c.eps = t->eps;
  c.g = t->qp->g;
  c.lo = static_cast<float>(t->qp->lo);
  c.hi = static_cast<float>(t->qp->hi);
  c.relu = t->relu != 0;
  c.enc = t->encoding;
  return c;
}

// Geometry checks shared by dlmcq_qconv_prepare (full = 0: only the filter and channel counts) and dlmcq_qconv.
int conv_check(const dlmcq_conv_geom* g, int full, int64_t* ho, int64_t* wo) {
  if (!g || g->cin < 1 || g->n < 1 || g->kh < 1 || g->kw < 1 || g->groups < 1) return DLMCQ_EINVAL;
  if (g->groups != 1 || g->cin % 64 != 0) return DLMCQ_EUNSUPPORTED;
  const int64_t k = static_cast<int64_t>(g->kh) * g->kw * g->cin;
  const int64_t classes = static_cast<int64_t>(g->kh + 1) * (g->kh + 1) * (g->kw + 1) * (g->kw + 1);
  if (g->kh > 255 || g->kw > 255 || k > 0x7fffff00LL || g->n > 0x7fffff00LL || classes * g->n > 0x7fffffffLL)
    return DLMCQ_EUNSUPPORTED;
  if (!full) return DLMCQ_OK;
  if (g->batch < 1 || g->h < 1 || g->w < 1 || g->stride_h < 1 || g->stride_w < 1 || g->pad_h < 0 || g->pad_w < 0 ||
      g->dil_h < 1 || g->dil_w < 1)
    return DLMCQ_EINVAL;
  const int64_t eh = static_cast<int64_t>(g->dil_h) * (g->kh - 1), ew = static_cast<int64_t>(g->dil_w) * (g->kw - 1);
  if (g->h + 2LL * g->pad_h - eh < 1 || g->w + 2LL * g->pad_w - ew < 1) return DLMCQ_EINVAL;   // no output pixel
  *ho = (g->h + 2LL * g->pad_h - eh - 1) / g->stride_h + 1;
  *wo = (g->w + 2LL * g->pad_w - ew - 1) / g->stride_w + 1;
  // TMA im2col limits: traversal stride <= 8, bounding-box corners -pad and pad - dil*(k-1) in [-128, 127]
  if (g->stride_h > 8 || g->stride_w > 8 || g->pad_h > 128 || g->pad_w > 128 || g->pad_h - eh < -128 ||
      g->pad_w - ew < -128 || g->pad_h - eh > 127 || g->pad_w - ew > 127)
    return DLMCQ_EUNSUPPORTED;
  // 32-bit coordinates and row indices
  const int64_t m = g->batch * *ho * *wo;
  if (g->batch > 0x7fffffffLL || g->h > 0x7fffffffLL || g->w > 0x7fffffffLL || m > 0x7fffff00LL ||
      g->h * g->w > (1LL << 40) / g->cin)                         // TMA strides < 2^40 bytes
    return DLMCQ_EUNSUPPORTED;
  if (((m + kBM - 1) / kBM) * ((g->n + kBN - 1) / kBN) > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
  return DLMCQ_OK;
}

ConvArgs conv_args(const dlmcq_conv_geom* geom, int64_t ho, int64_t wo, int chunk) {
  ConvArgs cv;
  cv.H = static_cast<int>(geom->h); cv.W = static_cast<int>(geom->w);
  cv.Ho = static_cast<int>(ho); cv.Wo = static_cast<int>(wo); cv.HoWo = static_cast<int>(ho * wo);
  cv.kh = geom->kh; cv.kw = geom->kw; cv.sh = geom->stride_h; cv.sw = geom->stride_w;
  cv.ph = geom->pad_h; cv.pw = geom->pad_w; cv.dh = geom->dil_h; cv.dw = geom->dil_w;
  cv.cchunks = static_cast<int>(geom->cin / chunk);
  return cv;
}

}  // namespace
}  // namespace dlmcq

using namespace dlmcq;

extern "C" int dlmcq_codes_forward(const void* x, void* codes, const dlmcq_layout* layout, const dlmcq_qparams* qp,
                                   int encoding, void* stream) {
  if (!layout || !qp || !qp->scale || layout->outer < 1 || layout->channels < 1 || layout->inner < 0) return DLMCQ_EINVAL;
  if (layout->dtype != DLMCQ_F32 && layout->dtype != DLMCQ_BF16) return DLMCQ_EINVAL;
  if (int e = code_range_ok(qp, encoding)) return e;
  if (layout->outer * layout->channels * layout->inner == 0) return DLMCQ_OK;
  if (!x || !codes) return DLMCQ_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (layout->dtype == DLMCQ_F32)
    return encoding == DLMCQ_QGEMM_I8 ? codes_form<float, DLMCQ_QGEMM_I8>(x, codes, layout, qp, st)
                                      : codes_form<float, DLMCQ_QGEMM_E4M3>(x, codes, layout, qp, st);
  return encoding == DLMCQ_QGEMM_I8 ? codes_form<__nv_bfloat16, DLMCQ_QGEMM_I8>(x, codes, layout, qp, st)
                                    : codes_form<__nv_bfloat16, DLMCQ_QGEMM_E4M3>(x, codes, layout, qp, st);
}

extern "C" int dlmcq_qgemm_prepare(const void* w_codes, int64_t n, int64_t k, int encoding, const dlmcq_qparams* act_qp,
                                   const dlmcq_qparams* wt_qp, int64_t wt_channels, const float* bias, float* alpha,
                                   float* beta, void* stream) {
  if (!w_codes || !act_qp || !wt_qp || !act_qp->scale || !wt_qp->scale || !alpha || !beta || n < 1 || k < 1)
    return DLMCQ_EINVAL;
  if (wt_channels != 1 && wt_channels != n) return DLMCQ_EINVAL;
  if (int e = code_range_ok(act_qp, encoding)) return e;
  if (int e = code_range_ok(wt_qp, encoding)) return e;
  // the product only factors for weights without an additive term: y_w = code * m_w
  if (wt_qp->form == DLMCQ_FORM_ZP || wt_qp->offset != nullptr) return DLMCQ_EUNSUPPORTED;
  if (encoding == DLMCQ_QGEMM_I8 && wt_qp->lo >= 0 && wt_qp->hi > 127) return DLMCQ_EUNSUPPORTED;   // B operand is s8
  if (int e = accumulator_ok(k, act_qp, wt_qp, encoding)) return e;
  const int64_t blocks = (n + kRowWarps - 1) / kRowWarps;
  if (blocks > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
  qgemm_prepare_kernel<<<static_cast<unsigned>(blocks), kRowWarps * 32, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint8_t*>(w_codes), n, k, encoding, act_qp->form, act_qp->scale, act_qp->offset, act_qp->g,
      static_cast<float>(act_qp->lo), static_cast<float>(act_qp->hi), wt_qp->form, wt_qp->scale, wt_qp->g,
      static_cast<float>(wt_qp->lo), static_cast<float>(wt_qp->hi), wt_channels, bias, alpha, beta);
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

extern "C" int dlmcq_qgemm(const void* a_codes, const void* w_codes, const float* alpha, const float* beta, void* out,
                           int64_t m, int64_t n, int64_t k, int encoding, int a_signed, int relu, int out_dtype,
                           void* stream) {
  if (m < 0 || n < 1 || k < 1 || !alpha || !beta) return DLMCQ_EINVAL;
  if (encoding != DLMCQ_QGEMM_I8 && encoding != DLMCQ_QGEMM_E4M3) return DLMCQ_EINVAL;
  if (out_dtype != DLMCQ_F32 && out_dtype != DLMCQ_BF16) return DLMCQ_EINVAL;
  if (m == 0) return DLMCQ_OK;
  if (!a_codes || !w_codes || !out) return DLMCQ_EINVAL;
  // TMA: 16-byte aligned base addresses and row pitch; 32-bit tile coordinates
  if (!aligned16(a_codes) || !aligned16(w_codes)) return DLMCQ_EALIGN;
  if ((k & 15) != 0 || m > 0x7fffff00LL || n > 0x7fffff00LL || k > 0x7fffff00LL) return DLMCQ_EUNSUPPORTED;
  if (((m + kBM - 1) / kBM) * ((n + kBN - 1) / kBN) > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
  CUtensorMap ma, mb;
  if (!make_map(&ma, a_codes, m, k, kBM) || !make_map(&mb, w_codes, n, k, kBN)) return DLMCQ_EUNSUPPORTED;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int bf = out_dtype == DLMCQ_BF16;
  return encoding == DLMCQ_QGEMM_I8
             ? gemm_launch<DLMCQ_QGEMM_I8>(ma, mb, alpha, beta, out, static_cast<int>(m), static_cast<int>(n),
                                           static_cast<int>(k), a_signed, relu, bf, st)
             : gemm_launch<DLMCQ_QGEMM_E4M3>(ma, mb, alpha, beta, out, static_cast<int>(m), static_cast<int>(n),
                                             static_cast<int>(k), a_signed, relu, bf, st);
}

extern "C" int dlmcq_qconv_prepare(const void* w_codes, const dlmcq_conv_geom* geom, int encoding,
                                   const dlmcq_qparams* act_qp, const dlmcq_qparams* wt_qp, int64_t wt_channels,
                                   const float* bias, float* alpha, float* beta, void* stream) {
  if (!w_codes || !act_qp || !wt_qp || !act_qp->scale || !wt_qp->scale || !alpha || !beta) return DLMCQ_EINVAL;
  int64_t ho = 0, wo = 0;
  if (int e = conv_check(geom, 0, &ho, &wo)) return e;
  const int64_t n = geom->n;
  if (wt_channels != 1 && wt_channels != n) return DLMCQ_EINVAL;
  if (int e = code_range_ok(act_qp, encoding)) return e;
  if (int e = code_range_ok(wt_qp, encoding)) return e;
  if (wt_qp->form == DLMCQ_FORM_ZP || wt_qp->offset != nullptr) return DLMCQ_EUNSUPPORTED;
  if (encoding == DLMCQ_QGEMM_I8 && wt_qp->lo >= 0 && wt_qp->hi > 127) return DLMCQ_EUNSUPPORTED;
  if (int e = accumulator_ok(static_cast<int64_t>(geom->kh) * geom->kw * geom->cin, act_qp, wt_qp, encoding)) return e;
  const size_t smem = static_cast<size_t>(geom->kh) * geom->kw * sizeof(int);
  if (smem > 48 * 1024) return DLMCQ_EUNSUPPORTED;
  qconv_prepare_kernel<<<static_cast<unsigned>(n), kConvPrepThreads, smem, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint8_t*>(w_codes), n, static_cast<int>(geom->cin), geom->kh, geom->kw, encoding, act_qp->form,
      act_qp->scale, act_qp->offset, act_qp->g, static_cast<float>(act_qp->lo), static_cast<float>(act_qp->hi),
      wt_qp->form, wt_qp->scale, wt_qp->g, static_cast<float>(wt_qp->lo), static_cast<float>(wt_qp->hi), wt_channels,
      bias, alpha, beta);
  DLMCQ_LAUNCH_CHECK();
  return DLMCQ_OK;
}

extern "C" int dlmcq_qconv(const void* a_codes, const void* w_codes, const float* alpha, const float* beta, void* out,
                           const dlmcq_conv_geom* geom, int encoding, int a_signed, int relu, int out_dtype,
                           void* stream) {
  if (!alpha || !beta) return DLMCQ_EINVAL;
  if (encoding != DLMCQ_QGEMM_I8 && encoding != DLMCQ_QGEMM_E4M3) return DLMCQ_EINVAL;
  if (out_dtype != DLMCQ_F32 && out_dtype != DLMCQ_BF16) return DLMCQ_EINVAL;
  int64_t ho = 0, wo = 0;
  if (int e = conv_check(geom, 1, &ho, &wo)) return e;
  if (!a_codes || !w_codes || !out) return DLMCQ_EINVAL;
  if (!aligned16(a_codes) || !aligned16(w_codes)) return DLMCQ_EALIGN;
  const int chunk = geom->cin % 128 == 0 ? 128 : 64;
  CUtensorMap ma, mb;
  const int64_t k = static_cast<int64_t>(geom->kh) * geom->kw * geom->cin;
  if (!make_im2col_map(&ma, a_codes, geom, chunk) || !make_map(&mb, w_codes, geom->n, k, kBN, chunk))
    return DLMCQ_EUNSUPPORTED;
  const ConvArgs cv = conv_args(geom, ho, wo, chunk);
  const int m = static_cast<int>(geom->batch * ho * wo), n = static_cast<int>(geom->n);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int bf = out_dtype == DLMCQ_BF16;
  if (encoding == DLMCQ_QGEMM_I8)
    return chunk == 128 ? conv_launch<DLMCQ_QGEMM_I8, 128>(ma, mb, alpha, beta, out, m, n, static_cast<int>(k), cv, a_signed, relu, bf, st)
                        : conv_launch<DLMCQ_QGEMM_I8, 64>(ma, mb, alpha, beta, out, m, n, static_cast<int>(k), cv, a_signed, relu, bf, st);
  return chunk == 128 ? conv_launch<DLMCQ_QGEMM_E4M3, 128>(ma, mb, alpha, beta, out, m, n, static_cast<int>(k), cv, a_signed, relu, bf, st)
                      : conv_launch<DLMCQ_QGEMM_E4M3, 64>(ma, mb, alpha, beta, out, m, n, static_cast<int>(k), cv, a_signed, relu, bf, st);
}

extern "C" int dlmcq_qgemm_codes(const void* a_codes, const void* w_codes, const float* alpha, const float* beta,
                                 void* codes_out, int64_t m, int64_t n, int64_t k, int encoding, int a_signed,
                                 const dlmcq_bnq_tail* tail, void* stream) {
  if (m < 0 || n < 1 || k < 1 || !alpha || !beta) return DLMCQ_EINVAL;
  if (encoding != DLMCQ_QGEMM_I8 && encoding != DLMCQ_QGEMM_E4M3) return DLMCQ_EINVAL;
  if (int e = tail_check(tail)) return e;
  if (n % 16 != 0) return DLMCQ_EUNSUPPORTED;                  // whole 16-byte code stores per row piece
  if (m == 0) return DLMCQ_OK;
  if (!a_codes || !w_codes || !codes_out) return DLMCQ_EINVAL;
  if (!aligned16(a_codes) || !aligned16(w_codes) || !aligned16(codes_out)) return DLMCQ_EALIGN;
  if ((k & 15) != 0 || m > 0x7fffff00LL || n > 0x7fffff00LL || k > 0x7fffff00LL) return DLMCQ_EUNSUPPORTED;
  if (((m + kBM - 1) / kBM) * ((n + kBN - 1) / kBN) > 0x7fffffffLL) return DLMCQ_EUNSUPPORTED;
  CUtensorMap ma, mb;
  if (!make_map(&ma, a_codes, m, k, kBM) || !make_map(&mb, w_codes, n, k, kBN)) return DLMCQ_EUNSUPPORTED;
  return chain_dispatch<0>(encoding, tail->inter_dtype == DLMCQ_BF16, ma, mb, alpha, beta, codes_out,
                           static_cast<int>(m), static_cast<int>(n), static_cast<int>(k), ConvArgs{}, a_signed,
                           make_tail(tail), static_cast<cudaStream_t>(stream));
}

extern "C" int dlmcq_qconv_codes(const void* a_codes, const void* w_codes, const float* alpha, const float* beta,
                                 void* codes_out, const dlmcq_conv_geom* geom, int encoding, int a_signed,
                                 const dlmcq_bnq_tail* tail, void* stream) {
  if (!alpha || !beta) return DLMCQ_EINVAL;
  if (encoding != DLMCQ_QGEMM_I8 && encoding != DLMCQ_QGEMM_E4M3) return DLMCQ_EINVAL;
  if (int e = tail_check(tail)) return e;
  int64_t ho = 0, wo = 0;
  if (int e = conv_check(geom, 1, &ho, &wo)) return e;
  if (geom->n % 16 != 0) return DLMCQ_EUNSUPPORTED;
  if (!a_codes || !w_codes || !codes_out) return DLMCQ_EINVAL;
  if (!aligned16(a_codes) || !aligned16(w_codes) || !aligned16(codes_out)) return DLMCQ_EALIGN;
  const int chunk = geom->cin % 128 == 0 ? 128 : 64;
  CUtensorMap ma, mb;
  const int64_t k = static_cast<int64_t>(geom->kh) * geom->kw * geom->cin;
  if (!make_im2col_map(&ma, a_codes, geom, chunk) || !make_map(&mb, w_codes, geom->n, k, kBN, chunk))
    return DLMCQ_EUNSUPPORTED;
  const ConvArgs cv = conv_args(geom, ho, wo, chunk);
  const int m = static_cast<int>(geom->batch * ho * wo), n = static_cast<int>(geom->n);
  const int bf = tail->inter_dtype == DLMCQ_BF16;
  const CodeTail t = make_tail(tail);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return chunk == 128 ? chain_dispatch<128>(encoding, bf, ma, mb, alpha, beta, codes_out, m, n, static_cast<int>(k), cv,
                                            a_signed, t, st)
                      : chain_dispatch<64>(encoding, bf, ma, mb, alpha, beta, codes_out, m, n, static_cast<int>(k), cv,
                                           a_signed, t, st);
}
