// bnq_kernels.cu - the activation fake-quant fused into its PRODUCER (SURVEY.md 8f row f2):
//
//     conv output x --BatchNorm--(+ residual)--(ReLU)--> a --QBase fake-quant--> a_q --> next QConv
//
// In the reference this is nn.BatchNorm2d -> (+=) -> nn.ReLU -> QBase.forward's input branch
// (dlmc/quantization/scalar/modules/base.py:96-102, entered from modules/conv.py:13-19): four separate passes over
// the activation per direction (cuDNN batch-norm 12 B/elem, add 12, ReLU 8, the eager fake-quant chain ~70) and
// their autograd mirror images.  Here the whole chain is
//     forward  : one statistics pass (read x: 4 B/elem) + one apply pass (read x [, identity]; write a_q [, a])
//     backward : one reduction pass (d gamma, d beta, d in_scale) + one pass that writes dx
// i.e. 12 + 20 = 32 B/elem for the plain chain including the quantizer, against 52 B/elem for an UN-quantised
// BatchNorm + ReLU in a library implementation.  Nothing here is a contraction: HBM-bound, no tensor cores.
//
// Layout: channels-last.  The tensor is a dense [rows, C] matrix (rows = N*H*W, C innermost), which is what a
// channels_last NCHW tensor or a [N, C] matrix is in memory.  A thread owns one 128-bit vector of channels
// (4 fp32 / 8 bf16) for the whole kernel, so every per-channel quantity (mean, gamma*invstd, beta, the running
// sums) lives in its registers; the txw threads across a row read one contiguous C*sizeof(T) run, `ty` such
// rows are adjacent, and every thread keeps kBnqU independent 128-bit loads in flight (16 KB per CTA).
// Per-channel reductions: per-thread sums -> fixed-order shared-memory fold over the ty rows -> per-CTA partials
// -> a finalisation kernel that adds the partials in double in a fixed order (deterministic, no atomics).
//
// Arithmetic: BatchNorm is floating-point reduction work - results agree with torch's F.batch_norm within
// reduction-order tolerance (stated in tests/test_gpu_bnq.py), not bit for bit.  The quantizer stage is the
// same `fq_vec<FORM_AFFINE>` code as the stand-alone kernels: given the BatchNorm output `a` (which the kernel
// can also write), a_q is BIT-IDENTICAL to dlmcq_fq_forward(a) - that is how parity with the reference's
// quantizer chain is carried over (tests: fused a_q == fq_forward(fused a)).
//
// Inference hand-off to the code GEMM (dlmcq_bnq_forward_codes): the apply pass can write the quantizer's CODES, one
// byte each in the consumer's operand encoding, instead of a_q - the consumer then reads 1 B/elem instead of running
// its own x -> codes pass over a 4 B/elem a_q.  The codes are the same intermediate a_q is dequantised from, so given a
// they equal dlmcq_codes_forward(a) byte for byte.
#include "bnq_math.cuh"
#include "codes.cuh"

namespace dlmcq {

constexpr int kBnqU = 4;          // independent 128-bit loads per thread per pass
constexpr int kBnqThreads = 256;

struct BnqGeom {
  int64_t rows;
  int32_t C;     // channels
  int32_t cv;    // 128-bit vectors per row
  int32_t txw;   // threads across a row (<= 256)
  int32_t ty;    // rows covered by one "thread row" step
  int32_t gy;    // CTAs across a row (cv > 256)
  int32_t nbx;   // CTAs along the rows for the REDUCING kernels (= number of per-channel partials)
  int64_t nfull4, nfull2;   // full row tiles with 4 / 2 rows per thread (host-side: no 64-bit division per thread)
};

template <typename T>
static inline BnqGeom make_bnq_geom(int64_t rows, int64_t C) {
  BnqGeom g;
  g.rows = rows;
  g.C = static_cast<int32_t>(C);
  g.cv = static_cast<int32_t>(C / Vec<T>::N);
  g.txw = g.cv < kBnqThreads ? g.cv : kBnqThreads;
  if (g.txw < 1) g.txw = 1;
  g.ty = kBnqThreads / g.txw;
  if (g.ty < 1) g.ty = 1;
  g.gy = (g.cv + g.txw - 1) / g.txw;
  const int64_t rpp = static_cast<int64_t>(g.ty) * kBnqU;
  const int64_t passes = (rows + rpp - 1) / rpp;
  int64_t target = static_cast<int64_t>(num_sms()) * 4 / g.gy;   // 4 resident CTAs per SM (64 registers per thread)
  if (target < 1) target = 1;
  int64_t cap = rows / 16;   // every CTA leaves 2*C partial floats behind: keep them well below the tensor itself
  if (cap < 1) cap = 1;
  int64_t nbx = passes < target ? passes : target;
  if (nbx > cap) nbx = cap;
  if (nbx < 1) nbx = 1;
  g.nbx = static_cast<int32_t>(nbx);
  g.nfull4 = rows / (static_cast<int64_t>(g.ty) * 4);
  g.nfull2 = rows / (static_cast<int64_t>(g.ty) * 2);
  return g;
}

// workspace: [header 256 B][partials nbx*2*C][scale partials nbx*gy][coef 2*C][keep mask: one word per (tile, thread)]
struct BnqWs {
  float* part;
  float* part_s;
  float* coef;
  uint32_t* mask;
};
static inline size_t bnq_mask_words(const BnqGeom& g) {
  const int64_t tile_rows = static_cast<int64_t>(g.ty) * kBnqU;
  return static_cast<size_t>((g.rows + tile_rows - 1) / tile_rows) * g.gy * kBnqThreads;
}
static inline size_t bnq_ws_floats(const BnqGeom& g) {
  return static_cast<size_t>(g.nbx) * 2 * g.C + static_cast<size_t>(g.nbx) * g.gy + 2 * static_cast<size_t>(g.C) +
         bnq_mask_words(g);
}
static inline BnqWs bnq_ws(void* ws, const BnqGeom& g) {
  BnqWs w;
  w.part = ws_partials(ws);
  w.part_s = w.part + static_cast<size_t>(g.nbx) * 2 * g.C;
  w.coef = w.part_s + static_cast<size_t>(g.nbx) * g.gy;
  w.mask = reinterpret_cast<uint32_t*>(w.coef + 2 * static_cast<size_t>(g.C));
  return w;
}

#define BNQ_THREAD_COORDS()                                             \
  const int tx = static_cast<int>(threadIdx.x) % gm.txw;               \
  const int ty = static_cast<int>(threadIdx.x) / gm.txw;               \
  const int col = static_cast<int>(blockIdx.y) * gm.txw + tx;          \
  const bool active = (col < gm.cv) && (ty < gm.ty);                   \
  const int64_t rpp = static_cast<int64_t>(gm.ty) * kBnqU

// fold the per-thread sums over the ty thread rows (fixed order) and store this CTA's partials [2][C]
template <int VN>
__device__ __forceinline__ void bnq_store_partials(const float (&s1)[VN], const float (&s2)[VN], float* sm,
                                                   const BnqGeom& gm, int tx, int ty, int col, bool active,
                                                   float* __restrict__ part) {
  float* mine = sm + (static_cast<size_t>(ty) * gm.txw + tx) * (2 * VN);
  if (ty < gm.ty) {
#pragma unroll
    for (int e = 0; e < VN; ++e) {
      mine[e] = s1[e];
      mine[VN + e] = s2[e];
    }
  }
  __syncthreads();
  if (ty == 0 && active) {
    float a1[VN], a2[VN];
#pragma unroll
    for (int e = 0; e < VN; ++e) { a1[e] = 0.f; a2[e] = 0.f; }
    for (int r = 0; r < gm.ty; ++r) {
      const float* p = sm + (static_cast<size_t>(r) * gm.txw + tx) * (2 * VN);
#pragma unroll
      for (int e = 0; e < VN; ++e) { a1[e] += p[e]; a2[e] += p[VN + e]; }
    }
    float* o = part + static_cast<size_t>(blockIdx.x) * 2 * gm.C + static_cast<size_t>(col) * VN;
#pragma unroll
    for (int e = 0; e < VN; ++e) { o[e] = a1[e]; o[gm.C + e] = a2[e]; }
  }
}

// ---------------------------------------------------------------------------------------
// forward, pass 1: per-channel sums of (x - k) and (x - k)^2, k = the channel's value in row 0 (a sample of the
// data: removes the cancellation of E[x^2] - mean^2 at no cost)
// ---------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kBnqThreads, 4)
bnq_stats_kernel(const T* __restrict__ x, BnqGeom gm, float* __restrict__ part) {
  using V = Vec<T>;
  using raw = typename V::raw;
  constexpr int VN = V::N;
  extern __shared__ __align__(16) float sm[];
  BNQ_THREAD_COORDS();
  pdl_wait();          // x is the output of the previous operation on the stream
  pdl_trigger();
  const raw* xv = reinterpret_cast<const raw*>(x);
  float s1[VN], s2[VN], k[VN];
#pragma unroll
  for (int e = 0; e < VN; ++e) { s1[e] = 0.f; s2[e] = 0.f; k[e] = 0.f; }
  if (active) {
    const raw r0 = __ldg(xv + col);
    V::unpack(r0, k);
  }
  for (int64_t r0 = static_cast<int64_t>(blockIdx.x) * rpp; r0 < gm.rows; r0 += static_cast<int64_t>(gridDim.x) * rpp) {
    raw r[kBnqU];
    bool ok[kBnqU];
#pragma unroll
    for (int u = 0; u < kBnqU; ++u) {
      const int64_t row = r0 + ty + static_cast<int64_t>(u) * gm.ty;
      ok[u] = active && row < gm.rows;
      if (ok[u]) r[u] = ld_stream(xv + row * gm.cv + col);
    }
#pragma unroll
    for (int u = 0; u < kBnqU; ++u) {
      if (!ok[u]) continue;
      float f[VN];
      V::unpack(r[u], f);
#pragma unroll
      for (int e = 0; e < VN; ++e) {
        const float d = f[e] - k[e];
        s1[e] += d;
        s2[e] = __fmaf_rn(d, d, s2[e]);
      }
    }
  }
  bnq_store_partials<VN>(s1, s2, sm, gm, tx, ty, col, active, part);
}

// Column sums of the per-CTA partials [nbx][2][C] for 32 adjacent channels, in a fixed order: thread (warp w, lane l)
// adds rows w, w + W, ... of channel c0 + l - every warp load is one coalesced 128-byte row segment (a warp per channel
// striding over the rows touched one 32-byte sector per 4 useful bytes and took 13 - 14 us on 592 x 256 partials) -
// and warp 0 folds the W warp sums in warp order.  Valid in warp 0 (lane = channel - c0) on return.
constexpr int kBnqFoldWarps = 16;
__device__ __forceinline__ void bnq_fold_partials(const float* __restrict__ part, int nbx, int C, int c0,
                                                  double (*sh)[2][32], double& s0, double& s1) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = c0 + lane;
  const size_t stride = 2 * static_cast<size_t>(C);
  double t0 = 0.0, t1 = 0.0;
  if (c < C) {
#pragma unroll 8
    for (int b = warp; b < nbx; b += kBnqFoldWarps) {
      t0 += static_cast<double>(__ldcg(part + b * stride + c));
      t1 += static_cast<double>(__ldcg(part + b * stride + C + c));
    }
  }
  sh[warp][0][lane] = t0;
  sh[warp][1][lane] = t1;
  __syncthreads();
  s0 = 0.0; s1 = 0.0;
  if (warp == 0) {
#pragma unroll
    for (int w = 0; w < kBnqFoldWarps; ++w) { s0 += sh[w][0][lane]; s1 += sh[w][1][lane]; }
  }
}

template <typename T>
__global__ void __launch_bounds__(kBnqFoldWarps * 32)
bnq_stats_finalize_kernel(const T* __restrict__ x, const float* __restrict__ part, BnqGeom gm, float eps, float momentum,
                          float* __restrict__ running_mean, float* __restrict__ running_var,
                          float* __restrict__ save_mean, float* __restrict__ save_invstd) {
  __shared__ double sh[kBnqFoldWarps][2][32];
  pdl_wait();          // the partials come from the statistics kernel launched just before
  pdl_trigger();
  double t1, t2;
  bnq_fold_partials(part, gm.nbx, gm.C, blockIdx.x * 32, sh, t1, t2);
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  if (threadIdx.x < 32 && c < gm.C) {
    const double n = static_cast<double>(gm.rows);
    const double k = static_cast<double>(to_f32<T>(x[c]));
    const double m1 = t1 / n;
    const double mean = k + m1;
    double var = t2 / n - m1 * m1;              // biased variance of the batch
    if (var < 0.0) var = 0.0;
    save_mean[c] = static_cast<float>(mean);
    save_invstd[c] = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
    if (running_mean) {
      const double mo = static_cast<double>(momentum);
      running_mean[c] = static_cast<float>((1.0 - mo) * static_cast<double>(running_mean[c]) + mo * mean);
      const double unbiased = n > 1.0 ? var * (n / (n - 1.0)) : var;
      running_var[c] = static_cast<float>((1.0 - mo) * static_cast<double>(running_var[c]) + mo * unbiased);
    }
  }
}

// eval mode: statistics are the running buffers
__global__ void bnq_eval_prepare_kernel(const float* __restrict__ running_mean, const float* __restrict__ running_var,
                                        int C, float eps, float* __restrict__ save_mean, float* __restrict__ save_invstd) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) {
    save_mean[c] = running_mean[c];
    save_invstd[c] = bn_eval_invstd(running_var[c], eps);
  }
}



// The streaming kernels below share one loop shape.  A CTA owns the row tiles blockIdx.x, blockIdx.x + gridDim.x, ...
// (a tile = ty * U rows); FULL tiles run without a single predicate or 64-bit multiply in the loop (one offset,
// bumped by a constant), the ragged last tile is handled once, by one CTA, on the generic path.  The grid is sized
// so that a CTA sees several tiles: the per-thread set-up (16 per-channel constants, the quantizer's reciprocal) costs
// ~150 instructions, which at one 16-element tile per thread was a third of all instructions issued.
// Per-channel values written by the kernel launched just before (mean / invstd / coef): a normal cached load issued
// AFTER griddepcontrol.wait.  Not ld.global.nc (the producer may still have been running when this kernel started), and
// not ld.global.cg either: every CTA of an SM reads the same few hundred bytes, which L1 serves after the first CTA -
// with .cg each of the thousands of CTAs sent 2048 more requests to L2 (measured: one-tile-per-CTA kernels 3x slower).
__device__ __forceinline__ float ld_ca(const float* p) {
  float v;
  asm volatile("ld.global.ca.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}

// constants in two phases: gamma / beta exist long before the kernel, mean / invstd may come from the kernel just before
template <int VN>
struct GammaBeta {
  float g[VN], b[VN];
};
template <int VN>
__device__ __forceinline__ GammaBeta<VN> load_gamma_beta(const float* __restrict__ gamma, const float* __restrict__ beta,
                                                         int ch0) {
  GammaBeta<VN> gb;
#pragma unroll
  for (int e = 0; e < VN; ++e) {
    gb.g[e] = gamma ? __ldg(gamma + ch0 + e) : 1.f;
    gb.b[e] = beta ? __ldg(beta + ch0 + e) : 0.f;
  }
  return gb;
}
template <int VN>
__device__ __forceinline__ void finish_bnch2(BnCh2<VN>& c2, const GammaBeta<VN>& gb, const float* __restrict__ mean,
                                             const float* __restrict__ invstd, int ch0) {
  BnCh<VN> c;
#pragma unroll
  for (int e = 0; e < VN; ++e) {
    c.mean[e] = ld_ca(mean + ch0 + e);
    c.istd[e] = ld_ca(invstd + ch0 + e);
    c.a[e] = bn_scale(gb.g[e], c.istd[e]);
    c.b[e] = gb.b[e];
  }
  load_bnch2<VN>(c2, c);
}

struct TileLoop {
  int64_t nfull;      // number of full tiles
  int64_t off;        // this thread's first vector of the CTA's first tile
  int64_t stride;     // vectors between consecutive tiles of this CTA
  int64_t du;         // vectors between the U rows a thread loads per tile
  int64_t tail_r0;    // first row of the ragged tile, or -1
};
__device__ __forceinline__ TileLoop make_tile_loop(const BnqGeom& gm, int U, int ty, int col) {
  TileLoop t;
  const int64_t tile_rows = static_cast<int64_t>(gm.ty) * U;
  t.nfull = U == 4 ? gm.nfull4 : gm.nfull2;
  t.du = static_cast<int64_t>(gm.ty) * gm.cv;
  t.off = (static_cast<int64_t>(blockIdx.x) * tile_rows + ty) * gm.cv + col;
  t.stride = static_cast<int64_t>(gridDim.x) * tile_rows * gm.cv;
  const bool mine = (t.nfull * tile_rows < gm.rows) &&
                    (blockIdx.x == static_cast<unsigned>(static_cast<uint64_t>(t.nfull) % gridDim.x));
  t.tail_r0 = mine ? t.nfull * tile_rows : -1;
  return t;
}

// ---------------------------------------------------------------------------------------
// forward, pass 2: normalise (+ identity) (+ ReLU) -> a (optional) and fake-quant(a) (optional)
// ---------------------------------------------------------------------------------------

// The VN codes of one thread's vector as VN contiguous bytes of the [rows, C] code matrix (4 B for fp32, 8 B for
// bf16), stored with q_out's streaming policy.  `idx` is the vector's index in the activation.
template <int ENC, int VN>
__device__ __forceinline__ void st_codes(uint8_t* codes, int64_t idx, const float (&code)[VN]) {
  uint32_t w[VN / 4];
#pragma unroll
  for (int i = 0; i < VN / 4; ++i) {
    w[i] = code_byte<ENC>(code[4 * i]) | (code_byte<ENC>(code[4 * i + 1]) << 8) |
           (code_byte<ENC>(code[4 * i + 2]) << 16) | (code_byte<ENC>(code[4 * i + 3]) << 24);
  }
  uint8_t* p = codes + idx * VN;
  if (VN == 4) {
    asm volatile("st.global.L1::no_allocate.u32 [%0], %1;" ::"l"(p), "r"(w[0]) : "memory");
  } else {
    asm volatile("st.global.L1::no_allocate.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(w[0]), "r"(w[VN / 4 - 1]) : "memory");
  }
}

// OUT: kBnqOutT writes a_q (T) to q_out; DLMCQ_QGEMM_I8 / DLMCQ_QGEMM_E4M3 write the codes of a_q, one byte each in that
// encoding, to q_out instead (QUANT must be true) - the quantizer's code, before dequantisation.
constexpr int kBnqOutT = -1;
template <typename T, bool HAS_ID, bool QUANT, int OUT = kBnqOutT>
__global__ void __launch_bounds__(kBnqThreads, 3)
bnq_apply_kernel(const T* __restrict__ x, const T* __restrict__ idn, const float* __restrict__ gamma,
                 const float* __restrict__ beta, const float* __restrict__ mean, const float* __restrict__ invstd,
                 T* __restrict__ a_out, void* __restrict__ q_out, BnqGeom gm, int relu, const float* __restrict__ scale,
                 const float* __restrict__ offset, float g, float lo, float hi) {
  using V = Vec<T>;
  using raw = typename V::raw;
  constexpr int VN = V::N;
  constexpr bool CODES = OUT != kBnqOutT;
  // bf16 codes: two rows in flight per thread - with four, the 8-wide vectors spill at 80 registers (3 CTAs / SM)
  constexpr int U = (CODES && VN == 8) ? 2 : kBnqU;
  static_assert(!CODES || QUANT, "codes are the quantizer's output");
  uint8_t* cb = static_cast<uint8_t*>(q_out);
  const int tx = static_cast<int>(threadIdx.x) % gm.txw;
  const int ty = static_cast<int>(threadIdx.x) / gm.txw;
  const int col = static_cast<int>(blockIdx.y) * gm.txw + tx;
  const bool active = (col < gm.cv) && (ty < gm.ty);
  const raw* xv = reinterpret_cast<const raw*>(x);
  const raw* iv = reinterpret_cast<const raw*>(idn);
  raw* av = reinterpret_cast<raw*>(a_out);
  raw* qv = reinterpret_cast<raw*>(q_out);
  const TileLoop tl = make_tile_loop(gm, U, ty, col);
  int64_t off = tl.off;
  int64_t t = blockIdx.x;
  raw rx[U], ri[U];
  // the first tile's loads go out BEFORE griddepcontrol.wait: x and the identity were written by kernels older than
  // the statistics pass, so they are valid as soon as this CTA runs; only mean / invstd depend on the finalisation
  // kernel launched just before, and its run time now overlaps these loads instead of preceding them
  if (active && t < tl.nfull) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      rx[u] = ld_stream(xv + off + u * tl.du);
      if (HAS_ID) ri[u] = ld_stream(iv + off + u * tl.du);
    }
  }
  GammaBeta<VN> gb;
  QuantK k;
  if (active) {
    gb = load_gamma_beta<VN>(gamma, beta, col * VN);
    if (QUANT) k = make_quantk(scale, offset, g, lo, hi);    // the consumer layer's parameters: older than this op
  }
  pdl_wait();
  pdl_trigger();
  if (!active) return;
  BnCh2<VN> c2;
  finish_bnch2<VN>(c2, gb, mean, invstd, col * VN);
  const bool fast_ok = c2.safe && (!QUANT || k.fast);
  const float floor = relu ? 0.f : -INFINITY;
  while (t < tl.nfull) {
    if constexpr (CODES) {
      // codes: the fast-path test per vector, so that only one vector is unpacked at a time (registers, see U)
#pragma unroll
      for (int u = 0; u < U; ++u) {
        float fx[VN], fi[VN], act[VN], y[VN], code[VN];
        V::unpack(rx[u], fx);
        float m = absmax_vec<VN>(fx, 0.f);
        if (HAS_ID) {
          V::unpack(ri[u], fi);
          m = absmax_vec<VN>(fi, m);
        }
        if (fast_ok && m <= kBnqSafe) {
#pragma unroll
          for (int e = 0; e < VN; e += 2) {
            const float2 tt = __fadd2_rn(make_float2(fx[e], fx[e + 1]), c2.nmean[e / 2]);
            float2 z = __ffma2_rn(tt, c2.a[e / 2], c2.b[e / 2]);
            if (HAS_ID) z = __fadd2_rn(z, make_float2(fi[e], fi[e + 1]));
            const float2 a2 = act_pair(z, floor);
            act[e] = a2.x;
            act[e + 1] = a2.y;
            float2 q, cc, cd;
            quant_pair(round_to_storage<T>(a2), k, q, cc, cd);
            code[e] = cd.x;
            code[e + 1] = cd.y;
          }
        } else {
          apply_generic_vec<T, VN, true>(fx, HAS_ID ? fi : nullptr, unpack_bnch<VN>(c2), relu != 0, k.p, lo, hi, act,
                                         y, code);
        }
        if (av) av[off + u * tl.du] = V::pack(act);
        st_codes<OUT, VN>(cb, off + u * tl.du, code);
      }
    } else {
      float fx[U][VN], fi[U][VN];
      float m = 0.f;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        V::unpack(rx[u], fx[u]);
        m = absmax_vec<VN>(fx[u], m);
        if (HAS_ID) {
          V::unpack(ri[u], fi[u]);
          m = absmax_vec<VN>(fi[u], m);
        }
      }
      if (fast_ok && m <= kBnqSafe) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
          float act[VN], y[VN], code[VN];
#pragma unroll
          for (int e = 0; e < VN; e += 2) {
            const float2 tt = __fadd2_rn(make_float2(fx[u][e], fx[u][e + 1]), c2.nmean[e / 2]);
            float2 z = __ffma2_rn(tt, c2.a[e / 2], c2.b[e / 2]);
            if (HAS_ID) z = __fadd2_rn(z, make_float2(fi[u][e], fi[u][e + 1]));
            const float2 a2 = act_pair(z, floor);
            act[e] = a2.x;
            act[e + 1] = a2.y;
            if (QUANT) {
              float2 q, cc, cd;
              quant_pair(round_to_storage<T>(a2), k, q, cc, cd);
              const float2 yy = dequant_pair(cd, k);
              y[e] = yy.x;
              y[e + 1] = yy.y;
            }
          }
          if (av) av[off + u * tl.du] = V::pack(act);   // re-read by the backward pass / the next block: default L2 policy
          if (QUANT) st_stream(qv + off + u * tl.du, V::pack(y));
        }
      } else {
        const BnCh<VN> c = unpack_bnch<VN>(c2);
#pragma unroll
        for (int u = 0; u < U; ++u) {
          float act[VN], y[VN], code[VN];
          apply_generic_vec<T, VN, QUANT>(fx[u], HAS_ID ? fi[u] : nullptr, c, relu != 0, k.p, lo, hi, act, y, code);
          if (av) av[off + u * tl.du] = V::pack(act);
          if (QUANT) st_stream(qv + off + u * tl.du, V::pack(y));
        }
      }
    }
    t += gridDim.x;
    off += tl.stride;
    if (t < tl.nfull) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        rx[u] = ld_stream(xv + off + u * tl.du);
        if (HAS_ID) ri[u] = ld_stream(iv + off + u * tl.du);
      }
    }
  }
  if (tl.tail_r0 >= 0) {
    const BnCh<VN> c = unpack_bnch<VN>(c2);
#pragma unroll 1
    for (int u = 0; u < U; ++u) {
      const int64_t row = tl.tail_r0 + ty + static_cast<int64_t>(u) * gm.ty;
      if (row >= gm.rows) break;
      const int64_t idx = row * gm.cv + col;
      float fx[VN], fi[VN], act[VN], y[VN], code[VN];
      V::unpack(ld_stream(xv + idx), fx);
      if (HAS_ID) V::unpack(ld_stream(iv + idx), fi);
      apply_generic_vec<T, VN, QUANT>(fx, HAS_ID ? fi : nullptr, c, relu != 0, k.p, lo, hi, act, y, code);
      if (av) av[idx] = V::pack(act);
      if (CODES) st_codes<OUT, VN>(cb, idx, code);
      else if (QUANT) st_stream(qv + idx, V::pack(y));
    }
  }
}

// ---------------------------------------------------------------------------------------
// backward.  dz = d(loss)/d(z), z = BatchNorm output (+ identity) before the ReLU:
//     da = d_a (gradient of the plain output, if any) + fake-quant backward(a, d_q)     [fq_vec_bwd<AFFINE>]
//     dz = da * 1[a > 0] (ReLU) or da
//   RESID = false: `a` is recomputed from x (nothing but x and the upstream gradients is read);
//   RESID = true : z contains the identity, so the saved plain output `a` is read instead, and dz - which IS the
//                  gradient of the identity branch - is written once and re-read by the dx pass.
// pass 1 (reduce): per-channel sum(dz), sum(dz * xhat), and the per-tensor scale-gradient sum.
// ---------------------------------------------------------------------------------------
// generic (guarded) per-vector code
template <typename T, int VN, bool RESID, bool QUANT>
__device__ __forceinline__ void bnq_dz_vec(const float (&fx)[VN], const float (&fa)[VN], const float* fda,
                                           const float (&fdq)[VN], const BnCh<VN>& c, bool relu, const ChanParams& p,
                                           float lo, float hi, float& acc_s, float (&dz)[VN]) {
  float act[VN];
  if (RESID) {
#pragma unroll
    for (int e = 0; e < VN; ++e) act[e] = fa[e];
  } else {
    bn_act_vec<VN>(fx, c, nullptr, relu, act);
    if (sizeof(T) == 2) {
#pragma unroll
      for (int e = 0; e < VN; ++e) act[e] = to_f32<T>(from_f32<T>(act[e]));
    }
  }
  float da[VN];
  if (QUANT) {
    float dummy = 0.f;
    fq_vec_bwd<DLMCQ_FORM_AFFINE, false, VN>(act, fdq, p, lo, hi, da, acc_s, dummy);
  } else {
#pragma unroll
    for (int e = 0; e < VN; ++e) da[e] = 0.f;
  }
  if (fda) {
#pragma unroll
    for (int e = 0; e < VN; ++e) da[e] += fda[e];
  }
#pragma unroll
  for (int e = 0; e < VN; ++e) dz[e] = relu ? ((act[e] > 0.f) ? da[e] : 0.f) : da[e];
}

// packed: dz for one pair.  `act` is the (storage-rounded) activation.
// keep0/1: the element passes d_q straight through (inside the clamp range AND above the ReLU floor)
template <bool QUANT>
__device__ __forceinline__ float2 dz_pair(float2 act, float2 dq, float2 da_in, bool has_da, float floor, const QuantK& k,
                                          float2& acc2, bool& keep0, bool& keep1) {
  float2 da = make_float2(0.f, 0.f);
  const bool up0 = act.x > floor, up1 = act.y > floor;
  keep0 = false;
  keep1 = false;
  if (QUANT) {
    float2 q, c, cd;
    quant_pair(act, k, q, c, cd);
    const float2 df = __fadd2_rn(cd, make_float2(-q.x, -q.y));
    const bool in0 = (c.x == q.x), in1 = (c.y == q.y);        // in range <=> the clamp was the identity (NaN: false)
    acc2 = __ffma2_rn(dq, make_float2(in0 ? df.x : cd.x, in1 ? df.y : cd.y), acc2);
    da = make_float2(in0 ? dq.x : 0.f, in1 ? dq.y : 0.f);
    keep0 = in0 && up0;
    keep1 = in1 && up1;
  }
  if (has_da) da = __fadd2_rn(da, da_in);
  return make_float2(up0 ? da.x : 0.f, up1 ? da.y : 0.f);
}

// U / MINB: rows in flight per thread and resident CTAs per SM.  The recomputing quantizer variant carries ~100 live
// registers with four rows in flight and runs <4, 2>, which keeps them all; the residual variants run <2, 3> and the
// plain BatchNorm variant <4, 3>.
template <typename T, bool RESID, bool QUANT, int U, int MINB>
__global__ void __launch_bounds__(kBnqThreads, MINB)
bnq_bwd_reduce_kernel(const T* __restrict__ x, const T* __restrict__ a_saved, const T* __restrict__ d_a,
                      const T* __restrict__ d_q, const float* __restrict__ gamma, const float* __restrict__ beta,
                      const float* __restrict__ mean, const float* __restrict__ invstd, T* __restrict__ dz_out,
                      BnqGeom gm, int relu, const float* __restrict__ scale, const float* __restrict__ offset, float g,
                      float lo, float hi, float* __restrict__ part, float* __restrict__ part_s,
                      uint32_t* __restrict__ keep_mask) {
  // keep_mask (plain quantizer chain): bit (u * VN + e) of word [(tile * gy + blockIdx.y) * 256 + thread]
  // says "dz == d_q" for that element (inside the clamp range and above the ReLU floor), so that the dx pass needs
  // neither the quantizer arithmetic nor its ~60 extra registers - 1/8 byte per element written here, read there.
  using V = Vec<T>;
  using raw = typename V::raw;
  constexpr int VN = V::N;
  extern __shared__ __align__(16) float sm[];
  __shared__ float red[64];
  const int tx = static_cast<int>(threadIdx.x) % gm.txw;
  const int ty = static_cast<int>(threadIdx.x) / gm.txw;
  const int col = static_cast<int>(blockIdx.y) * gm.txw + tx;
  const bool active = (col < gm.cv) && (ty < gm.ty);
  const bool has_da = d_a != nullptr;
  const raw* xv = reinterpret_cast<const raw*>(x);
  const raw* av = reinterpret_cast<const raw*>(a_saved);
  const raw* dav = reinterpret_cast<const raw*>(d_a);
  const raw* dqv = reinterpret_cast<const raw*>(d_q);
  raw* zv = reinterpret_cast<raw*>(dz_out);
  const TileLoop tl = make_tile_loop(gm, U, ty, col);
  int64_t off = tl.off;
  int64_t t = blockIdx.x;
  raw rx[U], ra[U], rda[U], rdq[U];
  auto load_tile = [&](int64_t o) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      rx[u] = ld_stream(xv + o + u * tl.du);
      if (RESID) ra[u] = ld_stream(av + o + u * tl.du);
      if (has_da) rda[u] = ld_stream(dav + o + u * tl.du);
      if (QUANT) rdq[u] = ld_stream(dqv + o + u * tl.du);
    }
  };
  pdl_wait();          // the upstream gradients are the output of the previous operation on the stream
  pdl_trigger();
  // the first tile's loads are issued before the per-channel constants and the quantizer's scale are fetched: the
  // two latencies overlap instead of adding up (the constants used to cost a CTA a full extra memory round trip)
  if (active && t < tl.nfull) load_tile(off);
  BnCh2<VN> c2;
  if (active) load_bnch2<VN>(c2, gamma, beta, mean, invstd, col * VN);
  QuantK k;
  if (QUANT) k = make_quantk(scale, offset, g, lo, hi);
  const bool fast_ok = active && c2.safe && (!QUANT || k.fast);
  const float floor = relu ? 0.f : -INFINITY;
  float2 sdb[VN / 2], sdg[VN / 2];
#pragma unroll
  for (int e = 0; e < VN / 2; ++e) { sdb[e] = make_float2(0.f, 0.f); sdg[e] = make_float2(0.f, 0.f); }
  float2 acc2 = make_float2(0.f, 0.f);
  float acc_slow = 0.f;

  // generic per-vector step (guarded arithmetic): the slow path of full tiles and the ragged tile
  auto generic_vec = [&](const BnCh<VN>& c, int64_t idx, const raw& rxx, const raw& raa, const raw& rdaa, const raw& rdqq,
                         uint32_t& bits, int shift) {
    float fx[VN], fa[VN], fda[VN], fdq[VN], dz[VN];
    V::unpack(rxx, fx);
    if (RESID) V::unpack(raa, fa);
    if (has_da) V::unpack(rdaa, fda);
    if (QUANT) V::unpack(rdqq, fdq);
    bnq_dz_vec<T, VN, RESID, QUANT>(fx, fa, has_da ? fda : nullptr, fdq, c, relu != 0, k.p, lo, hi, acc_slow, dz);
#pragma unroll
    for (int e = 0; e < VN; e += 2) {
      if (zv && sizeof(T) == 2) {
        dz[e] = to_f32<T>(from_f32<T>(dz[e]));
        dz[e + 1] = to_f32<T>(from_f32<T>(dz[e + 1]));
      }
      const float xh0 = (fx[e] - c.mean[e]) * c.istd[e], xh1 = (fx[e + 1] - c.mean[e + 1]) * c.istd[e + 1];
      sdb[e / 2].x += dz[e];
      sdb[e / 2].y += dz[e + 1];
      sdg[e / 2].x = __fmaf_rn(dz[e], xh0, sdg[e / 2].x);
      sdg[e / 2].y = __fmaf_rn(dz[e + 1], xh1, sdg[e / 2].y);
      // without d_a, dz is either d_q or 0: "dz != 0 or NaN" reproduces it from d_q (a zero d_q gives zero either way)
      bits |= (dz[e] != 0.f || dz[e] != dz[e] ? 1u : 0u) << (shift + e);
      bits |= (dz[e + 1] != 0.f || dz[e + 1] != dz[e + 1] ? 1u : 0u) << (shift + e + 1);
    }
    if (zv) zv[idx] = V::pack(dz);
  };

  if (active) {
    while (t < tl.nfull) {
      uint32_t bits = 0u;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        float fx[VN], fa[VN];
        V::unpack(rx[u], fx);
        float m = absmax_vec<VN>(fx, 0.f);
        if (RESID) {
          V::unpack(ra[u], fa);
          m = absmax_vec<VN>(fa, m);
        }
        if (fast_ok && m <= kBnqSafe) {
          float fda[VN], fdq[VN], dz[VN];
          if (has_da) V::unpack(rda[u], fda);
          if (QUANT) V::unpack(rdq[u], fdq);
#pragma unroll
          for (int e = 0; e < VN; e += 2) {
            const float2 tt = __fadd2_rn(make_float2(fx[e], fx[e + 1]), c2.nmean[e / 2]);
            float2 act;
            if (RESID) {
              act = make_float2(fa[e], fa[e + 1]);
            } else {
              act = round_to_storage<T>(act_pair(__ffma2_rn(tt, c2.a[e / 2], c2.b[e / 2]), floor));
            }
            bool k0, k1;
            float2 d2 = dz_pair<QUANT>(act, QUANT ? make_float2(fdq[e], fdq[e + 1]) : make_float2(0.f, 0.f),
                                       has_da ? make_float2(fda[e], fda[e + 1]) : make_float2(0.f, 0.f), has_da, floor,
                                       k, acc2, k0, k1);
            bits |= (k0 ? 1u : 0u) << (u * VN + e);
            bits |= (k1 ? 1u : 0u) << (u * VN + e + 1);
            if (zv) d2 = round_to_storage<T>(d2);   // the dx pass and the identity branch see the stored value
            dz[e] = d2.x;
            dz[e + 1] = d2.y;
            const float2 xh = __fmul2_rn(tt, c2.istd[e / 2]);
            sdb[e / 2] = __fadd2_rn(sdb[e / 2], d2);
            sdg[e / 2] = __ffma2_rn(d2, xh, sdg[e / 2]);
          }
          if (zv) zv[off + u * tl.du] = V::pack(dz);  // re-read by the dx pass (and the identity branch): default policy
        } else {
          generic_vec(unpack_bnch<VN>(c2), off + u * tl.du, rx[u], ra[u], rda[u], rdq[u], bits, u * VN);
        }
      }
      if (keep_mask) keep_mask[(static_cast<size_t>(t) * gridDim.y + blockIdx.y) * kBnqThreads + threadIdx.x] = bits;
      t += gridDim.x;
      off += tl.stride;
      if (t < tl.nfull) load_tile(off);
    }
    if (tl.tail_r0 >= 0) {
      const BnCh<VN> c = unpack_bnch<VN>(c2);
      uint32_t bits = 0u;
#pragma unroll 1
      for (int u = 0; u < U; ++u) {
        const int64_t row = tl.tail_r0 + ty + static_cast<int64_t>(u) * gm.ty;
        if (row >= gm.rows) break;
        const int64_t idx = row * gm.cv + col;
        raw r0 = ld_stream(xv + idx), r1 = r0, r2 = r0, r3 = r0;
        if (RESID) r1 = ld_stream(av + idx);
        if (has_da) r2 = ld_stream(dav + idx);
        if (QUANT) r3 = ld_stream(dqv + idx);
        generic_vec(c, idx, r0, r1, r2, r3, bits, u * VN);
      }
      if (keep_mask) keep_mask[(static_cast<size_t>(tl.nfull) * gridDim.y + blockIdx.y) * kBnqThreads + threadIdx.x] = bits;
    }
  }
  float s1[VN], s2[VN];
#pragma unroll
  for (int e = 0; e < VN; e += 2) {
    s1[e] = sdb[e / 2].x; s1[e + 1] = sdb[e / 2].y;
    s2[e] = sdg[e / 2].x; s2[e + 1] = sdg[e / 2].y;
  }
  bnq_store_partials<VN>(s1, s2, sm, gm, tx, ty, col, active, part);
  if (QUANT) {
    float acc[1] = {(acc2.x + acc2.y) + acc_slow};
    block_sum<1>(acc, red);
    if (threadIdx.x == 0) part_s[static_cast<size_t>(blockIdx.y) * gridDim.x + blockIdx.x] = acc[0];
  }
}

// per-channel d gamma / d beta and the coefficients of the dx pass (32 channels per CTA, folded as above); the last
// CTA reduces the scale gradient
__global__ void __launch_bounds__(kBnqFoldWarps * 32)
bnq_bwd_finalize_kernel(const float* __restrict__ part, const float* __restrict__ part_s, BnqGeom gm, int n_part_s,
                        int training, float g, float* __restrict__ dgamma, float* __restrict__ dbeta,
                        float* __restrict__ coef, float* __restrict__ dscale) {
  __shared__ double sh[kBnqFoldWarps][2][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  pdl_wait();
  pdl_trigger();
  if (blockIdx.x == gridDim.x - 1) {          // scale gradient: fixed-order sum of the per-CTA partials in double
    double s = 0.0;
    for (int i = threadIdx.x; i < n_part_s; i += blockDim.x) s += static_cast<double>(__ldcg(part_s + i));
    s = warp_sum(s);
    if (lane == 0) sh[warp][0][0] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int r = 0; r < kBnqFoldWarps; ++r) t += sh[r][0][0];
      if (dscale) dscale[0] = static_cast<float>(t) * g;     // chain through grad_scale (utils.py:24-27)
    }
    return;
  }
  double db, dg;
  bnq_fold_partials(part, gm.nbx, gm.C, blockIdx.x * 32, sh, db, dg);
  const int c = blockIdx.x * 32 + lane;
  if (warp == 0 && c < gm.C) {
    if (dbeta) dbeta[c] = static_cast<float>(db);
    if (dgamma) dgamma[c] = static_cast<float>(dg);
    const double n = static_cast<double>(gm.rows);
    coef[c] = training ? static_cast<float>(db / n) : 0.f;            // mean(dz)
    coef[gm.C + c] = training ? static_cast<float>(dg / n) : 0.f;     // mean(dz * xhat)
  }
}

// pass 2: dx = gamma*invstd * (dz - mean(dz) - xhat * mean(dz*xhat))     (eval mode: gamma*invstd * dz)
// Generic form: dz is recomputed from x and the upstream gradients (the light kernel below covers the residual form
// and the plain quantizer chain without d_a).  MINB: resident CTAs per SM, 2 with the quantizer, 3 without.
template <typename T, bool QUANT, int MINB>
__global__ void __launch_bounds__(kBnqThreads, MINB)
bnq_bwd_dx_kernel(const T* __restrict__ x, const T* __restrict__ d_a, const T* __restrict__ d_q,
                  const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ mean,
                  const float* __restrict__ invstd, const float* __restrict__ coef, T* __restrict__ dx, BnqGeom gm,
                  int relu, const float* __restrict__ scale, const float* __restrict__ offset, float g, float lo,
                  float hi) {
  using V = Vec<T>;
  using raw = typename V::raw;
  constexpr int VN = V::N;
  constexpr int U = kBnqU;
  const int tx = static_cast<int>(threadIdx.x) % gm.txw;
  const int ty = static_cast<int>(threadIdx.x) / gm.txw;
  const int col = static_cast<int>(blockIdx.y) * gm.txw + tx;
  const bool active = (col < gm.cv) && (ty < gm.ty);
  const bool has_da = d_a != nullptr;
  const raw* xv = reinterpret_cast<const raw*>(x);
  const raw* dav = reinterpret_cast<const raw*>(d_a);
  const raw* dqv = reinterpret_cast<const raw*>(d_q);
  raw* ov = reinterpret_cast<raw*>(dx);
  const TileLoop tl = make_tile_loop(gm, U, ty, col);
  int64_t off = tl.off;
  int64_t t = blockIdx.x;
  raw rx[U], r1[U], r2[U];
  auto load_tile = [&](int64_t o) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      rx[u] = ld_stream(xv + o + u * tl.du);
      if (has_da) r1[u] = ld_stream(dav + o + u * tl.du);
      if (QUANT) r2[u] = ld_stream(dqv + o + u * tl.du);
    }
  };
  // everything except coef is older than the finalisation kernel this launch depends on: fetch it before the wait
  if (active && t < tl.nfull) load_tile(off);
  BnCh2<VN> c2;
  QuantK k;
  if (active) {
    load_bnch2<VN>(c2, gamma, beta, mean, invstd, col * VN);
    if (QUANT) k = make_quantk(scale, offset, g, lo, hi);
  }
  pdl_wait();          // coef comes from the finalisation kernel launched just before
  pdl_trigger();
  if (!active) return;
  float2 nc1[VN / 2], c22[VN / 2], nistd[VN / 2];
#pragma unroll
  for (int e = 0; e < VN; e += 2) {
    nc1[e / 2] = make_float2(-ld_ca(coef + col * VN + e), -ld_ca(coef + col * VN + e + 1));
    c22[e / 2] = make_float2(ld_ca(coef + gm.C + col * VN + e), ld_ca(coef + gm.C + col * VN + e + 1));
    nistd[e / 2] = make_float2(-c2.istd[e / 2].x, -c2.istd[e / 2].y);
  }
  const bool fast_ok = c2.safe && (!QUANT || k.fast);
  const float floor = relu ? 0.f : -INFINITY;

  // dz of one vector (packed when `fast`), then the BatchNorm input gradient
  auto finish_vec = [&](const float (&fx)[VN], const float (&f1)[VN], const float (&f2)[VN], bool fast, int64_t idx) {
    float dzs[VN], o[VN];
    if (!fast) {
      float dummy = 0.f;
      bnq_dz_vec<T, VN, false, QUANT>(fx, fx, has_da ? f1 : nullptr, f2, unpack_bnch<VN>(c2), relu != 0, k.p, lo, hi, dummy,
                                      dzs);
    }
#pragma unroll
    for (int e = 0; e < VN; e += 2) {
      const float2 tt = __fadd2_rn(make_float2(fx[e], fx[e + 1]), c2.nmean[e / 2]);
      float2 d2;
      if (fast) {
        float2 dummy2 = make_float2(0.f, 0.f);
        bool k0, k1;
        const float2 act = round_to_storage<T>(act_pair(__ffma2_rn(tt, c2.a[e / 2], c2.b[e / 2]), floor));
        d2 = dz_pair<QUANT>(act, QUANT ? make_float2(f2[e], f2[e + 1]) : make_float2(0.f, 0.f),
                            has_da ? make_float2(f1[e], f1[e + 1]) : make_float2(0.f, 0.f), has_da, floor, k, dummy2, k0,
                            k1);
      } else {
        d2 = make_float2(dzs[e], dzs[e + 1]);
      }
      // a * ((dz - c1) - xhat * c2), xhat = t * invstd
      const float2 nxh = __fmul2_rn(tt, nistd[e / 2]);
      const float2 w = __ffma2_rn(nxh, c22[e / 2], __fadd2_rn(d2, nc1[e / 2]));
      const float2 r = __fmul2_rn(c2.a[e / 2], w);
      o[e] = r.x;
      o[e + 1] = r.y;
    }
    st_stream(ov + idx, V::pack(o));
  };

  while (t < tl.nfull) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      float fx[VN], f1[VN], f2[VN];
      V::unpack(rx[u], fx);
      if (has_da) V::unpack(r1[u], f1);
      if (QUANT) V::unpack(r2[u], f2);
      const bool fast = fast_ok && absmax_vec<VN>(fx, 0.f) <= kBnqSafe;
      finish_vec(fx, f1, f2, fast, off + u * tl.du);
    }
    t += gridDim.x;
    off += tl.stride;
    if (t < tl.nfull) load_tile(off);
  }
  if (tl.tail_r0 >= 0) {
#pragma unroll 1
    for (int u = 0; u < U; ++u) {
      const int64_t row = tl.tail_r0 + ty + static_cast<int64_t>(u) * gm.ty;
      if (row >= gm.rows) break;
      const int64_t idx = row * gm.cv + col;
      float fx[VN], f1[VN], f2[VN];
      V::unpack(ld_stream(xv + idx), fx);
      if (has_da) V::unpack(ld_stream(dav + idx), f1);
      if (QUANT) V::unpack(ld_stream(dqv + idx), f2);
      finish_vec(fx, f1, f2, false, idx);
    }
  }
}

// pass 2, light form: dz comes from memory - the stored dz (residual form) or d_q gated by the keep mask (plain
// quantizer chain) - so only the BatchNorm input-gradient arithmetic is left (~10 packed instructions per element, 64
// registers).  One tile per CTA; the tile's loads are issued BEFORE griddepcontrol.wait: x, d_q, dz and the mask were
// all written (or read) by kernels older than the finalisation kernel this launch depends on, so they are valid as
// soon as this CTA runs, and their latency overlaps the finalisation kernel instead of following it.
template <typename T, bool MASKED>
__global__ void __launch_bounds__(kBnqThreads, 3)
bnq_bwd_dx_light_kernel(const T* __restrict__ x, const T* __restrict__ src /* dz, or d_q when MASKED */,
                        const uint32_t* __restrict__ keep_mask, const float* __restrict__ gamma,
                        const float* __restrict__ beta, const float* __restrict__ mean, const float* __restrict__ invstd,
                        const float* __restrict__ coef, T* __restrict__ dx, BnqGeom gm) {
  using V = Vec<T>;
  using raw = typename V::raw;
  constexpr int VN = V::N;
  constexpr int U = kBnqU;
  const int tx = static_cast<int>(threadIdx.x) % gm.txw;
  const int ty = static_cast<int>(threadIdx.x) / gm.txw;
  const int col = static_cast<int>(blockIdx.y) * gm.txw + tx;
  const bool active = (col < gm.cv) && (ty < gm.ty);
  const raw* xv = reinterpret_cast<const raw*>(x);
  const raw* sv = reinterpret_cast<const raw*>(src);
  raw* ov = reinterpret_cast<raw*>(dx);
  const TileLoop tl = make_tile_loop(gm, U, ty, col);
  int64_t off = tl.off;
  int64_t t = blockIdx.x;
  raw rx[U], rs[U];
  uint32_t bits = 0u;
  if (active && t < tl.nfull) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      rx[u] = ld_stream(xv + off + u * tl.du);
      rs[u] = ld_stream(sv + off + u * tl.du);
    }
    if (MASKED) bits = __ldcg(keep_mask + (static_cast<size_t>(t) * gridDim.y + blockIdx.y) * kBnqThreads + threadIdx.x);
  }
  BnCh2<VN> c2;
  if (active) load_bnch2<VN>(c2, gamma, beta, mean, invstd, col * VN);   // forward-pass results: older than this op
  pdl_wait();          // only coef comes from the finalisation kernel launched just before
  pdl_trigger();
  if (!active) return;
  float2 nc1[VN / 2], c22[VN / 2], nistd[VN / 2];
#pragma unroll
  for (int e = 0; e < VN; e += 2) {
    nc1[e / 2] = make_float2(-ld_ca(coef + col * VN + e), -ld_ca(coef + col * VN + e + 1));
    c22[e / 2] = make_float2(ld_ca(coef + gm.C + col * VN + e), ld_ca(coef + gm.C + col * VN + e + 1));
    nistd[e / 2] = make_float2(-c2.istd[e / 2].x, -c2.istd[e / 2].y);
  }
  auto one = [&](const raw& rxx, const raw& rss, uint32_t b, int shift, int64_t idx) {
    float fx[VN], fs[VN], o[VN];
    V::unpack(rxx, fx);
    V::unpack(rss, fs);
#pragma unroll
    for (int e = 0; e < VN; e += 2) {
      float2 d2 = make_float2(fs[e], fs[e + 1]);
      if (MASKED) {
        d2.x = (b >> (shift + e)) & 1u ? d2.x : 0.f;
        d2.y = (b >> (shift + e + 1)) & 1u ? d2.y : 0.f;
      }
      const float2 tt = __fadd2_rn(make_float2(fx[e], fx[e + 1]), c2.nmean[e / 2]);
      const float2 nxh = __fmul2_rn(tt, nistd[e / 2]);
      const float2 w = __ffma2_rn(nxh, c22[e / 2], __fadd2_rn(d2, nc1[e / 2]));
      const float2 r = __fmul2_rn(c2.a[e / 2], w);
      o[e] = r.x;
      o[e + 1] = r.y;
    }
    st_stream(ov + idx, V::pack(o));
  };
  while (t < tl.nfull) {
#pragma unroll
    for (int u = 0; u < U; ++u) one(rx[u], rs[u], bits, u * VN, off + u * tl.du);
    t += gridDim.x;
    off += tl.stride;
    if (t < tl.nfull) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        rx[u] = ld_stream(xv + off + u * tl.du);
        rs[u] = ld_stream(sv + off + u * tl.du);
      }
      if (MASKED) bits = __ldcg(keep_mask + (static_cast<size_t>(t) * gridDim.y + blockIdx.y) * kBnqThreads + threadIdx.x);
    }
  }
  if (tl.tail_r0 >= 0) {
    const uint32_t b = MASKED ? __ldcg(keep_mask + (static_cast<size_t>(tl.nfull) * gridDim.y + blockIdx.y) * kBnqThreads + threadIdx.x) : 0u;
#pragma unroll 1
    for (int u = 0; u < U; ++u) {
      const int64_t row = tl.tail_r0 + ty + static_cast<int64_t>(u) * gm.ty;
      if (row >= gm.rows) break;
      const int64_t idx = row * gm.cv + col;
      one(ld_stream(xv + idx), ld_stream(sv + idx), b, u * VN, idx);
    }
  }
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
static inline int bnq_check(const dlmcq_bnq_desc* d) {
  if (!d || d->rows < 0 || d->channels < 1) return DLMCQ_EINVAL;
  if (d->dtype != DLMCQ_F32 && d->dtype != DLMCQ_BF16) return DLMCQ_EINVAL;
  const int64_t vn = d->dtype == DLMCQ_F32 ? 4 : 8;
  if (d->channels % vn != 0 || d->channels > (int64_t(1) << 20)) return DLMCQ_EUNSUPPORTED;
  return DLMCQ_OK;
}
// CTAs along the rows for the non-reducing kernels: about `tiles` tiles per CTA (amortises the per-thread set-up) but
// never fewer CTAs than 8 per SM while the tensor has that many tiles
static inline int apply_grid(const BnqGeom& g, int tiles) {
  const int64_t rpp = static_cast<int64_t>(g.ty) * kBnqU;
  const int64_t passes = (g.rows + rpp - 1) / rpp;
  const int64_t floor_ctas = static_cast<int64_t>(num_sms()) * 8 / g.gy;
  int64_t n = passes / tiles;
  if (n < floor_ctas) n = floor_ctas;
  if (n > passes) n = passes;
  return n < 1 ? 1 : static_cast<int>(n);
}
template <int VN>
static inline size_t bnq_smem(const BnqGeom& g) {
  return static_cast<size_t>(g.ty) * g.txw * 2 * VN * sizeof(float);
}

// the apply kernel for one output mode: a_q (out = kBnqOutT) or its codes in encoding `out`
template <typename T, int OUT>
static auto bnq_apply_for(bool idn, bool quant) {
  if (OUT != kBnqOutT) return idn ? bnq_apply_kernel<T, true, true, OUT> : bnq_apply_kernel<T, false, true, OUT>;
  return idn ? (quant ? bnq_apply_kernel<T, true, true> : bnq_apply_kernel<T, true, false>)
             : (quant ? bnq_apply_kernel<T, false, true> : bnq_apply_kernel<T, false, false>);
}

// q_out: a_q (out = kBnqOutT), or the codes in encoding `out` (eval mode only: dlmcq_bnq_forward_codes)
template <typename T>
static int bnq_forward_t(const void* x, const void* idn, const float* gamma, const float* beta, float* rmean,
                         float* rvar, float* smean, float* sinv, void* a_out, void* q_out, const dlmcq_bnq_desc* d,
                         const dlmcq_qparams* qp, void* ws, size_t ws_bytes, cudaStream_t st, int out = kBnqOutT) {
  constexpr int VN = Vec<T>::N;
  const BnqGeom g = make_bnq_geom<T>(d->rows, d->channels);
  if (ws_bytes < kWsHeaderBytes + bnq_ws_floats(g) * sizeof(float)) return DLMCQ_EWORKSPACE;
  const BnqWs w = bnq_ws(ws, g);
  const bool training = (d->flags & DLMCQ_BNQ_TRAINING) != 0;
  const T* xt = static_cast<const T*>(x);
  if (training) {
    cudaError_t e = launch_pdl(bnq_stats_kernel<T>, dim3(g.nbx, g.gy), dim3(kBnqThreads), bnq_smem<VN>(g), st, xt, g,
                               w.part);
    if (e != cudaSuccess) return set_cuda_error(e);
    e = launch_pdl(bnq_stats_finalize_kernel<T>, dim3((g.C + 31) / 32), dim3(kBnqFoldWarps * 32), 0, st, xt,
                   static_cast<const float*>(w.part), g, d->eps, d->momentum, rmean, rvar, smean, sinv);
    if (e != cudaSuccess) return set_cuda_error(e);
  } else {
    bnq_eval_prepare_kernel<<<(g.C + 255) / 256, 256, 0, st>>>(rmean, rvar, g.C, d->eps, smean, sinv);
  }
  DLMCQ_LAUNCH_CHECK();
  if (!a_out && !q_out) return DLMCQ_OK;     // statistics only
  const bool quant = q_out != nullptr;
  const int relu = (d->flags & DLMCQ_BNQ_RELU) ? 1 : 0;
  const float lo = quant ? static_cast<float>(qp->lo) : 0.f, hi = quant ? static_cast<float>(qp->hi) : 0.f;
  const float* sc = quant ? qp->scale : nullptr;
  const float* of = quant ? qp->offset : nullptr;
  const float gq = quant ? qp->g : 0.f;
  const dim3 grid(apply_grid(g, 8), g.gy);
  auto k = out == DLMCQ_QGEMM_I8     ? bnq_apply_for<T, DLMCQ_QGEMM_I8>(idn != nullptr, quant)
           : out == DLMCQ_QGEMM_E4M3 ? bnq_apply_for<T, DLMCQ_QGEMM_E4M3>(idn != nullptr, quant)
                                     : bnq_apply_for<T, kBnqOutT>(idn != nullptr, quant);
  cudaError_t e = launch_pdl(k, grid, dim3(kBnqThreads), 0, st, xt, static_cast<const T*>(idn), gamma, beta,
                             static_cast<const float*>(smean), static_cast<const float*>(sinv), static_cast<T*>(a_out),
                             q_out, g, relu, sc, of, gq, lo, hi);
  if (e != cudaSuccess) return set_cuda_error(e);
  return DLMCQ_OK;
}

template <typename T>
static int bnq_backward_t(const void* x, const void* a_saved, const void* d_a, const void* d_q, const float* gamma,
                          const float* beta, const float* smean, const float* sinv, void* dx, void* dz_out,
                          float* dgamma, float* dbeta, float* dscale, const dlmcq_bnq_desc* d, const dlmcq_qparams* qp,
                          void* ws, size_t ws_bytes, cudaStream_t st) {
  constexpr int VN = Vec<T>::N;
  const BnqGeom g = make_bnq_geom<T>(d->rows, d->channels);
  if (ws_bytes < kWsHeaderBytes + bnq_ws_floats(g) * sizeof(float)) return DLMCQ_EWORKSPACE;
  const BnqWs w = bnq_ws(ws, g);
  const bool resid = (d->flags & DLMCQ_BNQ_RESIDUAL) != 0;
  const bool quant = d_q != nullptr;
  const int relu = (d->flags & DLMCQ_BNQ_RELU) ? 1 : 0;
  const int training = (d->flags & DLMCQ_BNQ_TRAINING) ? 1 : 0;
  const float lo = quant ? static_cast<float>(qp->lo) : 0.f, hi = quant ? static_cast<float>(qp->hi) : 0.f;
  const float* sc = quant ? qp->scale : nullptr;
  const float* of = quant ? qp->offset : nullptr;
  const float gq = quant ? qp->g : 0.f;
  const T* xt = static_cast<const T*>(x);
  const T* at = static_cast<const T*>(a_saved);
  const T* dat = static_cast<const T*>(d_a);
  const T* dqt = static_cast<const T*>(d_q);
  // plain quantizer chain without a plain-output gradient: the reduce pass leaves a keep mask for a light dx pass
  const bool masked = !resid && quant && d_a == nullptr && dx != nullptr;
  {
    auto k = resid ? (quant ? bnq_bwd_reduce_kernel<T, true, true, 2, 3> : bnq_bwd_reduce_kernel<T, true, false, 2, 3>)
                   : (quant ? bnq_bwd_reduce_kernel<T, false, true, 4, 2> : bnq_bwd_reduce_kernel<T, false, false, 4, 3>);
    cudaError_t e = launch_pdl(k, dim3(g.nbx, g.gy), dim3(kBnqThreads), bnq_smem<VN>(g), st, xt, at, dat, dqt, gamma, beta,
                               smean, sinv, static_cast<T*>(dz_out), g, relu, sc, of, gq, lo, hi, w.part, w.part_s,
                               masked ? w.mask : static_cast<uint32_t*>(nullptr));
    if (e != cudaSuccess) return set_cuda_error(e);
  }
  {
    cudaError_t e = launch_pdl(bnq_bwd_finalize_kernel, dim3((g.C + 31) / 32 + 1), dim3(kBnqFoldWarps * 32), 0, st,
                               static_cast<const float*>(w.part), static_cast<const float*>(w.part_s), g,
                               quant ? g.nbx * g.gy : 0, training, gq, dgamma, dbeta, w.coef,
                               quant ? dscale : static_cast<float*>(nullptr));
    if (e != cudaSuccess) return set_cuda_error(e);
  }
  if (!dx) return DLMCQ_OK;
  const dim3 grid(apply_grid(g, 8), g.gy);
  cudaError_t e;
  if (resid || masked) {
    auto k = resid ? bnq_bwd_dx_light_kernel<T, false> : bnq_bwd_dx_light_kernel<T, true>;
    e = launch_pdl(k, grid, dim3(kBnqThreads), 0, st, xt, resid ? static_cast<const T*>(dz_out) : dqt,
                   static_cast<const uint32_t*>(w.mask), gamma, beta, smean, sinv, static_cast<const float*>(w.coef),
                   static_cast<T*>(dx), g);
  } else {
    auto k = quant ? bnq_bwd_dx_kernel<T, true, 2> : bnq_bwd_dx_kernel<T, false, 3>;
    e = launch_pdl(k, grid, dim3(kBnqThreads), 0, st, xt, dat, dqt, gamma, beta, smean, sinv,
                   static_cast<const float*>(w.coef), static_cast<T*>(dx), g, relu, sc, of, gq, lo, hi);
  }
  if (e != cudaSuccess) return set_cuda_error(e);
  return DLMCQ_OK;
}

}  // namespace dlmcq

using namespace dlmcq;

extern "C" size_t dlmcq_bnq_workspace_bytes(const dlmcq_bnq_desc* d) {
  if (bnq_check(d) != DLMCQ_OK) return 0;
  const BnqGeom g = d->dtype == DLMCQ_F32 ? make_bnq_geom<float>(d->rows, d->channels)
                                          : make_bnq_geom<__nv_bfloat16>(d->rows, d->channels);
  return kWsHeaderBytes + bnq_ws_floats(g) * sizeof(float);
}

extern "C" int dlmcq_bnq_forward(const void* x, const void* identity, const float* gamma, const float* beta,
                                 float* running_mean, float* running_var, float* save_mean, float* save_invstd,
                                 void* a_out, void* q_out, const dlmcq_bnq_desc* desc, const dlmcq_qparams* qp,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  if (int e = bnq_check(desc)) return e;
  if (desc->rows == 0) return DLMCQ_OK;
  if (!x || !save_mean || !save_invstd || !workspace) return DLMCQ_EINVAL;
  const bool training = (desc->flags & DLMCQ_BNQ_TRAINING) != 0;
  if (!training && (!running_mean || !running_var)) return DLMCQ_EINVAL;
  if ((running_mean == nullptr) != (running_var == nullptr)) return DLMCQ_EINVAL;
  if (q_out && (!qp || !qp->scale || qp->form != DLMCQ_FORM_AFFINE)) return DLMCQ_EINVAL;
  if (((desc->flags & DLMCQ_BNQ_RESIDUAL) != 0) != (identity != nullptr)) return DLMCQ_EINVAL;
  if (!aligned16(x) || !aligned16(identity) || !aligned16(a_out) || !aligned16(q_out)) return DLMCQ_EALIGN;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return desc->dtype == DLMCQ_F32
             ? bnq_forward_t<float>(x, identity, gamma, beta, running_mean, running_var, save_mean, save_invstd, a_out,
                                    q_out, desc, qp, workspace, workspace_bytes, st)
             : bnq_forward_t<__nv_bfloat16>(x, identity, gamma, beta, running_mean, running_var, save_mean, save_invstd,
                                            a_out, q_out, desc, qp, workspace, workspace_bytes, st);
}

extern "C" int dlmcq_bnq_forward_codes(const void* x, const void* identity, const float* gamma, const float* beta,
                                       float* running_mean, float* running_var, float* save_mean, float* save_invstd,
                                       void* a_out, void* codes_out, const dlmcq_bnq_desc* desc,
                                       const dlmcq_qparams* qp, int encoding, void* workspace, size_t workspace_bytes,
                                       void* stream) {
  if (int e = bnq_check(desc)) return e;
  if (desc->flags & DLMCQ_BNQ_TRAINING) return DLMCQ_EUNSUPPORTED;      // an inference hand-off: no backward
  if (!qp || !qp->scale || qp->form != DLMCQ_FORM_AFFINE) return DLMCQ_EINVAL;
  if (int e = code_range_ok(qp, encoding)) return e;                    // unknown encoding: DLMCQ_EINVAL
  if (desc->rows == 0) return DLMCQ_OK;
  if (!x || !codes_out || !save_mean || !save_invstd || !workspace || !running_mean || !running_var) return DLMCQ_EINVAL;
  if (((desc->flags & DLMCQ_BNQ_RESIDUAL) != 0) != (identity != nullptr)) return DLMCQ_EINVAL;
  if (!aligned16(x) || !aligned16(identity) || !aligned16(a_out) || !aligned16(codes_out)) return DLMCQ_EALIGN;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return desc->dtype == DLMCQ_F32
             ? bnq_forward_t<float>(x, identity, gamma, beta, running_mean, running_var, save_mean, save_invstd, a_out,
                                    codes_out, desc, qp, workspace, workspace_bytes, st, encoding)
             : bnq_forward_t<__nv_bfloat16>(x, identity, gamma, beta, running_mean, running_var, save_mean,
                                            save_invstd, a_out, codes_out, desc, qp, workspace, workspace_bytes, st,
                                            encoding);
}

extern "C" int dlmcq_bnq_backward(const void* x, const void* a_saved, const void* d_a, const void* d_q,
                                  const float* gamma, const float* beta, const float* save_mean,
                                  const float* save_invstd, void* dx, void* dz_out, float* dgamma, float* dbeta,
                                  float* dscale, const dlmcq_bnq_desc* desc, const dlmcq_qparams* qp, void* workspace,
                                  size_t workspace_bytes, void* stream) {
  if (int e = bnq_check(desc)) return e;
  if (desc->rows == 0) return DLMCQ_OK;
  if (!x || !save_mean || !save_invstd || !workspace || (!d_a && !d_q)) return DLMCQ_EINVAL;
  const bool resid = (desc->flags & DLMCQ_BNQ_RESIDUAL) != 0;
  if (resid && (!a_saved || !dz_out)) return DLMCQ_EINVAL;
  if (d_q && (!qp || !qp->scale || !dscale || qp->form != DLMCQ_FORM_AFFINE)) return DLMCQ_EINVAL;
  if (!aligned16(x) || !aligned16(a_saved) || !aligned16(d_a) || !aligned16(d_q) || !aligned16(dx) || !aligned16(dz_out))
    return DLMCQ_EALIGN;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return desc->dtype == DLMCQ_F32
             ? bnq_backward_t<float>(x, a_saved, d_a, d_q, gamma, beta, save_mean, save_invstd, dx, dz_out, dgamma, dbeta,
                                     dscale, desc, qp, workspace, workspace_bytes, st)
             : bnq_backward_t<__nv_bfloat16>(x, a_saved, d_a, d_q, gamma, beta, save_mean, save_invstd, dx, dz_out,
                                             dgamma, dbeta, dscale, desc, qp, workspace, workspace_bytes, st);
}
