/* dlmcq.h - C ABI of the B200-native fake-quantization library (libdlmcq.so).
 *
 * This is the drop-in boundary for ONE hot path of ilur98/DLMC-QUANT: the weight /
 * activation fake-quantizers of dlmc/quantization/scalar (quantize, clamp, round,
 * dequantize), their STE / LSQ / RootQ backward, and the PTQ observers.  The reference
 * has no FFI (it is pure Python); every entry point below names the reference
 * expression (file:line under /root/reference) that it replaces, and INTEGRATION.md
 * shows the ctypes stub a maintainer would add at that line.
 *
 * Conventions
 *   - plain C: raw DEVICE pointers, sizes, a CUDA stream passed as void* (cudaStream_t).
 *   - no allocation and no host synchronisation on the device-pointer entry points: outputs
 *     and workspaces are provided by the caller and every launch goes to `stream`.  The only
 *     process state is a cached SM count; the host-buffer entries keep theirs in a caller-owned context.
 *   - returns DLMCQ_OK (0) or a negative dlmcq_status; CUDA launch errors are reported
 *     as DLMCQ_ECUDA and the text is available from dlmcq_last_cuda_error().
 *   - arithmetic is IEEE fp32, one rounding per reference op, no FMA contraction, true
 *     division, round-half-even: integer codes and fp32 outputs are bit-identical to the
 *     reference's eager PyTorch chain.  bf16 tensors are up-converted, computed in fp32
 *     and rounded once (RNE) on store.
 *   - tensor layout: a contiguous tensor viewed as [outer, channels, inner]; the channel
 *     of flat element i is (i / inner) % channels.  Per-tensor qparams: channels = 1.
 *     Weights [C, K] with ch_axis=0: outer=1, channels=C, inner=K.  Activations [B,C,H,W]
 *     with ch_axis=1: outer=B, channels=C, inner=H*W.  scale/offset/zp arrays hold
 *     `channels` floats.
 */
#ifndef DLMCQ_H_
#define DLMCQ_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DLMCQ_VERSION 100 /* 0.1.0 */

typedef enum {
  DLMCQ_OK = 0,
  DLMCQ_EINVAL = -1,     /* bad argument (null pointer, negative size, unknown enum) */
  DLMCQ_EALIGN = -2,     /* pointer not aligned to the element size */
  DLMCQ_EWORKSPACE = -3, /* workspace too small (see dlmcq_workspace_bytes) */
  DLMCQ_ECUDA = -4,      /* CUDA runtime reported an error at launch */
  DLMCQ_EUNSUPPORTED = -5
} dlmcq_status;

typedef enum { DLMCQ_F32 = 0, DLMCQ_BF16 = 1 } dlmcq_dtype;

/* Which reference expression a fake-quant call reproduces. */
typedef enum {
  /* dlmc/quantization/scalar/utils.py:1-11  quantize()/emulate_quantize():
   *   codes = clamp(round((x-off)/(s+1e-7)), lo, hi);  y = codes*s + off          */
  DLMCQ_FORM_A1 = 0,
  /* dlmc/quantization/scalar/modules/base.py:96-102,131-133 (QBase, LSQ-style):
   *   s' = (s - s*g) + s*g;  codes = round_pass(clamp((x-off)/s', lo, hi));  y = codes*s' + off */
  DLMCQ_FORM_AFFINE = 1,
  /* dlmc/quantization/scalar/FSPTQuant/base.py:108-109 (integer zero-point):
   *   codes = clamp(round_pass(x/s) + zp, lo, hi);  y = (codes - zp)*s            */
  DLMCQ_FORM_ZP = 2,
  /* dlmc/quantization/scalar/FSPTQuant/base.py:149-152 (symmetric, per-channel weights):
   *   codes = clamp(round_pass(w/s), lo, hi);  y = codes*s                        */
  DLMCQ_FORM_SYM = 3
} dlmcq_form;

/* A contiguous tensor viewed as [outer, channels, inner]. */
typedef struct {
  int64_t outer;
  int64_t channels;
  int64_t inner;
  int32_t dtype; /* dlmcq_dtype of x / y / dy / dx */
} dlmcq_layout;

/* Quantisation parameters.  `scale` and `offset` are DEVICE arrays of layout.channels
 * floats (offset may be NULL = 0; for FORM_ZP it is the zero-point).  They stay on the
 * device so that learnable scales never force a host sync. */
typedef struct {
  int32_t form;        /* dlmcq_form */
  int32_t lo, hi;      /* integer clamp range, utils.py:14-22 get_qrange() */
  float g;             /* grad_scale factor 1/sqrt(numel*qmax) (FORM_AFFINE only) */
  const float* scale;
  const float* offset;
} dlmcq_qparams;

int dlmcq_version(void);
/* Diagnostic: compares the kernels' residual-corrected division (x*r, fma, fma with r = RN(1/s))
 * bitwise with IEEE division on blocks*256*per_thread*3 pseudo-random (x, s) pairs inside the
 * fast-path domain (2^-40<=|s|<=2^40, |x|<=2^60; quotients below 2^-100 only have to stay below
 * 2^-99); *mismatches_dev (zeroed by the caller) receives the count - expected 0. */
int dlmcq_selftest_fastdiv(uint64_t seed, int blocks, int per_thread, int narrow,
                           unsigned long long* mismatches_dev, void* stream);
const char* dlmcq_status_string(int status);
const char* dlmcq_last_cuda_error(void);

/* Bytes of zero-initialised device workspace the backward / observer entry points need
 * for this layout.  The library leaves the workspace zeroed again when a call finishes,
 * so one allocation (zeroed once) can be reused by successive calls on the same stream. */
size_t dlmcq_workspace_bytes(const dlmcq_layout* layout);

/* ---- fake-quant forward --------------------------------------------------------------
 * Replaces the eager chains at modules/base.py:102,133; FSPTQuant/base.py:108-109,149-152;
 * utils.py:1-11.  `y` (dequantised) and `codes` (fp32/bf16-valued integers) may each be
 * NULL; at least one must be given.  x may alias y. */
int dlmcq_fq_forward(const void* x, void* y, void* codes, const dlmcq_layout* layout,
                     const dlmcq_qparams* qp, void* stream);

/* ---- fake-quant backward -------------------------------------------------------------
 * One pass over (x, dy): writes dx and the reduced scale gradient dscale[channels]
 * (and, if doffset != NULL, the offset / zero-point gradient doffset[channels]).
 * Replaces autograd through the chains above (FORM_AFFINE: dscale includes the factor g;
 * FORM_ZP / FORM_SYM: plain sum; FORM_A1: FunLSQ.backward, modules/function.py:38-47,
 * strict masks, offset ignored, dscale includes g).  Deterministic: block partials are
 * combined in a fixed order by the last block to finish. */
int dlmcq_fq_backward(const void* x, const void* dy, void* dx, float* dscale, float* doffset,
                      const dlmcq_layout* layout, const dlmcq_qparams* qp,
                      void* workspace, size_t workspace_bytes, void* stream);

/* Deferred reduction for per-tensor layouts: dlmcq_fq_backward_partials writes dx and leaves the per-CTA
 * partial sums in `partials` (dlmcq_fq_partials_floats() floats, no initialisation needed) instead of
 * finalising in-kernel; dlmcq_fq_finalize_many then reduces any number of such calls - e.g. all layers
 * of a training step - in ONE launch, in a fixed order (deterministic).  `items` is a DEVICE array. */
typedef struct {
  const float* partials; /* as written by dlmcq_fq_backward_partials */
  float* dscale;         /* [1]; the offset gradient is not produced in deferred mode */
} dlmcq_finalize_item;
size_t dlmcq_fq_partials_floats(void);
int dlmcq_fq_backward_partials(const void* x, const void* dy, void* dx, const dlmcq_layout* layout,
                               const dlmcq_qparams* qp, float* partials, void* stream);
int dlmcq_fq_finalize_many(const dlmcq_finalize_item* items, int n_items, void* stream);

/* Diagnostic: the number of per-tensor (channels == 1, 16-byte aligned) forward / backward launches that this
 * thread captured into a CUDA graph as independent of their predecessor since the previous call, then resets it.
 * Such a launch directly follows another of these launches in the same capture sequence, and it reads nothing
 * that launch writes; its CTAs then load their first tile while the predecessor is still running.  Eager
 * launches never count. */
int dlmcq_capture_overlap_count(void);

/* utils.py:29-37 round_pass / floor_pass values and RootQ/function.py:5-8 sgn:
 * mode 0: (round(x)-x)+x   mode 1: (floor(x)-x)+x   mode 2: sign(x) (sign(NaN)=0) */
int dlmcq_ste_value(const void* x, void* y, int64_t numel, int dtype, int mode, void* stream);
/* utils.py:24-27 grad_scale value (s - s*g) + s*g for numel scales */
int dlmcq_grad_scale_value(const float* s, float* out, int64_t numel, float g, void* stream);

/* dequantize(): utils.py:5-6   y = codes*scale + offset */
int dlmcq_dequantize(const void* codes, void* y, const dlmcq_layout* layout,
                     const float* scale, const float* offset, void* stream);

/* ---- integer export (SURVEY.md 8f-f4; the reference only ever holds fp32-valued codes) ----------------
 * dlmcq_export_codes: the integer codes of any form as one byte per element (int8 two's complement when
 * qp->lo < 0, else uint8) or, with pack4 != 0 and a range that fits 4 bits, two codes per byte (low
 * nibble = even element).  dlmcq_import_codes unpacks and dequantises: its output is bit-identical to
 * dlmcq_fq_forward's y for the same qparams.  `layout->dtype` is the dtype of x / y. */
int dlmcq_export_codes(const void* x, void* codes_out, const dlmcq_layout* layout, const dlmcq_qparams* qp,
                       int pack4, void* stream);
int dlmcq_import_codes(const void* codes, void* y, const dlmcq_layout* layout, const dlmcq_qparams* qp,
                       int pack4, void* stream);

/* ---- AdaRound weight form (FSPTQuant/base.py:69-79,136-141,151-152) -------------------
 * soft=1: codes = clamp(floor(w/s) + clamp(sigmoid(alpha)*1.2-0.1,0,1), lo, hi)
 * soft=0: codes = clamp(floor(w/s) + (alpha>=0), lo, hi);       y = codes*s
 * backward (soft only): dscale[c] = sum dy*codes, dalpha elementwise; dw is identically 0. */
int dlmcq_adaround_forward(const void* w, const void* alpha, void* y, const dlmcq_layout* layout,
                           const float* scale, int lo, int hi, int soft, void* stream);
int dlmcq_adaround_backward(const void* w, const void* alpha, const void* dy, void* dalpha,
                            float* dscale, const dlmcq_layout* layout, const float* scale,
                            int lo, int hi, void* workspace, size_t workspace_bytes, void* stream);
/* init_alpha(): FSPTQuant/base.py:73-76 */
int dlmcq_adaround_init_alpha(const void* w, void* alpha, const dlmcq_layout* layout,
                              const float* scale, void* stream);

/* ---- RootQ (RootQ/base.py:77-156, RootQ/function.py) ----------------------------------
 * State block written by the *_prepare calls and consumed by forward/backward (device):
 *   act: [0]=sr' (effective scale) [1]=upper=sr'*Q [2]=g [3]=m [4]=Q
 *   wt : [0]=U [1]=L [2]=delta [3]=alpha' [4]=g [5]=m [6]=1[1e-4<alpha<1] [7]=Q
 * momentum and g are the reference's python doubles; (1-m), (1-g) are formed in double and
 * rounded to fp32 exactly where the eager chain does it. */
#define DLMCQ_ROOTQ_STATE_FLOATS 8

/* RootQ/base.py:92-106: EMA + gradient-mix of the activation scale; updates run_scale in
 * place when training (:101). */
int dlmcq_rootq_act_prepare(const float* in_scale, float* run_scale, double momentum, double g,
                            int lo, int hi, int training, float* state, void* stream);
/* RootQ/base.py:108-111 */
int dlmcq_rootq_act_forward(const void* x, void* y, int64_t numel, int dtype,
                            const float* state, void* stream);
int dlmcq_rootq_act_backward(const void* x, const void* dy, void* dx, float* d_in_scale,
                             int64_t numel, int dtype, const float* state,
                             void* workspace, size_t workspace_bytes, void* stream);
/* RootQ/base.py:131-145 */
int dlmcq_rootq_wt_prepare(const float* upper, const float* lower, const float* alpha,
                           float* run_upper, float* run_lower, double momentum, double g,
                           int lo, int hi, int training, float* state, void* stream);
/* RootQ/base.py:146-155 */
int dlmcq_rootq_wt_forward(const void* w, void* y, int64_t numel, int dtype,
                           const float* state, void* stream);
/* grads[0..2] = d wt_upper, d wt_lower, d wt_alpha */
int dlmcq_rootq_wt_backward(const void* w, const void* dy, void* dw, float* grads,
                            int64_t numel, int dtype, const float* state,
                            void* workspace, size_t workspace_bytes, void* stream);

/* Grouped RootQ launches: the scalar prologues (RootQ/base.py:92-101,131-147) of ALL quantizers of a model
 * in one launch, and all weight tensors quantised / differentiated in one launch each (the per-layer calls
 * above cost 6 launches per layer per step).  Descriptor tables live in DEVICE memory.
 *   prep: is_weight = 0: param_a = in_scale, run_a = in_run_scale (param_b, run_b, alpha unused);
 *         is_weight = 1: param_a/b = wt_upper/wt_lower, run_a/b = wt_run_upper/wt_run_lower, alpha = wt_alpha.
 *   item: x = w, y = w_q (forward) or dw (backward), dy = upstream gradient (backward), state = the prepared
 *         block, grads[3] = d wt_upper, d wt_lower, d wt_alpha.
 *   unit_prefix[k] = sum_{j<k} ceil(numel_j / DLMCQ_ROOTQ_UNIT), k = 0..n_items; partials: 3*total_units floats. */
#define DLMCQ_ROOTQ_UNIT 2048
typedef struct {
  const float *param_a, *param_b, *alpha;
  float *run_a, *run_b;
  float* state;
  double momentum, g;
  int32_t lo, hi, training, is_weight;
} dlmcq_rootq_prep;
typedef struct {
  const void* x;
  void* y;
  const void* dy;
  const float* state;
  float* grads;
  int64_t numel;
} dlmcq_rootq_item;
int dlmcq_rootq_prepare_many(const dlmcq_rootq_prep* items, int n_items, void* stream);
int dlmcq_rootq_wt_forward_grouped(const dlmcq_rootq_item* items, const int64_t* unit_prefix, int n_items,
                                   int64_t total_units, int dtype, void* stream);
int dlmcq_rootq_wt_backward_grouped(const dlmcq_rootq_item* items, const int64_t* unit_prefix, int n_items,
                                    int64_t total_units, int dtype, float* partials, void* stream);
/* The same launches for ACTIVATION quantizers (RootQ/base.py:92-111): several activation tensors that are resident at
 * the same time - the tensor a residual block feeds to both its first convolution and its shortcut convolution
 * (two quantizers, two in_scales), cached calibration activations, the quantizer set of BASELINE configs[0] - go
 * through one launch per direction.  item: x, y = x_q (forward) or dx (backward), dy, state = the block written by
 * dlmcq_rootq_act_prepare / _prepare_many, grads[1] = d in_scale.  partials: 3*total_units floats. */
int dlmcq_rootq_act_forward_grouped(const dlmcq_rootq_item* items, const int64_t* unit_prefix, int n_items,
                                    int64_t total_units, int dtype, void* stream);
int dlmcq_rootq_act_backward_grouped(const dlmcq_rootq_item* items, const int64_t* unit_prefix, int n_items,
                                     int64_t total_units, int dtype, float* partials, void* stream);

/* ---- observers (dlmc/quantization/scalar/ops.py) --------------------------------------
 * Statistics pass: one read of the tensor -> stats[channels][4] = {min, max, max|x|, sum|x|}
 * (NaN-propagating like torch.min/max).  Multi-GPU callers all-reduce `stats` between this
 * call and the *_finalize call. */
#define DLMCQ_STATS_PER_CHANNEL 4
#define DLMCQ_STATS_ABS_INPUT 1 /* take |x| first (quantize_minmax_pixel unsigned branch, ops.py:156-159) */
int dlmcq_obs_stats(const void* x, float* stats, const dlmcq_layout* layout, int flags,
                    void* workspace, size_t workspace_bytes, void* stream);
/* ops.py:20-34,121-140 (minmax_tensor / minmax_channel): signed: s = absmax/(2^(n-1)-1), off=0;
 * unsigned: s = (max-min)/(2^n-1), off = min (or 0 when allow_offset==0). */
int dlmcq_obs_minmax_finalize(const float* stats, float* scale, float* offset, int64_t channels,
                              int n_bits, int is_signed, int allow_offset, void* stream);
/* Same with the divisor convention made explicit.  `x / python_scalar` is not the same float32 operation on the two
 * devices the reference runs on: the CPU kernel divides (IEEE), the CUDA kernel multiplies by the float32 reciprocal of
 * the scalar (ATen BinaryDivTrueKernel.cu) - up to 1 ulp apart.  DLMCQ_DIV_IEEE reproduces the reference on the CPU
 * (what the committed fixtures pin; dlmcq_obs_minmax_finalize uses it), DLMCQ_DIV_CUDA_EAGER reproduces the reference
 * evaluated by eager PyTorch on the GPU, bit for bit (tests/test_gpu_parity_edges.py). */
#define DLMCQ_DIV_IEEE 0
#define DLMCQ_DIV_CUDA_EAGER 1
int dlmcq_obs_minmax_finalize_mode(const float* stats, float* scale, float* offset, int64_t channels,
                                   int n_bits, int is_signed, int allow_offset, int scalar_div_mode, void* stream);
/* mean|x| based initialisers; `count` = elements behind each stats row.
 *   mode 0: out = (mul_a*mean)/mul_b   modules/base.py:84,119 LSQ init 2*mean|x|/sqrt(qmax)
 *   mode 1: out = (mul_a*mean)*mul_b   RootQ/base.py:115-116   +-2*mean|w|*sqrt(qmax)        */
int dlmcq_obs_absmean_finalize(const float* stats, float* out, int64_t channels, double count,
                               double mul_a, double mul_b, int mode, void* stream);

/* Percentile-clipping observer (named by the north star; the reference's ops.py has no counterpart, so the
 * semantics are defined here and pinned against torch.kthvalue): EXACT order statistics by a 3-pass radix
 * select - value_j = the rank_j-th smallest element (1-based) of x, or of |x| with DLMCQ_STATS_ABS_INPUT;
 * NaN sorts last, -0 == +0.  Up to two ranks share the passes (lower / upper percentile).
 *   dlmcq_obs_kth_begin(state, rank0, rank1 /0 = unused/)
 *   for pass in 0,1,2:  dlmcq_obs_kth_hist(x, ..., pass, state)   one read of x; histogram of key digit `pass`
 *                       [multi-GPU: all-reduce(SUM) the 2*2048 uint32 counters at state+256]
 *                       dlmcq_obs_kth_select(pass, state)
 *   dlmcq_obs_kth_values(state, values[2])
 * state: dlmcq_obs_kth_state_bytes() bytes of DEVICE memory; no host synchronisation anywhere. */
size_t dlmcq_obs_kth_state_bytes(void);
int dlmcq_obs_kth_begin(void* state, int64_t rank0, int64_t rank1, void* stream);
int dlmcq_obs_kth_hist(const void* x, int64_t numel, int dtype, int flags, int pass, void* state, void* stream);
int dlmcq_obs_kth_select(int pass, void* state, void* stream);
int dlmcq_obs_kth_values(const void* state, float* values, void* stream);

/* The same order statistics in ONE full read (single GPU): the k-th element is bracketed from 16 384 pseudo-randomly
 * placed samples, the read counts what lies below the bracket and collects the few elements inside it, and an exact
 * radix select over those candidates gives the answer.  values[] are exact in every case: if the bracket missed or
 * the candidate buffer overflowed (probability ~1e-9 per call on ordinary data; any adversarially ordered input)
 * the same cooperative launch runs the three-digit select over the whole tensor instead.  *status (device) only
 * reports which happened: 1 = the bracket held (one read), 0 = the in-kernel full select ran (four reads).  Returns
 * DLMCQ_EUNSUPPORTED for numel < 65 536 (use the three-pass form).  The sample decides the speed, never the value. */
size_t dlmcq_obs_kth_fast_workspace_bytes(int64_t numel);
int dlmcq_obs_kth_fast(const void* x, int64_t numel, int dtype, int flags, int64_t rank0, int64_t rank1, float* values,
                       int32_t* status, void* workspace, size_t workspace_bytes, void* stream);
/* One entry for the observer: dlmcq_obs_kth_fast for numel >= 65536 (exact whether or not its bracket held), the
 * three-pass select below that.  state: dlmcq_obs_kth_state_bytes() bytes; scratch: dlmcq_obs_kth_fast_workspace_bytes
 * (numel) bytes (may be NULL / 0 for numel < 65536).  Stream-ordered, no host read; *status ends as 1 when the one-read
 * path's bracket held. */
int dlmcq_obs_kth_auto(const void* x, int64_t numel, int dtype, int flags, int64_t rank0, int64_t rank1, float* values,
                       int32_t* status, void* state, void* scratch, size_t scratch_bytes, void* stream);

/* ops.py:36-68 quantize_l2loss_tensor (unsigned branch): 80-candidate clip-ratio sweep.
 * Pass 1 (dlmcq_obs_stats) gives min/max; this pass accumulates the 80 squared-error sums
 * sse[80] in one read of x; the finalize picks the first strict minimum below 1000 of
 * sse[i]/rows_for_mean (l2_loss = sum over axis 1, mean over the rest).  */
#define DLMCQ_SWEEP_CANDIDATES 80
int dlmcq_obs_sweep_tensor_sse(const void* x, int64_t numel, int dtype, const float* stats,
                               int n_bits, int allow_offset, float* sse,
                               void* workspace, size_t workspace_bytes, void* stream);
int dlmcq_obs_sweep_tensor_finalize(const float* sse, const float* stats, double rows_for_mean,
                                    int n_bits, int allow_offset, float* scale, float* offset,
                                    int32_t* picked, void* stream);
/* ops.py:169-196 quantize_l2loss_channel on rows [channels, inner]: whole search per channel
 * in one launch, each row staged once in shared memory (bulk async copy) and swept 80 times
 * on chip.  Reproduces the reference's aliasing of the running minimum with the offset vector
 * and its disregard of `signed` in the search. */
int dlmcq_obs_sweep_channel(const void* x, int64_t channels, int64_t inner, int dtype,
                            int n_bits, int is_signed, float* scale, float* offset, void* stream);
/* Same, for one rank's block of `channels` rows out of a matrix of `geom_channels` rows (per-channel
 * observers sharded by output channel, SURVEY.md 8e): the launch geometry - and with it the order in which
 * a row's squared errors are summed - is chosen from geom_channels, so every row gets bit-identical qparams
 * whichever rank sweeps it. */
int dlmcq_obs_sweep_channel_geom(const void* x, int64_t channels, int64_t inner, int dtype, int n_bits,
                                 int is_signed, int64_t geom_channels, float* scale, float* offset,
                                 void* stream);

/* All per-channel sweeps of a model in ONE launch (the 23-54 weight tensors of a CNN cost 50-150 us each when swept
 * one by one).  Fill x / scale / offset / channels / inner / n_bits / is_signed, let dlmcq_obs_sweep_channel_plan choose
 * the launch geometry of each item (the same the per-tensor call uses, hence bit-identical results), build
 * cta_prefix[k] = sum_{j<k} ctas_j (k = 0..n_items-1) and copy both tables to DEVICE memory; smem_bytes = the largest
 * smem_bytes of the items in the launch (callers may split a model into launches by shared-memory class). */
typedef struct {
  const void* x;
  float* scale;  /* [channels] */
  float* offset; /* [channels] */
  int64_t channels, inner;
  int32_t n_bits, is_signed;
  int32_t wpr, row_floats, staged, pad; /* filled by dlmcq_obs_sweep_channel_plan */
  int64_t smem_bytes, ctas;             /* filled by dlmcq_obs_sweep_channel_plan */
} dlmcq_sweep_item;
int dlmcq_obs_sweep_channel_plan(dlmcq_sweep_item* item_host, int64_t geom_channels);
int dlmcq_obs_sweep_channel_grouped(const dlmcq_sweep_item* items, const int64_t* cta_prefix, int n_items,
                                    int64_t total_ctas, int dtype, int64_t smem_bytes, void* stream);

/* ops.py:71-83,198-215 l2norm fixed point, one iteration over rows [channels, inner]
 * (channels=1 for the per-tensor form):
 *   q = A1 codes(x, scale, offset);  new_scale[c] = sum(x*q)/sum(q*q + 1e-7)
 *   *diff = |new-s|/s (channels==1) or ||new-s||_2/||s||_2;  if *done is already set the call
 *   is a no-op; it sets *done when diff <= 1e-5 and then leaves `scale` = the converged value.
 * The caller launches iterations back to back and polls `done` every few launches. */
int dlmcq_obs_l2norm_step(const void* x, int64_t channels, int64_t inner, int dtype,
                          float* scale, const float* offset, int lo, int hi,
                          float* diff, int32_t* done, int32_t* iters,
                          void* workspace, size_t workspace_bytes, void* stream);

/* The whole fixed-point loop in ONE launch for tensors that fit in the GPU's shared memory (channels * ceil(inner/2048)
 * <= 24 * #SMs staged 8 KB items, i.e. up to ~7 M elements - every per-channel CNN weight matrix): rows are staged on
 * chip once and iterated there, convergence is decided on the device (grid barriers, cooperative launch), no HBM
 * re-reads and no host polling.  `scale` holds the starting scales and receives the result; *iters the iteration count,
 * *done whether `diff <= 1e-5` was reached within max_iters, *diff the last convergence measure.
 * Returns DLMCQ_EUNSUPPORTED when the tensor is too large to be resident (use dlmcq_obs_l2norm_step then). */
int dlmcq_obs_l2norm_resident(const void* x, int64_t channels, int64_t inner, int dtype, float* scale,
                              const float* offset, int lo, int hi, int max_iters, float* diff, int32_t* done,
                              int32_t* iters, void* workspace, size_t workspace_bytes, void* stream);

/* ---- grouped (multi-tensor) launches --------------------------------------------------
 * All weight tensors of a model in ONE launch: the per-layer tensors of a CNN (<= 9.4 MB)
 * are launch-latency-bound on B200 when quantised one by one.  `items` is a DEVICE array. */
#define DLMCQ_GROUP_SEG 4096 /* elements per work unit (one warp) */
typedef struct {
  const void* x;
  void* y;            /* forward: output; backward: dx */
  const void* dy;     /* backward only */
  const float* scale; /* [channels] */
  const float* offset;/* [channels] or NULL */
  float* dscale;      /* backward only, [channels] */
  int64_t channels;   /* rows of this tensor (1 = per-tensor qparams) */
  int64_t inner;      /* elements per row */
  int32_t form, lo, hi;
  float g;
} dlmcq_group_item;
/* unit_prefix[k] = sum_{j<k} channels_j * ceil(inner_j / DLMCQ_GROUP_SEG), k = 0..n_items (DEVICE);
 * chan_prefix[k] = sum_{j<k} channels_j (DEVICE); partials: total_units floats (DEVICE). */
int dlmcq_fq_forward_grouped(const dlmcq_group_item* items, const int64_t* unit_prefix, int n_items,
                             int64_t total_units, int dtype, void* stream);
int dlmcq_fq_backward_grouped(const dlmcq_group_item* items, const int64_t* unit_prefix,
                              const int64_t* chan_prefix, int n_items, int64_t total_units,
                              int64_t total_channels, int dtype, float* partials, void* stream);

/* ---- BN folding / RepVGG re-parameterisation feeding the per-channel observers ----------
 * dlmc/utils/merge_bn.py:84-100 (mode MERGE_BN) and model/classification/repvgg.py:92-123
 * (mode REPVGG), for every layer of a model in ONE launch: one warp per (layer, output channel)
 * writes the folded weight row and bias and - when `stats` is set - the row's
 * {min, max, max|w|, sum|w|}, i.e. the input of dlmcq_obs_minmax_finalize (ops.py:121-140), so the
 * observer never re-reads the folded weights.  fp32 only; w_out may alias w (merge_bn folds in place).
 *   MERGE_BN: var = running_var + 1e-7; w' = (w*gamma)/sqrt(var); b' = (gamma*(b-mean))/sqrt(var) + beta
 *             (bias == NULL: zeros, merge_bn.py:92-94).
 *   REPVGG:   std_k = sqrt(var_k + eps_k), t_k = gamma_k/std_k, bias_k = beta_k - (mean_k*gamma_k)/std_k;
 *             w' = (k3*t3 + pad(k1*t1)) + id*t_id; b' = (bias3 + bias1) + bias_id; gamma_id == NULL when
 *             the block has no identity branch (the reference then adds the integer 0). */
typedef enum { DLMCQ_FOLD_MERGE_BN = 0, DLMCQ_FOLD_REPVGG = 1 } dlmcq_fold_mode;
typedef struct {
  const float* w;      /* [channels, inner] conv weight (RepVGG: the 3x3 branch) */
  const float* bias;   /* [channels] or NULL (MERGE_BN only) */
  const float *gamma, *beta, *mean, *var;             /* BatchNorm of w */
  const float* w1;     /* REPVGG: [channels, cin_g] 1x1-branch weight */
  const float *gamma1, *beta1, *mean1, *var1;         /* REPVGG: BatchNorm of the 1x1 branch */
  const float *gamma_id, *beta_id, *mean_id, *var_id; /* REPVGG: identity BatchNorm, or all NULL */
  float* w_out;        /* [channels, inner] */
  float* bias_out;     /* [channels] */
  float* stats;        /* [channels, 4] or NULL */
  int64_t channels, inner; /* inner = cin_g * ksize * ksize */
  int32_t cin_g, ksize;    /* REPVGG: input channels per group, 3 */
  int32_t mode;            /* dlmcq_fold_mode */
  float eps, eps1, eps_id; /* REPVGG: the BatchNorms' eps */
} dlmcq_fold_item;
/* items: n_items descriptors (DEVICE); chan_prefix[k] = sum_{j<k} channels_j, k = 0..n_items (DEVICE). */
int dlmcq_fold_grouped(const dlmcq_fold_item* items, const int64_t* chan_prefix, int n_items,
                       int64_t total_channels, void* stream);

/* ---- activation fake-quant fused into its producer (SURVEY.md 8f row f2) ----------------
 * BatchNorm (+ residual add) (+ ReLU) -> QBase input fake-quant, for CHANNELS-LAST tensors: a dense [rows, channels]
 * matrix, channels innermost (a channels_last NCHW activation with rows = N*H*W, or a [N, C] matrix).  Replaces the
 * chain nn.BatchNorm2d -> (out += identity) -> nn.ReLU -> QBase.forward's input branch
 * (dlmc/quantization/scalar/modules/base.py:96-102, reached from modules/conv.py:13-19) and its autograd:
 *     z = (x - mean) * (gamma * invstd) + beta [+ identity];   a = relu(z) or z;
 *     a_q = FORM_AFFINE fake-quant of a with the CONSUMER layer's in_scale / in_offset (per-tensor)
 * forward : training -> batch statistics (biased variance for normalising, unbiased for the running buffer, momentum
 *           update in place, exactly nn.BatchNorm2d); eval -> the running buffers.  save_mean / save_invstd
 *           [channels] are written either way and are what the backward call needs.  a_out and q_out may each be
 *           NULL (both NULL: statistics only).  qp is required when q_out is given: form must be FORM_AFFINE,
 *           scale / offset point to ONE float each.
 * backward: d_a = gradient w.r.t. a_out (NULL if none), d_q = gradient w.r.t. q_out (NULL if none) ->
 *           dx, dgamma[channels], dbeta[channels] (either may be NULL), dscale[1] (with d_q; includes the factor g).
 *           With DLMCQ_BNQ_RESIDUAL the saved plain output a_saved is read instead of recomputing a (z contains
 *           the identity), and dz_out - the gradient of z, which IS the gradient of the identity input - is written.
 * Given a, a_q is bit-identical to dlmcq_fq_forward(a); BatchNorm itself is floating-point reduction work and agrees
 * with a library batch-norm within reduction-order tolerance.  Deterministic (fixed-order reductions, no atomics).
 * channels must be a multiple of 4 (fp32) / 8 (bf16) and all tensor pointers 16-byte aligned, otherwise
 * DLMCQ_EUNSUPPORTED / DLMCQ_EALIGN (callers then run the unfused chain).  Workspace: dlmcq_bnq_workspace_bytes(),
 * no initialisation needed. */
#define DLMCQ_BNQ_TRAINING 1
#define DLMCQ_BNQ_RELU 2
#define DLMCQ_BNQ_RESIDUAL 4
typedef struct {
  int64_t rows;     /* N*H*W */
  int64_t channels; /* C (innermost) */
  int32_t dtype;    /* dlmcq_dtype of x / identity / a / a_q / gradients */
  int32_t flags;    /* DLMCQ_BNQ_* */
  float eps;        /* nn.BatchNorm2d.eps */
  float momentum;   /* nn.BatchNorm2d.momentum (training) */
} dlmcq_bnq_desc;
size_t dlmcq_bnq_workspace_bytes(const dlmcq_bnq_desc* desc);
int dlmcq_bnq_forward(const void* x, const void* identity, const float* gamma, const float* beta,
                      float* running_mean, float* running_var, float* save_mean, float* save_invstd,
                      void* a_out, void* q_out, const dlmcq_bnq_desc* desc, const dlmcq_qparams* qp,
                      void* workspace, size_t workspace_bytes, void* stream);
int dlmcq_bnq_backward(const void* x, const void* a_saved, const void* d_a, const void* d_q,
                       const float* gamma, const float* beta, const float* save_mean, const float* save_invstd,
                       void* dx, void* dz_out, float* dgamma, float* dbeta, float* dscale,
                       const dlmcq_bnq_desc* desc, const dlmcq_qparams* qp, void* workspace,
                       size_t workspace_bytes, void* stream);

/* ---- host-buffer entries (end-to-end path), on a caller-owned context ----------------------
 * For callers whose tensors live in (pinned) HOST memory: per-tensor-scale fake-quant forward + backward with the
 * H2D / kernel / D2H stages of successive chunks pipelined over the context's own streams.  A context owns its
 * streams, events and device staging memory; the library keeps NO process-global state for this path.  One context is
 * used by one thread at a time (calls on it are serialised); different contexts are independent.  The device current
 * at dlmcq_host_ctx_create() is the context's device.  chunk_elems: elements per pipeline chunk, a multiple of 8
 * (4 M is a good value: 4 staging buffers of chunk_elems * 4 bytes per pipeline slot, 4 slots).
 *
 * Both calls ENQUEUE and return: host outputs (including *dscale_host, which should be pinned) are valid after
 * dlmcq_host_ctx_synchronize().  Inputs must stay untouched until then.
 *   dlmcq_host_ctx_fq_forward_backward   x, dy in; y, dx out in the tensor's dtype - same arithmetic as
 *                                        dlmcq_fq_forward + dlmcq_fq_backward.
 *   dlmcq_host_ctx_fq_codes              compact, LOSSLESS result format (the path is PCIe-bound: 8.6 instead of 16
 *                                        bytes per fp32 element cross the bus): codes_host receives the integer codes,
 *                                        one byte each (two's complement when lo < 0) or two 4-bit codes per byte with
 *                                        pack4 (low nibble = even element) - y is code * s' + offset, exactly what
 *                                        dlmcq_import_codes returns; keep_host receives one bit per element (bit e of
 *                                        byte i/8, LSB first): dx = keep ? dy : 0 with the dy the caller holds.
 *                                        dy_host == NULL: forward only (keep_host, dscale_host unused). */
typedef struct dlmcq_host_ctx dlmcq_host_ctx;
int dlmcq_host_ctx_create(dlmcq_host_ctx** ctx, int64_t chunk_elems);
int dlmcq_host_ctx_destroy(dlmcq_host_ctx* ctx);
int dlmcq_host_ctx_synchronize(dlmcq_host_ctx* ctx);
int dlmcq_host_ctx_fq_forward_backward(dlmcq_host_ctx* ctx, const void* x_host, const void* dy_host, void* y_host,
                                       void* dx_host, float* dscale_host, int64_t numel, int dtype, int form, int lo,
                                       int hi, float g, float scale, float offset);
int dlmcq_host_ctx_fq_codes(dlmcq_host_ctx* ctx, const void* x_host, const void* dy_host, void* codes_host,
                            void* keep_host, float* dscale_host, int64_t numel, int dtype, int form, int lo, int hi,
                            float g, float scale, float offset, int pack4);

/* ---- the layer's matrix product on the integer codes (consumer side of the activation quantizer) ----------------
 * Replaces `_forward_func(q_input, q_weight)` = F.linear / a 1x1 F.conv2d on the two FAKE-QUANTISED fp32 tensors
 * (modules/linear.py, modules/conv.py, entered from modules/base.py:140; FSPTQuant/base.py:111-113) for a per-tensor
 * activation quantizer and a per-output-channel or per-tensor weight quantizer without an additive weight term:
 *     sum_k y_a[m,k] * y_w[n,k] = alpha[n] * (sum_k ca[m,k] * cw[n,k]) + beta[n]
 * with the exact integer dot product of the codes on the tcgen05 tensor cores (TMA-staged one-byte operands, TMEM
 * accumulators).  Activations are read at ONE byte per element instead of four.
 *   encoding DLMCQ_QGEMM_I8    one byte per code, uint8 (lo >= 0) or two's complement; tcgen05.mma kind::i8, s32
 *                              accumulators: exact for every range dlmcq_export_codes accepts (weights: hi <= 127)
 *   encoding DLMCQ_QGEMM_E4M3  the code as an e4m3 byte, kind::f8f6f4, fp32 accumulators: |code| <= 16 only
 *
 * dlmcq_codes_forward   x -> codes, one byte each; the same arithmetic (and therefore the same codes) as
 *                       dlmcq_fq_forward / dlmcq_export_codes for every form and layout; NaN -> 0.
 * dlmcq_qgemm_prepare   per output channel n, from DEVICE-resident qparams (no host sync; AFFINE scales go through
 *                       the grad_scale value like the fake-quant kernels):
 *                         alpha[n] = m_a * m_w[n]
 *                         beta[n]  = ((o_a - z_a*m_a) * m_w[n]) * float(sum_k cw[n,k])  (+ bias[n] if bias != NULL)
 *                       m: dequantisation multiplier, o_a: A1 / AFFINE offset, z_a: ZP zero-point.  wt_qp->offset
 *                       must be NULL and wt_qp->form != ZP (DLMCQ_EUNSUPPORTED otherwise: the product would not
 *                       factor); wt_channels = n (per output channel) or 1.  w_codes: [n, k] bytes, row-major.
 * dlmcq_qgemm           out[m,n] = RN(RN(float(acc[m,n]) * alpha[n]) + beta[n]), optionally max(., 0);
 *                       a_codes [m, k], w_codes [n, k] bytes row-major, 16-byte aligned, k % 16 == 0
 *                       (DLMCQ_EUNSUPPORTED otherwise); out [m, n] row-major fp32 / bf16 (a channels-last activation
 *                       [B,H,W,C] is exactly such a matrix with m = B*H*W).  a_signed: activation codes are int8. */
#define DLMCQ_QGEMM_I8 0
#define DLMCQ_QGEMM_E4M3 1
int dlmcq_codes_forward(const void* x, void* codes, const dlmcq_layout* layout, const dlmcq_qparams* qp, int encoding,
                        void* stream);
int dlmcq_qgemm_prepare(const void* w_codes, int64_t n, int64_t k, int encoding, const dlmcq_qparams* act_qp,
                        const dlmcq_qparams* wt_qp, int64_t wt_channels, const float* bias, float* alpha, float* beta,
                        void* stream);
int dlmcq_qgemm(const void* a_codes, const void* w_codes, const float* alpha, const float* beta, void* out, int64_t m,
                int64_t n, int64_t k, int encoding, int a_signed, int relu, int out_dtype, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DLMCQ_H_ */
