/* TEST INFRASTRUCTURE ONLY - plain C restatement of DLMC-QUANT's fake-quant hot path.
 *
 * Second, torch-free statement of the reference arithmetic: scalar loops, one separately rounded
 * fp32 operation per reference op (compile with -ffp-contract=off, no -ffast-math), gradients in
 * CLOSED FORM (SURVEY.md App. A) instead of autograd.  It is pinned against the same golden
 * fixtures as oracle/restate.py (tests/test_c_oracle.py): forward values bit-exact, closed-form
 * gradients against the reference's autograd results.  Product code never links this file.
 *
 * Citations are into /root/reference/dlmc/quantization/scalar/.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

/* torch.clamp on CPU: std::min(std::max(v, lo), hi) - NaN propagates, -0.0 kept */
static inline float clampf(float v, float lo, float hi) {
  float t = (v < lo) ? lo : v;
  return (hi < t) ? hi : t;
}
/* utils.py:29-32 round_pass value */
static inline float round_pass(float v) {
  float r = rintf(v);
  return (r - v) + v;
}
/* utils.py:34-37 floor_pass value */
static inline float floor_pass(float v) {
  float f = floorf(v);
  return (f - v) + v;
}
static inline float reluf(float v) { return (v > 0.f) ? v : ((v != v) ? v : 0.f); }
/* utils.py:24-27 grad_scale value */
static inline float grad_scale_value(float s, float g) {
  float sg = s * g;
  return (s - sg) + sg;
}
static inline int64_t chan_of(int64_t i, int64_t channels, int64_t inner) {
  return channels == 1 ? 0 : (i / inner) % channels;
}

float orc_grad_scale_value(float s, float g) { return grad_scale_value(s, g); }

/* form: 0 = utils.py:1-11 (A1), 1 = modules/base.py:96-102,131-133 (AFFINE),
 *       2 = FSPTQuant/base.py:108-109 (ZP), 3 = FSPTQuant/base.py:149-152 (SYM).
 * layout [outer, channels, inner]; offset may be NULL. */
void orc_fq_forward(const float* x, float* y, float* codes, int64_t n, int64_t channels, int64_t inner,
                    const float* scale, const float* offset, int form, float lo, float hi, float g) {
  for (int64_t i = 0; i < n; ++i) {
    int64_t c = chan_of(i, channels, inner);
    float s = scale[c], off = offset ? offset[c] : 0.f, code, out;
    if (form == 0) {
      code = clampf(rintf((x[i] - off) / (s + 1e-7f)), lo, hi);
      out = code * s + off;
    } else if (form == 1) {
      float sp = grad_scale_value(s, g);
      code = round_pass(clampf((x[i] - off) / sp, lo, hi));
      out = code * sp + off;
    } else if (form == 2) {
      code = clampf(round_pass(x[i] / s) + off, lo, hi);
      out = (code - off) * s;
    } else {
      code = clampf(round_pass(x[i] / s), lo, hi);
      out = code * s;
    }
    if (y) y[i] = out;
    if (codes) codes[i] = code;
  }
}

/* Closed-form backward (SURVEY.md A.2-A.4): dx and per-channel dscale (double accumulation). */
void orc_fq_backward(const float* x, const float* dy, float* dx, double* dscale, int64_t n, int64_t channels,
                     int64_t inner, const float* scale, const float* offset, int form, float lo, float hi, float g) {
  for (int64_t c = 0; c < channels; ++c) dscale[c] = 0.0;
  for (int64_t i = 0; i < n; ++i) {
    int64_t c = chan_of(i, channels, inner);
    float s = scale[c], off = offset ? offset[c] : 0.f;
    if (form == 0) { /* modules/function.py:38-47 FunLSQ.backward: strict masks, offset ignored */
      float q = x[i] / s;
      int below = q < lo, above = q > hi;
      float term = below ? lo : (above ? hi : (rintf(q) - q));
      dscale[c] += (double)(term * dy[i]);
      dx[i] = ((below || above) ? 0.f : 1.f) * dy[i];
    } else if (form == 1) {
      float sp = grad_scale_value(s, g);
      float u = (x[i] - off) / sp;
      int in = (u >= lo) && (u <= hi);
      float code = round_pass(clampf(u, lo, hi));
      dscale[c] += (double)dy[i] * (in ? (double)code - (double)u : (double)code);
      dx[i] = in ? dy[i] : 0.f;
    } else {
      float v = x[i] / s;
      float t = (form == 2) ? round_pass(v) + off : round_pass(v);
      int in = (t >= lo) && (t <= hi);
      float deq = (form == 2) ? clampf(t, lo, hi) - off : clampf(t, lo, hi);
      dscale[c] += (double)dy[i] * (in ? (double)deq - (double)v : (double)deq);
      dx[i] = in ? dy[i] : 0.f;
    }
  }
  if (form == 0 || form == 1)
    for (int64_t c = 0; c < channels; ++c) dscale[c] *= (double)g; /* utils.py:24-27 chain / FunLSQ "* g" */
}

/* ---- RootQ (RootQ/base.py:92-155, RootQ/function.py) ------------------------------------ */
/* activation: given the effective scale rs (after EMA + grad mix) and upper = rs*Q */
void orc_rootq_act(const float* x, const float* dy, float* y, float* dx, double* d_rs, int64_t n, float rs, float up,
                   float q) {
  double acc = 0.0;
  for (int64_t i = 0; i < n; ++i) {
    float nl = 0.f - x[i];
    float x1 = x[i] + reluf(nl);          /* function.py:17 */
    float ov = x1 - up;
    float xq = x1 - reluf(ov);            /* function.py:19 */
    float v = xq / rs;
    float I = round_pass(v);              /* base.py:109 */
    y[i] = I * rs;                        /* base.py:111 */
    if (dy) {
      int hi_clip = ov > 0.f;
      acc += (double)dy[i] * (((double)I - (double)v) + (hi_clip ? (double)q : 0.0));
      dx[i] = ((nl <= 0.f) && (ov <= 0.f)) ? dy[i] : 0.f;   /* relu' passes NaN: dx(NaN) = 0 */
    }
  }
  if (d_rs) *d_rs = acc;                  /* caller multiplies by m*g (base.py:95,97) */
}

/* EMA + gradient mix of a running scalar: base.py:95,97 / 137-140 */
float orc_rootq_mix(float run, float param, double momentum, double g) {
  float r = run * (float)(1.0 - momentum) + (float)momentum * param;
  return (float)g * r + (float)(1.0 - g) * r;
}

/* weight: U, L are the mixed running bounds; grads[0..2] = un-chained d/dU, d/dL, d/dalpha' */
void orc_rootq_wt(const float* w, const float* dy, float* y, float* dw, double* grads, int64_t n, float U, float L,
                  float alpha, float q) {
  float delta = (U - L) / q;              /* base.py:147 */
  float a1 = alpha + reluf(1e-4f - alpha);
  float a2 = a1 - reluf(a1 - 1.f);        /* function.py:25-26 */
  float k = 2.f / delta;
  double gU = 0.0, gL = 0.0, gA = 0.0;
  for (int64_t i = 0; i < n; ++i) {
    float lw = L - w[i];
    float x1 = w[i] + reluf(lw);
    float ov = x1 - U;
    float c = x1 - reluf(ov);             /* base.py:146 */
    float t = (c - L) / delta;
    float I = floor_pass(t);              /* base.py:148 */
    float mi = (I + 0.5f) * delta + L;    /* base.py:149 */
    float z = c - mi;
    float sig = (z > 0.f) ? 1.f : ((z < 0.f) ? -1.f : 0.f);
    float lsig = sig;                     /* level sign sgn(pow(b,a)*sg): sign(z) when delta > 0 (b >= 1e-5) */
    if (!(k > 0.f)) {                     /* U < L: b may be negative, pow NaN (sgn 0) or b itself (a == 1) */
      float p = powf(k * fabsf(z) + 1e-5f, a2) * (z / (fabsf(z) + 1e-5f));
      lsig = (p > 0.f) ? 1.f : ((p < 0.f) ? -1.f : 0.f);
    }
    y[i] = ((lsig + 1.f) / 2.f + I) * delta + L;               /* function.py:63-67 */
    if (dy) {
      int m_lo = lw > 0.f, m_hi = ov > 0.f;
      double dcw = (m_lo || m_hi) ? 0.0 : 1.0, cu = m_hi ? 1.0 : 0.0, cl = (m_lo && !m_hi) ? 1.0 : 0.0;
      double az = fabs((double)z), den = az + 1e-5, sg = (double)z / den;
      double b = (double)k * az + 1e-5, pw = pow(b, (double)a2), lb = log(b);
      double dpdz = (double)a2 * pw / b * (double)k * (double)sig * sg + pw * 1e-5 / (den * den);
      double dpdd = -((double)a2 * pw / b * (double)k * az * sg) / (double)delta;
      double dpda = pw * lb * sg;
      double lvl = ((double)lsig + 1.0) * 0.5 + (double)I, hd = (double)delta * 0.5, iq = 1.0 / (double)q;
      gA += (double)dy[i] * hd * dpda;
      gU += (double)dy[i] * (hd * (dpdz * cu + dpdd * iq) + (cu - (double)t * iq) + lvl * iq);
      gL += (double)dy[i] * (hd * (dpdz * cl - dpdd * iq) + (cl - 1.0 + (double)t * iq) - lvl * iq + 1.0);
      dw[i] = (float)((double)dy[i] * dcw * (1.0 + hd * dpdz));
    }
  }
  if (grads) { grads[0] = gU; grads[1] = gL; grads[2] = gA; }
}

/* ---- observers (ops.py) -------------------------------------------------------------------- */
/* ops.py:20-34 / 121-140 on rows [channels, inner] */
void orc_minmax(const float* x, int64_t channels, int64_t inner, int n_bits, int is_signed, float* scale,
                float* offset) {
  for (int64_t c = 0; c < channels; ++c) {
    const float* r = x + c * inner;
    float mn = r[0], mx = r[0], am = fabsf(r[0]);
    for (int64_t j = 1; j < inner; ++j) {
      if (r[j] < mn) mn = r[j];
      if (r[j] > mx) mx = r[j];
      if (fabsf(r[j]) > am) am = fabsf(r[j]);
    }
    if (is_signed) { scale[c] = am / (float)((1 << (n_bits - 1)) - 1); offset[c] = 0.f; }
    else { scale[c] = (mx - mn) / (float)((1 << n_bits) - 1); offset[c] = mn; }
  }
}

static void candidate(int i, float lo, float hi, float qmax, float* sc, float* zp) {
  float r = (float)(1.0 - 0.01 * (double)i);           /* ops.py:53-54 python double -> fp32 */
  float c_hi = r * hi, c_lo = r * lo;
  *sc = (c_hi - c_lo) / qmax;                          /* ops.py:55 */
  *zp = rintf((-c_lo) / *sc);                          /* ops.py:58 */
}
static double sse_of(const float* x, int64_t n, float sc, float zp, float qmax) {
  double s = 0.0;
  for (int64_t j = 0; j < n; ++j) {
    float q = rintf(x[j] / sc) + zp;                   /* ops.py:59 */
    q = (clampf(q, 0.f, qmax) - zp) * sc;              /* ops.py:60 */
    float d = q - x[j];
    s += (double)(d * d);
  }
  return s;
}
/* ops.py:36-68 unsigned branch; rows_for_mean = numel / shape[1] (l2_loss: sum axis 1, mean the rest) */
int orc_sweep_tensor(const float* x, int64_t n, double rows_for_mean, int n_bits, float* scale, float* offset,
                     double* losses) {
  float mn = x[0], mx = x[0];
  for (int64_t j = 1; j < n; ++j) { if (x[j] < mn) mn = x[j]; if (x[j] > mx) mx = x[j]; }
  float qmax = (float)((1 << n_bits) - 1);
  double best = 1000.0;
  int pick = -1;
  *scale = mx / qmax; *offset = 0.f;                   /* ops.py:49-50 */
  for (int i = 0; i < 80; ++i) {
    float sc, zp;
    candidate(i, mn, mx, qmax, &sc, &zp);
    double loss = sse_of(x, n, sc, zp, qmax) / rows_for_mean;
    if (losses) losses[i] = loss;
    if (loss < best) { best = loss; pick = i; *scale = sc; *offset = zp; }   /* ops.py:62-66 */
  }
  return pick;
}
/* ops.py:169-196 incl. the aliasing of min_val with offset and the disregard of `signed` */
void orc_sweep_channel(const float* x, int64_t channels, int64_t inner, int n_bits, int is_signed, float* scale,
                       float* offset) {
  float qmax = (float)((1 << n_bits) - 1);
  orc_minmax(x, channels, inner, n_bits, is_signed, scale, offset);
  for (int64_t c = 0; c < channels; ++c) {
    float min_v = offset[c];
    float max_v = offset[c] + scale[c] * qmax;         /* ops.py:173 */
    double best = 1000.0;
    for (int i = 0; i < 80; ++i) {
      float sc, zp;
      candidate(i, min_v, max_v, qmax, &sc, &zp);
      double loss = sse_of(x + c * inner, inner, sc, zp, qmax);
      if (best > loss) { scale[c] = sc; offset[c] = zp; min_v = zp; best = loss; }   /* ops.py:191-194 */
    }
  }
}
/* ops.py:71-83 per-tensor l2norm fixed point; returns the iteration count (bounded) */
int orc_l2norm_tensor(const float* x, int64_t n, int n_bits, int is_signed, int max_iters, float* scale,
                      float* offset) {
  orc_minmax(x, 1, n, n_bits, is_signed, scale, offset);
  float hi = is_signed ? (float)((1 << (n_bits - 1)) - 1) : (float)((1 << n_bits) - 1);
  float lo = is_signed ? -hi : 0.f;
  int it = 0;
  for (; it < max_iters; ++it) {
    double a = 0.0, b = 0.0;
    for (int64_t j = 0; j < n; ++j) {
      float q = clampf(rintf((x[j] - *offset) / (*scale + 1e-7f)), lo, hi);   /* utils.py:1-2 */
      a += (double)(x[j] * q);
      b += (double)(q * q + 1e-7f);
    }
    float ns = (float)a / (float)b;
    float diff = fabsf(ns - *scale) / *scale;
    *scale = ns;
    if (!(diff > 1e-5f)) { ++it; break; }
  }
  return it;
}

/* ---- weight-space re-parameterisation (SURVEY.md 8f, row f3) -----------------------------------------
 * sqrtf here is the correctly rounded IEEE square root (what torch computes on CUDA; torch's CPU sqrt goes
 * through MKL VML and is only faithfully rounded - see oracle/restate.py::sqrt_ieee). */

/* dlmc/utils/merge_bn.py:84-100: var = running_var + 1e-7; w' = (w*gamma)/sqrt(var);
 * b' = (gamma*(b-mean))/sqrt(var) + beta; bias == NULL -> zeros (:92-94) */
void orc_merge_bn(const float* w, const float* bias, const float* gamma, const float* beta, const float* mean,
                  const float* var, int64_t channels, int64_t inner, float* w_out, float* bias_out) {
  for (int64_t c = 0; c < channels; ++c) {
    const float v = var[c] + 1e-7f;
    const float sd = sqrtf(v);
    for (int64_t j = 0; j < inner; ++j) w_out[c * inner + j] = (w[c * inner + j] * gamma[c]) / sd;
    const float b = bias ? bias[c] : 0.f;
    bias_out[c] = (gamma[c] * (b - mean[c])) / sd + beta[c];
  }
}

/* model/classification/repvgg.py:92-123: bn* = gamma, beta, mean, var arrays (bn_id_gamma == NULL: no identity
 * branch, the reference then adds the integer 0); k3 [C, cin_g, 3, 3], k1 [C, cin_g] */
void orc_repvgg_fuse(const float* k3, const float* g3, const float* b3, const float* m3, const float* v3, float eps3,
                     const float* k1, const float* g1, const float* b1, const float* m1, const float* v1, float eps1,
                     const float* gi, const float* bi, const float* mi, const float* vi, float epsi,
                     int64_t channels, int64_t cin_g, float* w_out, float* bias_out) {
  for (int64_t c = 0; c < channels; ++c) {
    const float std3 = sqrtf(v3[c] + eps3), t3 = g3[c] / std3;
    const float bias3 = b3[c] - (m3[c] * g3[c]) / std3;
    const float std1 = sqrtf(v1[c] + eps1), t1 = g1[c] / std1;
    const float bias1 = b1[c] - (m1[c] * g1[c]) / std1;
    float tid = 0.f, biasid = 0.f;
    if (gi) {
      const float stdi = sqrtf(vi[c] + epsi);
      tid = gi[c] / stdi;
      biasid = bi[c] - (mi[c] * gi[c]) / stdi;
    }
    for (int64_t ci = 0; ci < cin_g; ++ci) {
      for (int p = 0; p < 9; ++p) {
        const int64_t j = (c * cin_g + ci) * 9 + p;
        const float a = k3[j] * t3;
        const float b = (p == 4) ? k1[c * cin_g + ci] * t1 : 0.f;                 /* F.pad(kernel1x1, [1,1,1,1]) */
        const float d = gi ? ((p == 4 && ci == c % cin_g) ? 1.f : 0.f) * tid : 0.f;  /* id_tensor * t, or + 0 */
        w_out[j] = (a + b) + d;
      }
    }
    bias_out[c] = (bias3 + bias1) + biasid;
  }
}

/* ---- percentile observer (extension, no reference counterpart): the k-th smallest value (1-based) of x or |x|,
 * NaN sorts last like torch.sort / torch.kthvalue, -0 == +0.  O(n log n) by sorting a copy. */
static int cmp_float_nan_last(const void* a, const void* b) {
  const float x = *(const float*)a, y = *(const float*)b;
  const int nx = x != x, ny = y != y;
  if (nx || ny) return nx - ny;
  return (x > y) - (x < y);
}
float orc_kth_value(const float* x, int64_t n, int64_t k, int abs_input) {
  float* t = (float*)malloc((size_t)n * sizeof(float));
  for (int64_t i = 0; i < n; ++i) t[i] = abs_input ? fabsf(x[i]) : x[i];
  qsort(t, (size_t)n, sizeof(float), cmp_float_nan_last);
  const float v = t[k - 1];
  free(t);
  return v;
}

/* ---- the layer product on the integer codes (oracle/restate.py::code_gemm in plain C) ------------------------------
 * Reference expression: modules/base.py:140 -> modules/linear.py / conv.py `_forward_func(q_input, q_weight)` with
 * y_a = (ca - z_a)*m_a + o_a and y_w = cw*m_w[n]; factored as alpha[n]*acc + beta[n] (include/dlmcq.h, dlmcq_qgemm):
 * exact integer dot product, then alpha[n] = m_a*m_w[n], beta[n] = ((o_a - z_a*m_a)*m_w[n])*float(sum_k cw) (+ bias),
 * out = float(acc)*alpha + beta - every fp32 rounding where the kernels round.  a_codes [m,k], w_codes [n,k] hold
 * integer-valued floats (as orc_fq_forward writes them); m_w has n or 1 entries. */
void orc_code_gemm(const float* a_codes, const float* w_codes, int64_t m, int64_t n, int64_t k, float m_a, float o_a,
                   float z_a, const float* m_w, int64_t m_w_count, const float* bias, int relu, float* out) {
  for (int64_t j = 0; j < n; ++j) {
    long long wsum = 0;
    for (int64_t t = 0; t < k; ++t) wsum += (long long)w_codes[j * k + t];
    const float mw = m_w[m_w_count == 1 ? 0 : j];
    const float alpha = m_a * mw;
    const float zm = z_a * m_a;
    const float tt = o_a - zm;
    const float tw = tt * mw;
    float beta = tw * (float)wsum;
    if (bias) beta = beta + bias[j];
    for (int64_t i = 0; i < m; ++i) {
      long long acc = 0;
      for (int64_t t = 0; t < k; ++t) acc += (long long)a_codes[i * k + t] * (long long)w_codes[j * k + t];
      const float prod = (float)acc * alpha;
      float o = prod + beta;
      if (relu) o = reluf(o);
      out[i * n + j] = o;
    }
  }
}
