"""TEST INFRASTRUCTURE ONLY - CPU restatement of DLMC-QUANT's fake-quant hot path.

This file is the *oracle* of the repo: a self-contained restatement, in plain
eager torch ops, of the arithmetic the reference performs in
`dlmc/quantization/scalar/{utils.py, ops.py, modules/base.py, RootQ/, FSPTQuant/}`.
It exists because `/root/reference` cannot travel to the GPU box.  Every function
cites the reference file:line it follows and keeps the reference's operation
ORDER (each torch op is one separately rounded IEEE fp32 op), because "bit-exact"
for this path means exactly that order.  Gradients come from autograd over the
same chain, which is how the reference itself obtains them.

Pinning: `oracle/make_golden.py` runs the unmodified reference (through
`oracle/ref_shim.py`) and this file on the same seeded inputs and stores the
reference's outputs in `tests/golden/`; `tests/test_oracle_golden.py` re-checks
this file against those fixtures wherever the tests run.  The reference has no
tests or golden vectors of its own (SURVEY.md section 4), so the fixtures minted
from its live code are the pin.

Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s cpu_baseline /
`--impl reference` legs may import this module.  The product package never does.
"""
import math

import torch
import torch.nn.functional as F

N_SWEEP = 80          # ops.py:52,177  `for i in range(80)`
SWEEP_MIN_LOSS = 1000  # ops.py:48,176


# --------------------------------------------------------------------------- #
# scalar/utils.py
# --------------------------------------------------------------------------- #
def qrange(signed, n_bits):
    """utils.py:14-22 - symmetric signed range (no -2^(n-1)), or [0, 2^n-1]."""
    if signed:
        hi = 2 ** (n_bits - 1) - 1
        return -hi, hi
    return 0, 2 ** n_bits - 1


def codes_a1(x, scale, offset, lo, hi):
    """utils.py:1-2 - round THEN clamp, +1e-7 on the divisor only."""
    return ((x - offset) / (scale + 1e-7)).round().clamp(lo, hi)


def dequant_a1(codes, scale, offset):
    """utils.py:5-6 - uses the scale WITHOUT the epsilon."""
    return codes * scale + offset


def emulate_a1(x, scale, offset, lo, hi):
    """utils.py:9-11."""
    return dequant_a1(codes_a1(x, scale, offset, lo, hi), scale, offset)


def grad_scale(s, g):
    """utils.py:24-27 - value (s - s*g) + s*g, gradient scaled by g."""
    sg = s * g
    return (s - sg).detach() + sg


def round_ste(v):
    """utils.py:29-32."""
    return (v.round() - v).detach() + v


def floor_ste(v):
    """utils.py:34-37."""
    return (v.floor() - v).detach() + v


def l2_loss(a, b):
    """trainer/loss/loss.py:22-24 - sum over axis 1, mean over the rest."""
    return ((a - b) ** 2).sum(axis=1).mean()


# --------------------------------------------------------------------------- #
# modules/base.py (QBase): A.2 "affine, float offset" form
# --------------------------------------------------------------------------- #
def lsq_g(numel, qmax):
    """modules/base.py:96,131 - python double."""
    return 1 / math.sqrt(numel * qmax)


def fq_affine(x, scale, offset, lo, hi, g):
    """modules/base.py:97,102 (activation) and :132-133 (weight).
    clamp THEN round, no epsilon, scale passed through grad_scale first."""
    s = grad_scale(scale, g)
    return round_ste(((x - offset) / s).clamp(lo, hi)) * s + offset


def fq_affine_codes(x, scale, offset, lo, hi, g):
    """The integer codes inside fq_affine (fp32-valued integers)."""
    s = grad_scale(scale, g)
    return round_ste(((x - offset) / s).clamp(lo, hi))


def fq_affine_fwd_bwd(x, scale, offset, lo, hi, g, dy):
    """Forward + autograd backward of fq_affine -> (y, dx, dscale)."""
    x = x.detach().clone().requires_grad_(True)
    scale = scale.detach().clone().requires_grad_(True)
    y = fq_affine(x, scale, offset, lo, hi, g)
    dx, ds = torch.autograd.grad(y, (x, scale), dy)
    return y.detach(), dx, ds


def bn_act_fq_chain(x, gamma, beta, running_mean, running_var, training, momentum, eps, identity, relu,
                    scale, offset, lo, hi, g):
    """The producer chain the fused kernels replace (SURVEY.md 8f-f2), as the reference runs it: the model's
    nn.BatchNorm2d -> `out += identity` -> nn.ReLU (e.g. model/classification/cifarresnet_large.py:24-46,
    torchvision Bottleneck.forward) followed by QBase.forward's input branch, modules/base.py:96-102.
    Returns (a, a_q); a_q is None when scale is None.  running_* are updated in place like nn.BatchNorm2d."""
    z = F.batch_norm(x, running_mean, running_var, gamma, beta, training, momentum, eps)
    if identity is not None:
        z = z + identity
    a = F.relu(z) if relu else z
    if scale is None:
        return a, None
    return a, fq_affine(a, scale, offset, lo, hi, g)


def fma_f32(a, b, c):
    """fp32 fma(a, b, c) rounded ONCE to nearest-even, as the fused kernels' __fmaf_rn / __ffma2_rn compute it
    (the fused BatchNorm's z = fma(x - mean, gamma * invstd, beta)), from float32 tensors of one shape.
    a * b is exact in float64 (24 + 24 significant bits); the float64 sum s = RN64(a*b + c) can differ from the exact
    sum, and rounding s to fp32 then gives a different result from rounding the exact sum in exactly one case: s lands
    on the midpoint of two fp32 neighbours while the exact sum does not.  TwoSum recovers the exact error e of s, and
    the sign of e says on which side of that midpoint the exact sum lies.  Non-finite sums are rounded as they are.
    One case is not corrected: a float64 sum exactly on the fp32 overflow threshold 2^128 - 2^103 with the exact sum
    below it returns inf where fmaf returns FLT_MAX (the midpoint there is computed as inf).  Callers stay far below."""
    p = a.double() * b.double()
    cd = c.double()
    s = p + cd
    bb = s - p
    e = (p - (s - bb)) + (cd - bb)                 # TwoSum: p + c == s + e exactly (finite s)
    r = s.float()
    rd = r.double()
    up = s > rd
    toward = torch.nextafter(r, torch.where(up, torch.full_like(r, math.inf), torch.full_like(r, -math.inf)))
    mid = (rd + toward.double()) * 0.5              # exact in float64
    fix = (s == mid) & ((e > 0) | (e < 0)) & ((e > 0) == up)     # e is NaN for a non-finite s
    return torch.where(fix, toward, r)


def lsq_init_scale(x, qmax):
    """modules/base.py:84,119 - LSQ initial scale 2*mean|x|/sqrt(qmax)."""
    return 2 * x.detach().abs().mean() / math.sqrt(qmax)


def fun_lsq_backward(w, scale, lo, hi, g, dy):
    """modules/function.py:38-47 - FunLSQ.backward restated (strict < / > masks,
    offset ignored) -> (dw, dscale[1])."""
    q = w / scale
    below = (q < lo).float()
    above = (q > hi).float()
    mid = torch.ones(w.shape, device=w.device) - below - above
    ds = ((lo * below + hi * above + mid * (-q + q.round())) * dy).sum().unsqueeze(dim=0) * g
    return mid * dy, ds


# --------------------------------------------------------------------------- #
# FSPTQuant/base.py: A.3 integer zero-point form, A.4 symmetric per-channel
# --------------------------------------------------------------------------- #
def fq_zp(x, scale, zp, lo, hi):
    """FSPTQuant/base.py:108-109 - round, add zp, clamp; no epsilon."""
    q = (round_ste(x / scale) + zp).clamp(lo, hi)
    return (q - zp) * scale


def fq_zp_codes(x, scale, zp, lo, hi):
    return (round_ste(x / scale) + zp).clamp(lo, hi)


def fq_zp_fwd_bwd(x, scale, zp, lo, hi, dy):
    x = x.detach().clone().requires_grad_(True)
    scale = scale.detach().clone().requires_grad_(True)
    y = fq_zp(x, scale, zp, lo, hi)
    dx, ds = torch.autograd.grad(y, (x, scale), dy)
    return y.detach(), dx, ds


def fq_sym(w, scale, lo, hi):
    """FSPTQuant/base.py:149-152 - symmetric per-channel weight fake-quant."""
    return round_ste(w / scale).clamp(lo, hi) * scale


def fq_sym_codes(w, scale, lo, hi):
    return round_ste(w / scale).clamp(lo, hi)


def fq_sym_fwd_bwd(w, scale, lo, hi, dy):
    w = w.detach().clone().requires_grad_(True)
    scale = scale.detach().clone().requires_grad_(True)
    y = fq_sym(w, scale, lo, hi)
    dw, ds = torch.autograd.grad(y, (w, scale), dy)
    return y.detach(), dw, ds


# --------------------------------------------------------------------------- #
# the layer product on the two fake-quantised tensors (consumer side of row f2)
# --------------------------------------------------------------------------- #
def layer_product_reference(q_input, q_weight, bias=None, dtype=torch.float64):
    """modules/linear.py / conv.py `_forward_func(q_input, q_weight)` for a Linear / 1x1 convolution, written as the
    matrix product it is: q_input [m, k] (fake-quantised activations), q_weight [n, k].  Evaluated in `dtype`
    (float64 = the exact value of the reference expression up to 1e-16; float32 = what the reference's library call
    computes up to its own summation order)."""
    y = q_input.to(dtype) @ q_weight.to(dtype).t()
    return y if bias is None else y + bias.to(dtype)


def code_gemm(a_codes, w_codes, m_a, o_a, z_a, m_w, bias=None, relu=False):
    """The factored form of the same product that dlmcq_qgemm evaluates (include/dlmcq.h), every fp32 rounding where
    the kernels round:  acc = exact integer dot product;  alpha[n] = m_a*m_w[n];
    beta[n] = ((o_a - z_a*m_a) * m_w[n]) * float(sum_k cw[n,k]) (+ bias[n]);  out = (float(acc) * alpha) + beta.
    a_codes [m,k], w_codes [n,k]: integer-valued tensors; m_a, o_a, z_a: fp32 scalars; m_w: fp32 [n] or [1]."""
    f32 = torch.float32
    ca, cw = a_codes.to(torch.int64), w_codes.to(torch.int64)
    acc = ca @ cw.t()
    wsum = cw.sum(dim=1)
    m_a, o_a, z_a = (torch.as_tensor(v, dtype=f32).reshape(()) for v in (m_a, o_a, z_a))
    m_w = torch.as_tensor(m_w, dtype=f32).reshape(-1).expand(cw.shape[0])
    alpha = m_a * m_w
    t = o_a - z_a * m_a
    beta = (t * m_w) * wsum.to(f32)
    if bias is not None:
        beta = beta + bias.to(f32)
    out = acc.to(f32) * alpha + beta
    return torch.relu(out) if relu else out


ADAROUND_GAMMA, ADAROUND_ZETA = -0.1, 1.1   # FSPTQuant/base.py:62


def adaround_soft_targets(alpha):
    """FSPTQuant/base.py:78-79."""
    return torch.clamp(torch.sigmoid(alpha) * (ADAROUND_ZETA - ADAROUND_GAMMA) + ADAROUND_GAMMA, 0, 1)


def adaround_init_alpha(w, scale):
    """FSPTQuant/base.py:73-76."""
    w_floor = torch.floor(w.detach() / scale)
    rest = w.detach() / scale - w_floor
    return -torch.log((ADAROUND_ZETA - ADAROUND_GAMMA) / (rest - ADAROUND_GAMMA) - 1)


def fq_adaround(w, scale, alpha, lo, hi, training):
    """FSPTQuant/base.py:136-141,151-152 - floor has NO straight-through here."""
    q = torch.floor(w / scale)
    if training:
        q = q + adaround_soft_targets(alpha)
    else:
        q = q + (alpha >= 0).float()
    return q.clamp(lo, hi) * scale


def fq_adaround_fwd_bwd(w, scale, alpha, lo, hi, dy):
    w = w.detach().clone().requires_grad_(True)
    scale = scale.detach().clone().requires_grad_(True)
    alpha = alpha.detach().clone().requires_grad_(True)
    y = fq_adaround(w, scale, alpha, lo, hi, True)
    ds, da = torch.autograd.grad(y, (scale, alpha), dy)
    return y.detach(), ds, da


# --------------------------------------------------------------------------- #
# RootQ/function.py + RootQ/base.py: A.5
# --------------------------------------------------------------------------- #
def rootq_clipping(x, upper, lower):
    """RootQ/function.py:15-20 - relu trick, NOT clamp (loses low bits, inf->nan)."""
    x = x + F.relu(lower - x)
    x = x - F.relu(x - upper)
    return x


def rootq_phi(x, mi, alpha, delta):
    """RootQ/function.py:22-32 - root-function estimator."""
    alpha = alpha + F.relu(1e-4 - alpha)
    alpha = alpha - F.relu(alpha - 1)
    x = x - mi
    sg = x / (torch.abs(x) + 1e-5)
    k = 2 / delta
    return torch.pow(k * abs(x) + 1e-5, alpha) * sg


class _SignSTE(torch.autograd.Function):
    """RootQ/function.py:5-12 - value sgn(x), gradient identity."""

    @staticmethod
    def forward(ctx, x):
        return x.sgn()

    @staticmethod
    def backward(ctx, g):
        return g


def rootq_dequant(sig, lower, delta, interval):
    """RootQ/function.py:63-67."""
    return ((sig + 1) / 2 + interval) * delta + lower


def rootq_act_init(x, lo, hi):
    """RootQ/base.py:80 - first-call activation scale."""
    return (torch.max(x) - torch.min(x)) / (hi - lo)


def rootq_wt_init(w, hi):
    """RootQ/base.py:115-116 - first-call weight bounds (upper, lower)."""
    up = 2 * w.detach().abs().mean() * math.sqrt(hi)
    dn = -2 * w.detach().abs().mean() * math.sqrt(hi)
    return up, dn


def rootq_act(x, in_scale, run_scale, momentum, lo, hi, training):
    """RootQ/base.py:92-111 -> (y, new_run_scale).  `run_scale` is not modified."""
    if training:
        g = 1 / math.sqrt(x.numel() * hi)
        rs = run_scale.mul(1 - momentum).add(momentum * in_scale)
        rs = g * rs + (1 - g) * rs.detach()
        upper = rs * (hi - lo)
        new_run = rs.data.detach().clone()
    else:
        rs = run_scale
        upper = rs * (hi - lo)
        new_run = run_scale.detach().clone()
    xq = rootq_clipping(x, upper, 0)
    interval = round_ste(xq / rs)
    return interval * rs, new_run


def rootq_act_fwd_bwd(x, in_scale, run_scale, momentum, lo, hi, dy):
    x = x.detach().clone().requires_grad_(True)
    in_scale = in_scale.detach().clone().requires_grad_(True)
    y, new_run = rootq_act(x, in_scale, run_scale, momentum, lo, hi, True)
    dx, ds = torch.autograd.grad(y, (x, in_scale), dy)
    return y.detach(), new_run, dx, ds


def rootq_wt(w, upper, lower, alpha, run_upper, run_lower, momentum, lo, hi, training):
    """RootQ/base.py:131-155 -> (w_q, new_run_upper, new_run_lower)."""
    if training:
        g = 1 / math.sqrt(w.numel() * hi)
        ru = run_upper.mul(1 - momentum).add(momentum * upper)
        rl = run_lower.mul(1 - momentum).add(momentum * lower)
        ru = g * ru + (1 - g) * ru.detach()
        rl = g * rl + (1 - g) * rl.detach()
        new_ru, new_rl = ru.data.clone(), rl.data.clone()
    else:
        ru, rl = run_upper, run_lower
        new_ru, new_rl = run_upper.detach().clone(), run_lower.detach().clone()
    c = rootq_clipping(w, ru, rl)
    delta = (ru - rl) / (hi - lo)
    interval = floor_ste((c - rl) / delta)
    mi = (interval + 0.5) * delta + rl
    p = rootq_phi(c, mi.detach(), alpha, delta)
    sig = _SignSTE.apply(p)
    return rootq_dequant(sig, rl, delta, interval), new_ru, new_rl


def rootq_wt_fwd_bwd(w, upper, lower, alpha, run_upper, run_lower, momentum, lo, hi, dy):
    w = w.detach().clone().requires_grad_(True)
    upper = upper.detach().clone().requires_grad_(True)
    lower = lower.detach().clone().requires_grad_(True)
    alpha = alpha.detach().clone().requires_grad_(True)
    y, nru, nrl = rootq_wt(w, upper, lower, alpha, run_upper, run_lower, momentum, lo, hi, True)
    dw, du, dl, da = torch.autograd.grad(y, (w, upper, lower, alpha), dy)
    return y.detach(), nru, nrl, dw, du, dl, da


# --------------------------------------------------------------------------- #
# scalar/ops.py: observers
# --------------------------------------------------------------------------- #
def _rows(t, ch_axis):
    """ops.py:112-118 - channel-major 2-D view and the broadcast shape."""
    shape = [1] * t.dim()
    shape[ch_axis] = -1
    return t.transpose(0, ch_axis).reshape(t.shape[ch_axis], -1), shape


def obs_minmax_tensor(t, n_bits, signed, allow_offset=True):
    """ops.py:20-34."""
    if signed:
        return t.abs().max() / ((2 ** (n_bits - 1)) - 1), torch.tensor(0)
    lo = t.min()
    if not allow_offset:
        assert (lo >= 0).all()
        lo = torch.tensor(0)
    return (t.max() - lo) / ((2 ** n_bits) - 1), lo


def obs_minmax_channel(t, n_bits, signed, ch_axis=0, allow_offset=True):
    """ops.py:121-140."""
    rows, shape = _rows(t, ch_axis)
    if signed:
        scale = rows.abs().max(dim=1)[0] / ((2 ** (n_bits - 1)) - 1)
        offset = torch.zeros_like(scale)
    else:
        lo = rows.min(dim=1)[0]
        if not allow_offset:
            assert (lo >= 0).all()
            lo[:] = 0.
        scale = (rows.max(dim=1)[0] - lo) / ((2 ** n_bits) - 1)
        offset = lo
    return scale.reshape(shape), offset.reshape(shape)


def obs_minmax_pixel(t, n_bits, signed, allow_offset=True):
    """ops.py:142-167 - reduce over (Cout, Cin) per kernel position; the unsigned
    branch takes abs() before min/max (reference quirk A.7-10, reproduced)."""
    shape = [t.shape[2], t.shape[3]] if t.dim() == 4 else [t.shape[2]]
    t3 = t.reshape([t.shape[0], t.shape[1], -1])
    if signed:
        amax = t3.abs().max(dim=0)[0].max(dim=0)[0]
        scale = amax / ((2 ** (n_bits - 1)) - 1)
        offset = torch.zeros_like(scale)
    else:
        lo = t3.abs().min(dim=0)[0].min(dim=0)[0]
        hi = t3.abs().max(dim=0)[0].max(dim=0)[0]
        if not allow_offset:
            assert (lo >= 0).all()
            lo[:] = 0.
        scale = (hi - lo) / ((2 ** n_bits) - 1)
        offset = lo
    return scale.reshape(shape), offset.reshape(shape)


def obs_l2loss_tensor(t, n_bits, signed, allow_offset=True, return_index=False):
    """ops.py:36-68 - 80-point clip-ratio MSE sweep, per tensor.  Signed inputs take
    the min/max answer (:37-40).  First strict minimum below 1000 wins (:48,62)."""
    if signed:
        out = t.abs().max() / ((2 ** (n_bits - 1)) - 1), torch.tensor(0)
        return out + (-1,) if return_index else out
    lo = t.min()
    if not allow_offset:
        assert (lo >= 0).all()
        lo = torch.tensor(0)
    hi = t.max()
    qmax = (2 ** n_bits) - 1
    best = SWEEP_MIN_LOSS
    scale, offset, pick = hi / qmax, torch.tensor(0), -1
    for i in range(N_SWEEP):
        r = 1 - 0.01 * i
        c_hi, c_lo = r * hi, r * lo
        c_scale = (c_hi - c_lo) / qmax
        c_zp = torch.round(-c_lo / c_scale)
        q = torch.round(t / c_scale) + c_zp
        q = (q.clamp(0, qmax) - c_zp) * c_scale
        loss = l2_loss(q, t)
        if loss < best:
            pick, best, scale, offset = i, loss, c_scale, c_zp
    return (scale, offset, pick) if return_index else (scale, offset)


def obs_l2loss_channel(t, n_bits, signed, ch_axis=0):
    """ops.py:169-196 - per-channel sweep.  Reproduces two reference defects on
    purpose (SURVEY.md A.7-1/2): `signed` is ignored by the search (always clamps
    to [0, 2^n-1]) and the running minimum ALIASES the offset vector, so accepting
    a candidate rewrites the minimum used by the following candidates."""
    rows, shape = _rows(t, ch_axis)
    scale, offset = obs_minmax_channel(rows, n_bits, signed, ch_axis=0, allow_offset=True)
    qmax = (2 ** n_bits) - 1
    lo = offset                      # alias, as at ops.py:172
    hi = offset + scale * qmax       # fresh tensor
    for c in range(rows.shape[0]):
        best = SWEEP_MIN_LOSS
        for i in range(N_SWEEP):
            r = 1 - 0.01 * i
            c_lo, c_hi = r * lo[c], r * hi[c]
            c_scale = (c_hi - c_lo) / qmax
            c_zp = torch.round(-c_lo / c_scale)
            q = torch.round(rows[c] / c_scale)
            q = (q + c_zp).clamp(0, qmax)
            q = (q - c_zp) * c_scale
            loss = l2_loss(rows[c].view(1, -1), q.view(1, -1))
            if best > loss:
                scale[c] = c_scale
                offset[c] = c_zp     # also rewrites lo[c]
                best = loss
    return scale.reshape(shape), offset.reshape(shape)


def obs_l2norm_tensor(t, n_bits, signed, return_iters=False):
    """ops.py:71-83 - fixed point s <- sum(x q)/sum(q q + 1e-7) from the min/max start."""
    scale, offset = obs_minmax_tensor(t, n_bits, signed, allow_offset=True)
    lo, hi = qrange(signed, n_bits)
    diff, iters = float('inf'), 0
    while diff > 1e-5:
        q = codes_a1(t, scale, offset, lo, hi)
        new = (t * q).sum() / (q * q + 1e-7).sum()
        diff = (new - scale).abs() / scale
        scale = new
        iters += 1
    return (scale, offset, iters) if return_iters else (scale, offset)


def obs_l2norm_channel(t, n_bits, signed, ch_axis=0, return_iters=False):
    """ops.py:198-215 - per-channel fixed point, global L2 stopping rule."""
    rows, shape = _rows(t, ch_axis)
    scale, offset = obs_minmax_channel(rows, n_bits, signed, ch_axis=0, allow_offset=True)
    lo, hi = qrange(signed, n_bits)
    diff, iters = float('inf'), 0
    while diff > 1e-5:
        q = codes_a1(rows, scale, offset, lo, hi)
        new = ((rows * q).sum(axis=1) / (q * q + 1e-7).sum(axis=1)).reshape(scale.shape)
        diff = ((new - scale) ** 2).sum().sqrt() / (scale ** 2).sum().sqrt()
        scale = new
        iters += 1
    out = scale.reshape(shape), offset.reshape(shape)
    return out + (iters,) if return_iters else out


def obs_percentile_tensor(t, n_bits, signed, percentile=99.99, allow_offset=True):
    """EXTENSION without a reference counterpart (the north star names a percentile observer; ops.py has none):
    exact order statistics via torch.kthvalue, then the min/max formulas of ops.py:20-34.  Parity for this one
    observer is pinned to torch.kthvalue, not to the reference."""
    flat = t.detach().float().flatten()
    n = flat.numel()
    k_hi = min(n, max(1, math.ceil(percentile / 100.0 * n)))
    k_lo = n + 1 - k_hi
    if signed:
        a = flat.abs().kthvalue(k_hi)[0]
        return a / (2 ** (n_bits - 1) - 1), torch.tensor(0)
    hi = flat.kthvalue(k_hi)[0]
    lo = flat.kthvalue(k_lo)[0] if allow_offset else torch.zeros(())
    return (hi - lo) / (2 ** n_bits - 1), lo


OBSERVERS = {
    "minmax_tensor": obs_minmax_tensor,
    "minmax_channel": obs_minmax_channel,
    "minmax_pixel": obs_minmax_pixel,
    "l2loss_tensor": obs_l2loss_tensor,
    "l2loss_channel": obs_l2loss_channel,
    "l2norm_tensor": obs_l2norm_tensor,
    "l2norm_channel": obs_l2norm_channel,
}


# --------------------------------------------------------------------------- #
# weight-space re-parameterisation (SURVEY.md 8f, row f3)
# --------------------------------------------------------------------------- #
def sqrt_ieee(t):
    """Correctly rounded fp32 square root (the hardware instruction, via numpy) - what `Tensor.sqrt()`
    computes on CUDA.  torch's CPU `sqrt` goes through MKL VML, which is only faithfully rounded: e.g.
    sqrt(0x1.17783ep+0) returns 0x1.0b7a40p+0 there, the correctly rounded value is 0x1.0b7a42p+0 [probed,
    torch 2.11.0 + MKL 2024.2].  About 3 % of random inputs differ by that one ulp, so a reference run on
    the CPU can differ from its own CUDA run (and from this oracle) by 1 ulp of std in those channels."""
    import numpy as np
    return torch.from_numpy(np.sqrt(t.detach().cpu().numpy()))


def merge_bn_fold(w, bias, gamma, beta, mean, running_var):
    """dlmc/utils/merge_bn.py:84-100 - fold a BatchNorm2d into the preceding Conv2d.
    var = running_var + 1e-7 (NOT the module's eps); a missing conv bias is zeros (:92-94)."""
    var = running_var + 1e-7
    cout = w.shape[0]
    if bias is None:
        bias = torch.zeros(cout)
    new_bias = gamma * (bias - mean) / sqrt_ieee(var) + beta
    new_w = (w.reshape(cout, -1) * gamma.reshape(-1, 1) / sqrt_ieee(var).reshape(-1, 1)).reshape(w.shape)
    return new_w, new_bias


def _repvgg_branch(kernel, gamma, beta, mean, var, eps):
    """model/classification/repvgg.py:121-123."""
    std = sqrt_ieee(var + eps)
    t = (gamma / std).reshape(-1, 1, 1, 1)
    return kernel * t, beta - mean * gamma / std


def repvgg_fuse(k3, bn3, k1, bn1, bn_id, groups=1):
    """repvgg.py:92-123 get_equivalent_kernel_bias.  bn* = (gamma, beta, running_mean, running_var, eps);
    bn_id is None when the block has no identity branch (the reference then adds the integer 0)."""
    kernel3, bias3 = _repvgg_branch(k3, *bn3)
    kernel1, bias1 = _repvgg_branch(k1, *bn1)
    if bn_id is None:
        kernel_id, bias_id = 0, 0
    else:
        in_channels = k3.shape[1] * groups
        input_dim = in_channels // groups                              # repvgg.py:108
        id_tensor = torch.zeros(in_channels, input_dim, 3, 3)
        for i in range(in_channels):
            id_tensor[i, i % input_dim, 1, 1] = 1                      # :110-111
        kernel_id, bias_id = _repvgg_branch(id_tensor, *bn_id)
    return kernel3 + F.pad(kernel1, [1, 1, 1, 1]) + kernel_id, bias3 + bias1 + bias_id


def get_qparams_tensor(t, qtype, **kwargs):
    """ops.py:15-18 - name dispatch."""
    return OBSERVERS[qtype](t, **kwargs)
