"""The convolution on the integer codes written out in float64 / fp32 torch ops (test infrastructure for
dlmcq_qconv, include/dlmcq.h).

`code_conv` is the factored form the kernels evaluate, with their two fp32 roundings: the exact integer convolution
of the codes (a float64 conv2d of integers, exact below 2^53) and the border rule for beta - the reference pads the
FAKE-QUANTISED tensor with real zeros (scalar/_layers.py `_conv_forward` -> F.conv2d(..., padding)), so a padded tap
contributes neither to the integer sum nor to the offset term.  `conv_reference` is the reference expression itself:
F.conv2d of the two dequantised tensors in float64."""
import torch
import torch.nn.functional as F


def _tap_weight_sums(cw):
    """[n, 1, kh, kw]: sum over input channels of the weight codes per filter tap."""
    return cw.sum(dim=1, keepdim=True)


def code_conv(a_codes, w_codes, m_a, o_a, z_a, m_w, bias=None, stride=1, padding=0, dilation=1, relu=False,
              whole_k_beta=False):
    """a_codes [B, Cin, H, W], w_codes [n, Cin, kh, kw]: integer-valued tensors; m_a, o_a, z_a fp32 scalars; m_w fp32
    [n] or [1].  Returns [B, n, Ho, Wo] fp32:
        out = RN(RN(float(acc) * alpha[n]) + beta),  acc = sum over the taps inside the image (exact)
        beta = RN(RN(t * m_w[n]) * float(sum of cw over the taps inside the image)) (+ bias[n]),  t = o_a - z_a*m_a.
    whole_k_beta=True uses sum_k cw for every pixel (the 1x1 rule; wrong at borders when t != 0)."""
    f32, f64 = torch.float32, torch.float64
    ca, cw = a_codes.to(f64), w_codes.to(f64)
    kw_ = dict(stride=stride, padding=padding, dilation=dilation)
    acc = F.conv2d(ca, cw, **kw_)
    if whole_k_beta:
        wsum = cw.sum(dim=(1, 2, 3)).reshape(1, -1, 1, 1).expand_as(acc)
    else:
        ones = torch.ones(1, 1, *ca.shape[2:], dtype=f64)
        wsum = F.conv2d(ones, _tap_weight_sums(cw), **kw_)                   # [1, n, Ho, Wo]: valid taps only
    m_a, o_a, z_a = (torch.as_tensor(v, dtype=f32).reshape(()) for v in (m_a, o_a, z_a))
    n = cw.shape[0]
    m_w = torch.as_tensor(m_w, dtype=f32).reshape(-1).expand(n).reshape(1, n, 1, 1)
    alpha = m_a * m_w
    t = o_a - z_a * m_a
    beta = (t * m_w) * wsum.to(f32)
    if bias is not None:
        beta = beta + bias.to(f32).reshape(1, n, 1, 1)
    out = acc.to(f32) * alpha + beta
    return torch.relu(out) if relu else out


def conv_reference(q_input, q_weight, bias=None, stride=1, padding=0, dilation=1):
    """modules/conv.py `_forward_func(q_input, q_weight)`: F.conv2d of the two fake-quantised tensors, float64; and
    the magnitude conv2d(|y_a|, |y_w|) (+ |bias|) the relative tolerance is measured against."""
    qa, qw = q_input.double(), q_weight.double()
    kw_ = dict(stride=stride, padding=padding, dilation=dilation)
    ref = F.conv2d(qa, qw, None if bias is None else bias.double(), **kw_)
    mag = F.conv2d(qa.abs(), qw.abs(), None if bias is None else bias.double().abs(), **kw_)
    return ref, mag


A1, AFFINE, ZP, SYM = 0, 1, 2, 3

# (kh, kw, stride, padding, dilation, H, W) - every geometry the oracle and the kernel tests cover
GEOMETRIES = {
    "3x3_pad1": (3, 3, 1, 1, 1, 10, 9),
    "3x3_pad1_stride2": (3, 3, 2, 1, 1, 11, 10),
    "1x1_stride2": (1, 1, 2, 0, 1, 9, 8),
    "5x5_pad2": (5, 5, 1, 2, 1, 9, 11),
    "3x3_dilation2": (3, 3, 1, 2, 2, 10, 9),
    "1x3": (1, 3, 1, (0, 1), 1, 7, 8),
    "3x1": (3, 1, 1, (1, 0), 1, 8, 7),
    "3x3_pad0": (3, 3, 1, 0, 1, 9, 10),
    "3x3_odd_hw": (3, 3, 1, 1, 1, 7, 5),
    "7x7_image_3x3_stride2": (3, 3, 2, 1, 1, 7, 7),
    "3x3_pad_eq_dil_k": (3, 3, 1, 4, 2, 8, 9),              # padding = d*(k-1): upper corner 0
}


def conv_problem(a_form, w_form, geom, batch=2, cin=8, n=6, n_bits=4, a_signed=False, per_channel=True, bias=True,
                 seed=0):
    """Random activation / weight, their fake-quantised tensors (oracle/restate.py chain) and codes.
    Returns dict(x, w, qa, qw, ca, cw, m_a, o_a, z_a, m_w, s_a, off, s_w, g_a, g_w, ranges, bias, conv kwargs)."""
    from oracle import restate as R
    kh, kw, stride, padding, dilation, h, w_ = geom
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(batch, cin, h, w_, generator=g)
    if not a_signed:
        x = torch.relu(x) + 0.1 + 0.05 * torch.rand(batch, cin, h, w_, generator=g)
    w = torch.randn(n, cin, kh, kw, generator=g) * 0.05
    a_lo, a_hi = R.qrange(a_signed, n_bits)
    w_lo, w_hi = R.qrange(True, n_bits)
    s_a = (x.abs().max() / a_hi * 0.9).reshape(1)
    off = {ZP: torch.tensor([3.0 if not a_signed else 0.0]), A1: torch.tensor([0.07]),
           AFFINE: torch.tensor([0.11 if not a_signed else -0.02]), SYM: torch.zeros(1)}[a_form]
    s_w = (w.abs().amax(dim=(1, 2, 3)) / w_hi + 1e-6) if per_channel else (w.abs().max() / w_hi).reshape(1)
    s_w4 = s_w.reshape(-1, 1, 1, 1) if per_channel else s_w
    g_a = R.lsq_g(x.numel(), a_hi) if a_form == AFFINE else 0.0
    g_w = R.lsq_g(w.numel(), w_hi) if w_form == AFFINE else 0.0
    if a_form == AFFINE:
        qa, ca, m_a = R.fq_affine(x, s_a, off, a_lo, a_hi, g_a), R.fq_affine_codes(x, s_a, off, a_lo, a_hi, g_a), R.grad_scale(s_a, g_a)
    elif a_form == ZP:
        qa, ca, m_a = R.fq_zp(x, s_a, off, a_lo, a_hi), R.fq_zp_codes(x, s_a, off, a_lo, a_hi), s_a
    elif a_form == A1:
        qa, ca, m_a = R.emulate_a1(x, s_a, off, a_lo, a_hi), R.codes_a1(x, s_a, off, a_lo, a_hi), s_a
    else:
        qa, ca, m_a = R.fq_sym(x, s_a, a_lo, a_hi), R.fq_sym_codes(x, s_a, a_lo, a_hi), s_a
    if w_form == AFFINE:
        z = torch.zeros(1)
        qw, cw, m_w = (R.fq_affine(w, s_w4, z, w_lo, w_hi, g_w), R.fq_affine_codes(w, s_w4, z, w_lo, w_hi, g_w),
                       R.grad_scale(s_w, g_w))
    else:
        qw, cw, m_w = R.fq_sym(w, s_w4, w_lo, w_hi), R.fq_sym_codes(w, s_w4, w_lo, w_hi), s_w
    return dict(x=x, w=w, qa=qa.detach(), qw=qw.detach(), ca=ca.detach(), cw=cw.detach(), m_a=m_a.detach(),
                o_a=off if a_form in (A1, AFFINE) else torch.zeros(1), z_a=off if a_form == ZP else torch.zeros(1),
                m_w=m_w.detach().reshape(-1), s_a=s_a, off=None if a_form == SYM else off, s_w=s_w, g_a=g_a, g_w=g_w,
                a_range=(a_lo, a_hi), w_range=(w_lo, w_hi), a_form=a_form, w_form=w_form,
                bias=torch.randn(n, generator=g) if bias else None,
                conv=dict(stride=stride, padding=padding, dilation=dilation))
