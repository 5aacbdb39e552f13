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
    f64 = torch.float64
    ca, cw = a_codes.to(f64), w_codes.to(f64)
    kw_ = dict(stride=stride, padding=padding, dilation=dilation)
    acc = F.conv2d(ca, cw, **kw_)
    if whole_k_beta:
        wsum = cw.sum(dim=(1, 2, 3)).reshape(1, -1, 1, 1).expand_as(acc)
    else:
        ones = torch.ones(1, 1, *ca.shape[2:], dtype=f64)
        wsum = F.conv2d(ones, _tap_weight_sums(cw), **kw_)                   # [1, n, Ho, Wo]: valid taps only
    return conv_epilogue(acc, wsum, m_a, o_a, z_a, m_w, bias, relu)


def conv_epilogue(acc, wsum, m_a, o_a, z_a, m_w, bias=None, relu=False):
    """The kernels' two fp32 roundings on an exact integer convolution acc [B, n, Ho, Wo] and the per-pixel sum of
    the weight codes over the taps inside the image wsum [1, n, Ho, Wo] (both float64, on any device)."""
    f32 = torch.float32
    dev = acc.device
    m_a, o_a, z_a = (torch.as_tensor(v, dtype=f32).to(dev).reshape(()) for v in (m_a, o_a, z_a))
    n = acc.shape[1]
    m_w = torch.as_tensor(m_w, dtype=f32).to(dev).reshape(-1).expand(n).reshape(1, n, 1, 1)
    alpha = m_a * m_w
    t = o_a - z_a * m_a
    beta = (t * m_w) * wsum.to(f32)
    if bias is not None:
        beta = beta + bias.to(device=dev, dtype=f32).reshape(1, n, 1, 1)
    out = acc.to(f32) * alpha + beta
    return torch.relu(out) if relu else out


def conv_pairs(stride, padding, dilation):
    """(stride_h, stride_w), (pad_h, pad_w), (dil_h, dil_w) of an int-or-pair geometry."""
    return tuple((v, v) if isinstance(v, int) else tuple(v) for v in (stride, padding, dilation))


def _out_size(size, k, s, p, d):
    return (size + 2 * p - d * (k - 1) - 1) // s + 1


def exact_conv_acc(a_codes, w_codes, stride=1, padding=0, dilation=1):
    """The integer convolution of a_codes [B, Cin, H, W] with w_codes [n, Cin, kh, kw] (integer-valued, any memory
    format) as one float64 matmul per filter tap over a zero-padded, strided view of the channels-last codes, on the
    codes' device.  Every product and partial sum is an integer below 2^53, so the sum is exact in any order (no
    library convolution: its algorithm choice is not ours).  Returns float64 [B, n, Ho, Wo] (channels-last storage)."""
    (sh, sw), (ph, pw), (dh, dw) = conv_pairs(stride, padding, dilation)
    b, cin, h, w = a_codes.shape
    n, _, kh, kw = w_codes.shape
    ho, wo = _out_size(h, kh, sh, ph, dh), _out_size(w, kw, sw, pw, dw)
    f64 = torch.float64
    x = torch.zeros(b, h + 2 * ph, w + 2 * pw, cin, dtype=f64, device=a_codes.device)
    x[:, ph:ph + h, pw:pw + w] = a_codes.permute(0, 2, 3, 1).to(f64)
    wt = w_codes.to(device=a_codes.device, dtype=f64).permute(2, 3, 1, 0)          # [kh, kw, Cin, n]
    acc = torch.zeros(b * ho * wo, n, dtype=f64, device=a_codes.device)
    for r in range(kh):
        for s in range(kw):
            tap = x[:, r * dh:r * dh + (ho - 1) * sh + 1:sh, s * dw:s * dw + (wo - 1) * sw + 1:sw]
            acc.addmm_(tap.reshape(-1, cin), wt[r, s])
    return acc.view(b, ho, wo, n).permute(0, 3, 1, 2)


def valid_tap_wsum(w_codes, h, w, stride=1, padding=0, dilation=1):
    """[1, n, Ho, Wo] float64: per output pixel, the sum of the weight codes over the filter taps inside the image
    (the border rule of beta), on w_codes' device."""
    (sh, sw), (ph, pw), (dh, dw) = conv_pairs(stride, padding, dilation)
    n, _, kh, kw = w_codes.shape
    ho, wo = _out_size(h, kh, sh, ph, dh), _out_size(w, kw, sw, pw, dw)
    dev, f64 = w_codes.device, torch.float64

    def valid(k, o, s, p, d, size):                                     # [k, o]: tap inside the image
        pos = (torch.arange(o, device=dev) * s - p).reshape(1, -1) + (torch.arange(k, device=dev) * d).reshape(-1, 1)
        return ((pos >= 0) & (pos < size)).to(f64)
    taps = w_codes.to(f64).sum(dim=1)                                   # [n, kh, kw]
    return torch.einsum("rh,sw,nrs->nhw", valid(kh, ho, sh, ph, dh, h), valid(kw, wo, sw, pw, dw, w), taps)[None]


def exact_conv(a_codes, w_codes, m_a, o_a, z_a, m_w, bias=None, stride=1, padding=0, dilation=1, relu=False):
    """code_conv's result from exact_conv_acc and valid_tap_wsum: the same value, on the codes' device."""
    kw_ = dict(stride=stride, padding=padding, dilation=dilation)
    acc = exact_conv_acc(a_codes, w_codes, **kw_)
    wsum = valid_tap_wsum(w_codes.to(acc.device), a_codes.shape[2], a_codes.shape[3], **kw_)
    return conv_epilogue(acc, wsum, m_a, o_a, z_a, m_w, bias, relu)


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
    # per-axis strides / dilations / paddings: an h <-> w swap anywhere in the kernel's geometry shows here
    "3x3_stride_1x2": (3, 3, (1, 2), 1, 1, 9, 13),
    "3x3_stride_2x1": (3, 3, (2, 1), 1, 1, 13, 9),
    "3x3_stride_3x1": (3, 3, (3, 1), 1, 1, 14, 8),
    "3x3_dil_2x1": (3, 3, 1, 0, (2, 1), 11, 9),
    "3x3_dil_2x1_pad_2x1": (3, 3, 1, (2, 1), (2, 1), 10, 9),
    "3x3_stride4": (3, 3, 4, 1, 1, 17, 15),
    "3x3_stride8": (3, 3, 8, 1, 1, 30, 27),
    # windows clipped on both sides of an axis: the image is smaller than the filter's span
    "3x3_pad1_1x1_image": (3, 3, 1, 1, 1, 1, 1),
    "3x3_pad1_1xW_image": (3, 3, 1, 1, 1, 1, 9),
    "5x5_pad2_2x3_image": (5, 5, 1, 2, 1, 2, 3),
    "3x3_dil3_pad3_2x2_image": (3, 3, 1, 3, 3, 2, 2),       # the middle tap of a window can be the only one inside
    # the im2col bounding-box corner extremes: -pad = pad - dil*(k-1) = -128 (tap offset 256); pad - dil*(k-1) = 127
    "3x1_dil128_pad128_corner": (3, 1, 1, (128, 0), (128, 1), 3, 4),
    "1x1_pad127_stride8_corner": (1, 1, 8, 127, 1, 3, 5),
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
