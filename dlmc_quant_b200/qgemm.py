"""The layer's matrix product on the integer codes (SURVEY.md section 8f row f2, consumer side).

Reference: `_forward_func(q_input, q_weight)` - F.linear / F.conv2d on the two FAKE-QUANTISED fp32 tensors
(dlmc/quantization/scalar/modules/linear.py, modules/conv.py, entered from modules/base.py:140 and
FSPTQuant/base.py:111-113).  For a per-tensor activation quantizer and a per-output-channel (or per-tensor) weight
quantizer without an additive weight term that product factors into an exact integer dot product of the codes and a
per-output-channel affine map (include/dlmcq.h, `dlmcq_qgemm`).  The integer product runs on the tcgen05 tensor cores
(csrc/qgemm_kernels.cu); the activation is read at one byte per element instead of four.

Two levels:
  * functional: `codes_forward`, `qgemm_prepare`, `qgemm`, and for k x k / strided / padded convolutions
    `qconv_prepare`, `qconv` (implicit GEMM over channels-last codes) - thin wrappers over the C ABI;
  * module: `enable_code_gemm(model)` switches every eligible quantised `nn.Linear` / 1x1 `nn.Conv2d` of a model to
    the code path for inference (`module.eval()`, no autograd), `enable_code_gemm(model, convolutions=True)` also the
    other quantised `nn.Conv2d` layers `qconv` serves; training / calibration / ineligible layers keep the
    reference's path (fake-quant kernels + the library convolution).  Opt-in: results equal the fake-quant path up
    to the rounding of the fp32 product (the integer accumulation itself is exact; cuDNN's TF32 / fp32 sums are not).
"""
import ctypes as C
import math
import types

import torch
from torch import nn

from . import _lib
from . import functional as F
from ._lib import BF16, F32, FORM_AFFINE, FORM_SYM, FORM_ZP, QGEMM_E4M3, QGEMM_I8, BnqTail, ConvGeom, DlmcqError, QParams

__all__ = ["codes_forward", "qgemm_prepare", "qgemm", "qconv_prepare", "qconv", "bnq_tail", "qgemm_codes", "qconv_codes",
           "enable_code_gemm", "disable_code_gemm", "QGEMM_I8", "QGEMM_E4M3"]


def _qp(form, lo, hi, g, scale, offset):
    return QParams(int(form), int(lo), int(hi), float(g), scale.data_ptr(), offset.data_ptr() if offset is not None else None)


def codes_forward(x, scale, offset, lo, hi, form, g=0.0, ch_axis=None, encoding=QGEMM_I8):
    """x -> its integer codes, one byte per element (uint8 tensor of x's shape and memory format; two's complement
    for signed ranges, or the e4m3 byte of the code with `encoding=QGEMM_E4M3`).  Same codes as `fq_forward`."""
    F._require_cuda(x, "x")
    x = F._dense(x.detach(), ch_axis)
    lay = F.layout_of(x, ch_axis)
    s = F._qvec(scale, lay.channels, x.device, "scale")
    o = F._qvec(offset, lay.channels, x.device, "offset")
    codes = torch.empty_like(x, dtype=torch.uint8)
    qp = _qp(form, lo, hi, g, s, o)
    with F._on(x.device):
        _lib.check(_lib.lib().dlmcq_codes_forward(F._ptr(x), F._ptr(codes), C.byref(lay), C.byref(qp), int(encoding),
                                                  F._stream_ptr()))
    return codes


def _prepare_args(dev, n, act, wt, bias):
    a_s, a_o, a_lo, a_hi, a_form, a_g = act
    w_s, w_lo, w_hi, w_form, w_g = wt
    a_s = F._qvec(a_s, 1, dev, "activation scale")
    a_o = F._qvec(a_o, 1, dev, "activation offset")
    w_ch = n if (isinstance(w_s, torch.Tensor) and w_s.numel() == n and n != 1) else 1
    w_s = F._qvec(w_s, w_ch, dev, "weight scale")
    b = None
    if bias is not None:
        b = bias.detach().to(device=dev, dtype=torch.float32).contiguous()
        if b.numel() != n:
            raise DlmcqError("bias must have n entries")
    # the QParams hold raw pointers: the tensors are returned with them so that they outlive the call
    return _qp(a_form, a_lo, a_hi, a_g, a_s, a_o), _qp(w_form, w_lo, w_hi, w_g, w_s, None), w_ch, b, (a_s, a_o, w_s)


def qgemm_prepare(w_codes, act, wt, bias=None, encoding=QGEMM_I8):
    """alpha[n], beta[n] of `qgemm` from device-resident quantizer parameters (no host sync).
    act = (scale, offset_or_zero_point, lo, hi, form, g), wt = (scale [n] or [1], lo, hi, form, g); w_codes [n, k]."""
    F._require_cuda(w_codes, "w_codes")
    if w_codes.dtype != torch.uint8 or w_codes.dim() != 2 or not w_codes.is_contiguous():
        raise DlmcqError("w_codes must be a contiguous [n, k] uint8 tensor")
    n, k = w_codes.shape
    dev = w_codes.device
    qa, qw, w_ch, b, keep = _prepare_args(dev, n, act, wt, bias)
    alpha = torch.empty(n, dtype=torch.float32, device=dev)
    beta = torch.empty(n, dtype=torch.float32, device=dev)
    with F._on(dev):
        _lib.check(_lib.lib().dlmcq_qgemm_prepare(F._ptr(w_codes), n, k, int(encoding), C.byref(qa), C.byref(qw), w_ch,
                                                  F._ptr(b), F._ptr(alpha), F._ptr(beta), F._stream_ptr()))
    del keep
    return alpha, beta


def _pair(v, name):
    t = (v, v) if isinstance(v, int) else tuple(v)
    if len(t) != 2 or not all(isinstance(e, int) for e in t):
        raise DlmcqError(f"{name} must be an int or a pair of ints")
    return t


def _geom(batch, h, w, cin, n, kh, kw, stride=1, padding=0, dilation=1):
    (sh, sw), (ph, pw), (dh, dw) = _pair(stride, "stride"), _pair(padding, "padding"), _pair(dilation, "dilation")
    return ConvGeom(batch, h, w, cin, n, kh, kw, sh, sw, ph, pw, dh, dw, 1)


def conv_out_size(size, k, stride, padding, dilation):
    return (size + 2 * padding - dilation * (k - 1) - 1) // stride + 1


def qconv_prepare(w_codes, act, wt, bias=None, encoding=QGEMM_I8):
    """alpha [n] and the border-class beta table [(kh+1)^2 (kw+1)^2, n] of `qconv` from device-resident quantizer
    parameters (no host sync): beta[class] covers the filter taps of a window that lie inside the image
    (include/dlmcq.h, `dlmcq_qconv_prepare`).  w_codes: [n, kh, kw, cin] uint8 (channels-last weight codes);
    act, wt as in `qgemm_prepare`."""
    F._require_cuda(w_codes, "w_codes")
    if w_codes.dtype != torch.uint8 or w_codes.dim() != 4 or not w_codes.is_contiguous():
        raise DlmcqError("w_codes must be a contiguous [n, kh, kw, cin] uint8 tensor")
    n, kh, kw, cin = w_codes.shape
    dev = w_codes.device
    qa, qw, w_ch, b, keep = _prepare_args(dev, n, act, wt, bias)
    alpha = torch.empty(n, dtype=torch.float32, device=dev)
    beta = torch.empty((kh + 1) ** 2 * (kw + 1) ** 2, n, dtype=torch.float32, device=dev)
    g = _geom(1, 1, 1, cin, n, kh, kw)
    with F._on(dev):
        _lib.check(_lib.lib().dlmcq_qconv_prepare(F._ptr(w_codes), C.byref(g), int(encoding), C.byref(qa), C.byref(qw),
                                                  w_ch, F._ptr(b), F._ptr(alpha), F._ptr(beta), F._stream_ptr()))
    del keep
    return alpha, beta


def qconv(a_codes, w_codes, alpha, beta, stride=1, padding=0, dilation=1, relu=False, out_dtype=torch.float32,
          a_signed=False, encoding=QGEMM_I8, out=None):
    """Convolution of channels-last codes: a_codes [B, H, W, cin], w_codes [n, kh, kw, cin] (uint8, contiguous) ->
    out [B, Ho, Wo, n] = alpha[n] * acc + beta[border class][n] (two fp32 roundings), optional ReLU; zero padding
    of the fake-quantised tensor, i.e. padded taps contribute neither to acc nor to beta."""
    F._require_cuda(a_codes, "a_codes")
    F._require_cuda(w_codes, "w_codes")
    if a_codes.dtype != torch.uint8 or w_codes.dtype != torch.uint8 or a_codes.dim() != 4 or w_codes.dim() != 4:
        raise DlmcqError("a_codes [B, H, W, cin] and w_codes [n, kh, kw, cin] must be uint8 tensors")
    if not (a_codes.is_contiguous() and w_codes.is_contiguous()):
        raise DlmcqError("code tensors must be contiguous (channels innermost)")
    bsz, h, w, cin = a_codes.shape
    n, kh, kw, cin2 = w_codes.shape
    if cin != cin2 or alpha.numel() != n or tuple(beta.shape) != ((kh + 1) ** 2 * (kw + 1) ** 2, n):
        raise DlmcqError("shape mismatch between a_codes, w_codes, alpha, beta")
    if out_dtype not in (torch.float32, torch.bfloat16):
        raise DlmcqError("out_dtype must be float32 or bfloat16")
    g = _geom(bsz, h, w, cin, n, kh, kw, stride, padding, dilation)
    ho = conv_out_size(h, kh, g.stride_h, g.pad_h, g.dil_h)
    wo = conv_out_size(w, kw, g.stride_w, g.pad_w, g.dil_w)
    if ho < 1 or wo < 1:
        raise DlmcqError("the convolution has no output pixel")
    shape = (bsz, ho, wo, n)
    if out is None:
        out = torch.empty(shape, dtype=out_dtype, device=a_codes.device)
    elif tuple(out.shape) != shape or out.dtype != out_dtype or not out.is_contiguous() or out.device != a_codes.device:
        raise DlmcqError("out must be a contiguous [B, Ho, Wo, n] tensor of out_dtype on the operands' device")
    if bsz == 0:
        return out                           # an empty batch, as qgemm with m = 0 (dlmcq_qconv refuses batch 0)
    with F._on(a_codes.device):
        _lib.check(_lib.lib().dlmcq_qconv(F._ptr(a_codes), F._ptr(w_codes), F._ptr(alpha), F._ptr(beta), F._ptr(out),
                                          C.byref(g), int(encoding), int(bool(a_signed)), int(bool(relu)),
                                          F32 if out_dtype == torch.float32 else BF16, F._stream_ptr()))
    return out


def qgemm(a_codes, w_codes, alpha, beta, relu=False, out_dtype=torch.float32, a_signed=False, encoding=QGEMM_I8,
          out=None):
    """out[m, n] = alpha[n] * (sum_k a_codes[m, k] * w_codes[n, k]) + beta[n]  (two fp32 roundings), optional ReLU."""
    F._require_cuda(a_codes, "a_codes")
    if a_codes.dtype != torch.uint8 or w_codes.dtype != torch.uint8 or a_codes.dim() != 2 or w_codes.dim() != 2:
        raise DlmcqError("a_codes [m, k] and w_codes [n, k] must be uint8 matrices")
    if not (a_codes.is_contiguous() and w_codes.is_contiguous()):
        raise DlmcqError("code matrices must be contiguous (row-major, K innermost)")
    m, k = a_codes.shape
    n, k2 = w_codes.shape
    if k != k2 or alpha.numel() != n or beta.numel() != n:
        raise DlmcqError("shape mismatch between a_codes, w_codes, alpha, beta")
    if out_dtype not in (torch.float32, torch.bfloat16):
        raise DlmcqError("out_dtype must be float32 or bfloat16")
    if out is None:
        out = torch.empty(m, n, dtype=out_dtype, device=a_codes.device)
    elif out.shape != (m, n) or out.dtype != out_dtype or not out.is_contiguous() or out.device != a_codes.device:
        raise DlmcqError("out must be a contiguous [m, n] tensor of out_dtype on the operands' device")
    with F._on(a_codes.device):
        _lib.check(_lib.lib().dlmcq_qgemm(F._ptr(a_codes), F._ptr(w_codes), F._ptr(alpha), F._ptr(beta), F._ptr(out), m, n,
                                          k, int(encoding), int(bool(a_signed)), int(bool(relu)),
                                          F32 if out_dtype == torch.float32 else BF16, F._stream_ptr()))
    return out


def bnq_tail(running_mean, running_var, scale, offset, lo, hi, g, gamma=None, beta=None, eps=1e-5, relu=True,
             inter_dtype=torch.float32, encoding=QGEMM_I8):
    """What `qgemm_codes` / `qconv_codes` apply to the layer output in the epilogue (include/dlmcq.h, dlmcq_bnq_tail):
    eval BatchNorm with the running buffers (gamma / beta None: 1 / 0), optional ReLU, then the consumer's per-tensor
    AFFINE input quantizer (scale, offset: one fp32 element each; code range [lo, hi]; grad_scale factor g), whose codes
    are written in `encoding`.  inter_dtype: the dtype the unchained layer output has (float32 or bfloat16)."""
    if inter_dtype not in (torch.float32, torch.bfloat16):
        raise DlmcqError("inter_dtype must be float32 or bfloat16")
    F._require_cuda(running_mean, "running_mean")
    dev, ch = running_mean.device, running_mean.numel()
    bn = (running_mean, running_var, gamma, beta)
    for name, v in zip(("running_mean", "running_var", "gamma", "beta"), bn):
        if v is None and name.startswith("running"):
            raise DlmcqError(f"{name} is required")
        if v is not None and not (isinstance(v, torch.Tensor) and v.dtype is torch.float32 and v.device == dev and
                                  v.numel() == ch and v.is_contiguous()):
            raise DlmcqError(f"{name} must be a contiguous float32 tensor of {ch} elements on {dev}")
    scale = F._qvec(scale, 1, dev, "scale")
    offset = F._qvec(offset, 1, dev, "offset")
    qp = _qp(FORM_AFFINE, lo, hi, g, scale, offset)
    t = BnqTail(F._ptr(gamma), F._ptr(beta), F._ptr(running_mean), F._ptr(running_var), float(eps), int(bool(relu)),
                F32 if inter_dtype == torch.float32 else BF16, C.pointer(qp), int(encoding))
    # the descriptor holds raw pointers: keep the tensors alive with it
    t._keep = [v.detach() for v in (*bn, scale, offset) if v is not None]
    t._channels, t._device = ch, dev
    return t


def _check_tail(tail, n, device):
    """The tail's BatchNorm covers the n output channels, on the operands' device (`bnq_tail` checked the rest)."""
    if not isinstance(tail, BnqTail) or getattr(tail, '_channels', None) is None:
        raise DlmcqError("tail must come from bnq_tail")
    if tail._channels != n or tail._device != device:
        raise DlmcqError(f"the tail's BatchNorm has {tail._channels} channels on {tail._device}; the layer has {n} "
                         f"output channels on {device}")


def qgemm_codes(a_codes, w_codes, alpha, beta, tail, a_signed=False, encoding=QGEMM_I8, out=None):
    """`qgemm` followed by the BatchNorm / ReLU / quantizer `tail` (`bnq_tail`) in the same kernel: the consumer's codes
    [m, n] (uint8), byte-identical to `qgemm` with out_dtype = the tail's inter_dtype and then the fused BatchNorm
    producer's codes of that output (include/dlmcq.h, dlmcq_qgemm_codes).  n must be a multiple of 16."""
    F._require_cuda(a_codes, "a_codes")
    if a_codes.dtype != torch.uint8 or w_codes.dtype != torch.uint8 or a_codes.dim() != 2 or w_codes.dim() != 2:
        raise DlmcqError("a_codes [m, k] and w_codes [n, k] must be uint8 matrices")
    if not (a_codes.is_contiguous() and w_codes.is_contiguous()):
        raise DlmcqError("code matrices must be contiguous (row-major, K innermost)")
    m, k = a_codes.shape
    n, k2 = w_codes.shape
    if k != k2 or alpha.numel() != n or beta.numel() != n:
        raise DlmcqError("shape mismatch between a_codes, w_codes, alpha, beta")
    if out is None:
        out = torch.empty(m, n, dtype=torch.uint8, device=a_codes.device)
    elif out.shape != (m, n) or out.dtype != torch.uint8 or not out.is_contiguous() or out.device != a_codes.device:
        raise DlmcqError("out must be a contiguous [m, n] uint8 tensor on the operands' device")
    _check_tail(tail, n, a_codes.device)
    with F._on(a_codes.device):
        _lib.check(_lib.lib().dlmcq_qgemm_codes(F._ptr(a_codes), F._ptr(w_codes), F._ptr(alpha), F._ptr(beta),
                                                F._ptr(out), m, n, k, int(encoding), int(bool(a_signed)), C.byref(tail),
                                                F._stream_ptr()))
    return out


def qconv_codes(a_codes, w_codes, alpha, beta, tail, stride=1, padding=0, dilation=1, a_signed=False,
                encoding=QGEMM_I8, out=None):
    """`qconv` followed by the BatchNorm / ReLU / quantizer `tail` (`bnq_tail`) in the same kernel: the consumer's codes
    [B, Ho, Wo, n] (uint8, channels-last), byte-identical to `qconv` with out_dtype = the tail's inter_dtype and then the
    fused BatchNorm producer's codes of that output (include/dlmcq.h, dlmcq_qconv_codes).  n must be a multiple of 16."""
    F._require_cuda(a_codes, "a_codes")
    F._require_cuda(w_codes, "w_codes")
    if a_codes.dtype != torch.uint8 or w_codes.dtype != torch.uint8 or a_codes.dim() != 4 or w_codes.dim() != 4:
        raise DlmcqError("a_codes [B, H, W, cin] and w_codes [n, kh, kw, cin] must be uint8 tensors")
    if not (a_codes.is_contiguous() and w_codes.is_contiguous()):
        raise DlmcqError("code tensors must be contiguous (channels innermost)")
    bsz, h, w, cin = a_codes.shape
    n, kh, kw, cin2 = w_codes.shape
    if cin != cin2 or alpha.numel() != n or tuple(beta.shape) != ((kh + 1) ** 2 * (kw + 1) ** 2, n):
        raise DlmcqError("shape mismatch between a_codes, w_codes, alpha, beta")
    g = _geom(bsz, h, w, cin, n, kh, kw, stride, padding, dilation)
    ho = conv_out_size(h, kh, g.stride_h, g.pad_h, g.dil_h)
    wo = conv_out_size(w, kw, g.stride_w, g.pad_w, g.dil_w)
    if ho < 1 or wo < 1:
        raise DlmcqError("the convolution has no output pixel")
    shape = (bsz, ho, wo, n)
    if out is None:
        out = torch.empty(shape, dtype=torch.uint8, device=a_codes.device)
    elif tuple(out.shape) != shape or out.dtype != torch.uint8 or not out.is_contiguous() or out.device != a_codes.device:
        raise DlmcqError("out must be a contiguous [B, Ho, Wo, n] uint8 tensor on the operands' device")
    _check_tail(tail, n, a_codes.device)
    if bsz == 0:
        return out
    with F._on(a_codes.device):
        _lib.check(_lib.lib().dlmcq_qconv_codes(F._ptr(a_codes), F._ptr(w_codes), F._ptr(alpha), F._ptr(beta),
                                                F._ptr(out), C.byref(g), int(encoding), int(bool(a_signed)),
                                                C.byref(tail), F._stream_ptr()))
    return out


# ---------------------------------------------------------------------------------------------------------------
# module level
# ---------------------------------------------------------------------------------------------------------------
def _family(mod):
    """(activation form, weight form) of a quantised layer, or None for families the code path does not serve."""
    from .scalar.FSPTQuant.base import FSPTQBase
    from .scalar.modules.base import QBase
    if isinstance(mod, QBase):
        return FORM_AFFINE, FORM_AFFINE
    if isinstance(mod, FSPTQBase):
        if mod.qconfig['weight'].get('recon_type') in ('adaround', 'dist_recon'):
            return None                      # AdaRound codes come from a different rounding rule (adaround_kernels.cu)
        return FORM_ZP, FORM_SYM
    return None


def _geometry_ok(mod):
    if isinstance(mod, nn.Linear):
        return mod.in_features % 16 == 0
    if isinstance(mod, nn.Conv2d):
        one = (1, 1)
        return (tuple(mod.kernel_size) == one and tuple(mod.stride) == one and tuple(mod.dilation) == one and
                tuple(mod.padding) == (0, 0) and mod.groups == 1 and mod.padding_mode == 'zeros' and
                mod.in_channels % 16 == 0)
    return False


def _conv_geometry_ok(mod):
    """Conv2d layers the implicit-GEMM kernel serves (dlmcq_qconv): one group, zero padding, Cin a multiple of 64,
    stride <= 8 and im2col bounding-box corners -pad, pad - dil*(k-1) in [-128, 127].  Stride-1 1x1 layers without
    padding keep the plain GEMM (`_geometry_ok`)."""
    if not isinstance(mod, nn.Conv2d) or isinstance(mod.padding, str) or _geometry_ok(mod):
        return False
    if mod.groups != 1 or mod.padding_mode != 'zeros' or mod.in_channels % 64 != 0:
        return False
    for k, s, p, d in zip(mod.kernel_size, mod.stride, mod.padding, mod.dilation):
        if not (1 <= s <= 8 and 0 <= p <= 128 and -128 <= p - d * (k - 1) <= 127 and k <= 255):
            return False
    return True


def _enabled(mod):
    q = mod.qconfig
    if hasattr(mod, 'act_quant'):            # FSPTQBase switches (change_quant_state)
        return bool(mod.act_quant) and bool(mod.wt_quant)
    return bool(q['input']['enable']) and bool(q['weight']['enable'])


class _CodeGemmState:
    """Per-layer cache of the weight codes and the epilogue vectors, rebuilt when any tensor they derive from changes."""

    def __init__(self, encoding, conv=False):
        self.encoding = encoding
        self.conv = conv                     # implicit-GEMM convolution (qconv) instead of the [m, k] GEMM
        self.key = None
        self.w_codes = self.alpha = self.beta = None
        self.usable = None                   # None = not decided yet (needs initialised qparams)

    def refresh(self, mod, forms):
        a_form, w_form = forms
        off = getattr(mod, 'wt_offset', None)
        key = (mod.weight._version, mod.wt_scale._version, mod.in_scale._version,
               None if mod.in_offset is None else (mod.in_offset.data_ptr(), mod.in_offset._version),
               None if mod.bias is None else mod.bias._version, mod.weight.data_ptr())
        if key == self.key:
            return self.usable
        self.key = key
        n = mod.weight.shape[0]
        ws, ins = mod.wt_scale.detach(), mod.in_scale.detach()
        usable = ins.numel() == 1 and ws.numel() in (1, n)
        if usable and w_form == FORM_AFFINE and isinstance(off, torch.Tensor):
            usable = not bool(off.any())     # one sync per weight update, never per forward
        if usable and a_form == FORM_ZP and isinstance(mod.in_offset, torch.Tensor):
            # FSPTQuant/base.py:108-109 adds whatever offset the observer returned; only an INTEGRAL zero-point keeps
            # clamp(round(x/s) + zp) an integer code (the min/max observer of a post-ReLU tensor gives 0)
            zp = mod.in_offset.detach()
            usable = bool((zp == zp.round()).all())
        lo_w, hi_w, lo_a, hi_a = mod.wt_min_val, mod.wt_max_val, mod.in_min_val, mod.in_max_val
        if self.encoding == QGEMM_E4M3:
            usable = usable and lo_w >= -16 and hi_w <= 16 and lo_a >= -16 and hi_a <= 16
        else:
            usable = usable and lo_w >= -128 and hi_w <= 127 and lo_a >= -128 and hi_a <= 255 and (lo_a >= 0 or hi_a <= 127)
        usable = usable and accumulator_exact(self.encoding, mod.weight[0].numel(), lo_a, hi_a, lo_w, hi_w)
        self.usable = usable
        if not usable:
            self.w_codes = self.alpha = self.beta = None
            return False
        w = mod.weight.detach()
        if self.conv:
            w2 = w.permute(0, 2, 3, 1).contiguous()      # [n, kh, kw, cin]: K in (r, s, c) order
        else:
            w2 = w.reshape(n, -1)            # 1x1 conv weights [n, k, 1, 1] are [n, k] matrices in either memory format
            w2 = w2 if w2.is_contiguous() else w2.contiguous()
        g_w = 1 / math.sqrt(w.numel() * hi_w) if w_form == FORM_AFFINE else 0.0
        per_ch = ws.numel() == n and n != 1
        self.w_codes = codes_forward(w2, ws.reshape(-1), None, lo_w, hi_w, w_form, g_w, ch_axis=0 if per_ch else None,
                                     encoding=self.encoding)
        self._wt = (ws.reshape(-1), lo_w, hi_w, w_form, g_w)
        self._g_a = 0.0                      # the activation's grad_scale factor depends on the input's numel: epilogue()
        self.alpha = self.beta = None
        self._ab_numel = None
        return True

    def epilogue(self, mod, forms, numel):
        """alpha / beta; for the AFFINE activation form the multiplier is the grad_scale value (s - s*g) + s*g with
        g = 1/sqrt(numel * qmax) (modules/base.py:96-97), so the vectors are keyed on the input's element count."""
        a_form, _ = forms
        if self.alpha is not None and (a_form != FORM_AFFINE or self._ab_numel == numel):
            return self.alpha, self.beta
        g_a = 1 / math.sqrt(numel * mod.in_max_val) if a_form == FORM_AFFINE else 0.0
        act = (mod.in_scale.detach().reshape(-1), mod.in_offset, mod.in_min_val, mod.in_max_val, a_form, g_a)
        prepare = qconv_prepare if self.conv else qgemm_prepare
        self.alpha, self.beta = prepare(self.w_codes, act, self._wt, mod.bias, self.encoding)
        self._ab_numel = numel
        self._g_a = g_a
        return self.alpha, self.beta


def _code_state(mod, dtype, dim):
    """The layer's _CodeGemmState when this call runs on the code path, else None: a switched, enabled and initialised
    layer in eval mode without autograd, an input it serves, and qparams the state finds usable."""
    st = mod.__dict__.get('_code_gemm')
    # inference only: under autograd the layer keeps the differentiable fake-quant path
    if (st is None or mod.training or torch.is_grad_enabled() or dtype not in (torch.float32, torch.bfloat16)
            or not _enabled(mod) or not (mod._ready('in', mod.in_init_state) and mod._ready('wt', mod.wt_init_state))):
        return None
    if isinstance(mod, nn.Conv2d) and dim != 4:
        return None
    return st if st.refresh(mod, mod.__dict__['_code_gemm_forms']) else None


def code_input_spec(consumer, numel, dtype, dim):
    """(encoding, g) when `consumer` - a layer switched by enable_code_gemm - takes its input of `numel` elements as
    codes in this call: the operand encoding and the AFFINE quantizer's grad_scale factor g = 1/sqrt(numel * qmax)
    (modules/base.py:96) its own x -> codes pass would use.  None otherwise (the layer then quantises what it is
    given).  Producers that can emit the codes themselves (fuse.py) ask this before every call."""
    st = _code_state(consumer, dtype, dim)
    if st is None or consumer.__dict__['_code_gemm_forms'][0] != FORM_AFFINE:
        return None
    return st.encoding, 1 / math.sqrt(numel * consumer.in_max_val)


def output_shape(mod, in_shape):
    """Shape of a switched layer's output (and of its codes from `forward_codes` with a tail) for an input of
    `in_shape`."""
    n = mod.weight.shape[0]
    if not isinstance(mod, nn.Conv2d):
        return tuple(in_shape[:-1]) + (n,)
    b, _, h, w = in_shape
    if not mod.__dict__['_code_gemm'].conv:
        return (b, n, h, w)
    (kh, kw), (sh, sw), (ph, pw), (dh, dw) = mod.kernel_size, mod.stride, mod.padding, mod.dilation
    return (b, n, conv_out_size(h, kh, sh, ph, dh), conv_out_size(w, kw, sw, pw, dw))


def forward_codes(mod, a_codes, out_dtype, tail=None):
    """The switched layer on its input's codes (uint8, the input's shape: [..., K] for Linear, an NCHW view of
    channels-last [B, H, W, Cin] storage for Conv2d), in the encoding of the layer's state.  Call only when
    `code_input_spec` (or `_code_state`) accepted the layer for this input.
    tail = (bn, relu, consumer, encoding, g): return instead the consumer's input codes of relu(bn(output)) (uint8, the
    output's shape and memory format) from the same kernel - eval `bn` with running statistics, the consumer's
    per-tensor AFFINE input quantizer with grad_scale factor g, codes in `encoding` (`code_input_spec`), byte-identical
    to the output in out_dtype followed by the fused BatchNorm producer's codes (fuse.py)."""
    st = mod.__dict__['_code_gemm']
    mod.__dict__.pop('_wq', None)                        # a weight group's pre-hook may have staged its copy: unused here
    alpha, beta = st.epilogue(mod, mod.__dict__['_code_gemm_forms'], a_codes.numel())
    t = None
    if tail is not None:
        bn, relu, consumer, encoding, g = tail
        t = bnq_tail(bn.running_mean, bn.running_var, consumer.in_scale.detach().reshape(-1),
                     consumer.in_offset.detach().reshape(-1), consumer.in_min_val, consumer.in_max_val, g,
                     bn.weight, bn.bias, bn.eps, relu, out_dtype, encoding)
    a_signed = mod.in_min_val < 0
    if st.conv:
        a = a_codes.permute(0, 2, 3, 1)
        if t is not None:
            out = qconv_codes(a, st.w_codes, alpha, beta, t, mod.stride, mod.padding, mod.dilation, a_signed=a_signed,
                              encoding=st.encoding)
        else:
            out = qconv(a, st.w_codes, alpha, beta, mod.stride, mod.padding, mod.dilation, out_dtype=out_dtype,
                        a_signed=a_signed, encoding=st.encoding)
        return out.permute(0, 3, 1, 2)                           # NCHW view of channels-last storage
    n = mod.weight.shape[0]
    if isinstance(mod, nn.Conv2d):
        b, k, h, w = a_codes.shape
        # elementwise codes keep x's memory order: channels-last NCHW storage is the [B*H*W, C] matrix
        a = a_codes.permute(0, 2, 3, 1).reshape(b * h * w, k)
        if t is not None:
            out = qgemm_codes(a, st.w_codes, alpha, beta, t, a_signed=a_signed, encoding=st.encoding)
        else:
            out = qgemm(a, st.w_codes, alpha, beta, out_dtype=out_dtype, a_signed=a_signed, encoding=st.encoding)
        return out.view(b, h, w, n).permute(0, 3, 1, 2)          # NCHW view of channels-last storage
    k = a_codes.shape[-1]
    a = a_codes.reshape(-1, k)
    if t is not None:
        out = qgemm_codes(a, st.w_codes, alpha, beta, t, a_signed=a_signed, encoding=st.encoding)
    else:
        out = qgemm(a, st.w_codes, alpha, beta, out_dtype=out_dtype, a_signed=a_signed, encoding=st.encoding)
    return out.view(*a_codes.shape[:-1], n)


def input_codes(mod, input):
    """A switched layer's input codes for this call (`_code_state` accepted it): the codes a fused producer handed over
    (`_dlmcq_codes`), else its own x -> codes pass; None when a fused producer handed over the fake-quantised tensor
    instead (`_dlmcq_q`: the layer then runs its original forward on it)."""
    pre = getattr(input, '_dlmcq_codes', None)           # (consumer, codes) from a fused producer (fuse.py)
    if pre is not None and pre[0] is mod:
        return pre[1]
    pre = getattr(input, '_dlmcq_q', None)
    if pre is not None and pre[0] is mod:
        return None
    st = mod.__dict__['_code_gemm']
    a_form, _ = mod.__dict__['_code_gemm_forms']
    if isinstance(mod, nn.Conv2d):
        x = input if input.is_contiguous(memory_format=torch.channels_last) else \
            input.contiguous(memory_format=torch.channels_last)
    else:
        x = input if input.is_contiguous() else input.contiguous()
    st.epilogue(mod, mod.__dict__['_code_gemm_forms'], x.numel())
    return codes_forward(x, mod.in_scale.detach().reshape(-1), mod.in_offset, mod.in_min_val, mod.in_max_val, a_form,
                         st._g_a, encoding=st.encoding)


def _code_forward(self, input):
    st = _code_state(self, input.dtype, input.dim()) if input.is_cuda else None
    if st is None:
        return self._code_gemm_orig_forward(input)
    a_codes = input_codes(self, input)
    if a_codes is None:
        return self._code_gemm_orig_forward(input)      # a fused producer already handed over the fake-quantised tensor
    return forward_codes(self, a_codes, input.dtype)


def accumulator_exact(encoding, k, a_lo, a_hi, w_lo, w_hi):
    """Whether every partial sum of k code products fits the encoding's accumulator exactly (include/dlmcq.h):
    k * max|a| * max|w| <= 2^24 for e4m3 (fp32 accumulators), <= 2^31 - 1 for the integer kind (s32).  The prepare
    entries refuse the layers that fail it."""
    bound = (1 << 24) if encoding == QGEMM_E4M3 else (1 << 31) - 1
    return k * max(-a_lo, a_hi) * max(-w_lo, w_hi) <= bound


def _auto_encoding(mod):
    """e4m3 operands (fp32 accumulators: no int -> float conversion in the epilogue) when every code of the layer is
    exactly representable (|code| <= 16, i.e. up to 4-bit unsigned / 5-bit signed ranges) and the layer's K keeps the
    fp32 accumulation exact, the integer kind otherwise, None when neither accumulates exactly.  Both are bit-identical
    where both apply (tests/qgemm_cases.py)."""
    k = mod.weight[0].numel()
    ranges = (mod.in_min_val, mod.in_max_val, mod.wt_min_val, mod.wt_max_val)
    small = mod.wt_min_val >= -16 and mod.wt_max_val <= 16 and mod.in_min_val >= -16 and mod.in_max_val <= 16
    if small and accumulator_exact(QGEMM_E4M3, k, *ranges):
        return QGEMM_E4M3
    return QGEMM_I8 if accumulator_exact(QGEMM_I8, k, *ranges) else None


def enable_code_gemm(model, encoding=None, convolutions=False):
    """Route every eligible quantised Linear / 1x1 Conv2d of `model` through the integer-code GEMM in eval mode
    (`encoding`: QGEMM_I8, QGEMM_E4M3, or None = per layer by code range and K, `_auto_encoding`; a layer that
    no encoding accumulates exactly is not switched).  With `convolutions=True` also every
    quantised Conv2d the implicit-GEMM kernel serves (k x k, strided, padded, dilated; one group, zero padding,
    Cin % 64 == 0): `qconv` on the channels-last codes.
    Returns the list of module names switched.  Eligibility that depends on calibrated state (per-tensor activation
    scale, zero weight offset, ...) is re-checked lazily and a layer that fails it silently keeps its original path."""
    names = []
    for name, mod in model.named_modules():
        forms = _family(mod)
        if forms is None or '_code_gemm' in mod.__dict__:
            continue
        conv = convolutions and _conv_geometry_ok(mod)
        if not (conv or _geometry_ok(mod)):
            continue
        enc = _auto_encoding(mod) if encoding is None else encoding
        if enc is None:
            continue                         # no operand encoding accumulates this layer's K exactly
        mod.__dict__['_code_gemm'] = _CodeGemmState(enc, conv)
        mod.__dict__['_code_gemm_forms'] = forms
        mod.__dict__['_code_gemm_orig_forward'] = mod.forward
        mod.forward = types.MethodType(_code_forward, mod)
        names.append(name)
    return names


def disable_code_gemm(model):
    for mod in model.modules():
        if '_code_gemm' in mod.__dict__:
            del mod.__dict__['forward']
            for k in ('_code_gemm', '_code_gemm_forms', '_code_gemm_orig_forward'):
                mod.__dict__.pop(k, None)
