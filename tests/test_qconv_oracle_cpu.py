"""CPU check of the algebra behind the convolution on the integer codes (tests/qconv_oracle.py::code_conv, the
definition dlmcq_qconv is held to bit for bit on the GPU): for every activation form and every geometry the factored
expression - exact integer convolution of the codes, alpha[n], and beta from the filter taps that lie inside the
image - equals the reference's F.conv2d of the two fake-quantised tensors (float64) to 1e-5 of conv2d(|y_a|, |y_w|).
A version with the 1x1 rule's whole-K beta must fail that bar at the border: the test sees the border rule."""
import pytest
import torch
import torch.nn.functional as F

from tests.qconv_oracle import (A1, AFFINE, GEOMETRIES, SYM, ZP, code_conv, conv_pairs, conv_problem, conv_reference,
                                exact_conv, exact_conv_acc)

FORMS = [(AFFINE, AFFINE), (AFFINE, SYM), (ZP, SYM), (A1, SYM), (SYM, SYM)]


def _err(p, whole_k_beta=False, relu=False):
    got = code_conv(p["ca"], p["cw"], p["m_a"], p["o_a"], p["z_a"], p["m_w"], p["bias"], whole_k_beta=whole_k_beta,
                    relu=relu, **p["conv"])
    ref, mag = conv_reference(p["qa"], p["qw"], p["bias"], **p["conv"])
    if relu:
        ref = torch.relu(ref)
    return got, ((got.double() - ref).abs() / mag.clamp_min(1e-30))


@pytest.mark.parametrize("geom", sorted(GEOMETRIES))
@pytest.mark.parametrize("a_form,w_form", FORMS)
@pytest.mark.parametrize("per_channel", [True, False])
def test_factored_conv_equals_reference_conv(geom, a_form, w_form, per_channel):
    p = conv_problem(a_form, w_form, GEOMETRIES[geom], per_channel=per_channel, seed=len(geom))
    got, err = _err(p)
    assert got.dtype == torch.float32
    assert err.max().item() <= 1e-5, err.max().item()


@pytest.mark.parametrize("geom", ["3x3_pad1", "5x5_pad2"])
def test_eight_bit_and_signed_activations(geom):
    for a_signed in (False, True):
        p = conv_problem(SYM if a_signed else ZP, SYM, GEOMETRIES[geom], n_bits=8, a_signed=a_signed, cin=64, seed=3)
        _, err = _err(p)
        assert err.max().item() <= 1e-5
    p = conv_problem(AFFINE, SYM, GEOMETRIES[geom], seed=4)
    got, err = _err(p, relu=True)
    assert (got >= 0).all() and err.max().item() <= 1e-5


@pytest.mark.parametrize("geom", [g for g in sorted(GEOMETRIES) if any(conv_pairs(*GEOMETRIES[g][2:5])[1])])
@pytest.mark.parametrize("a_form", [AFFINE, ZP, A1])
def test_whole_k_beta_fails_at_the_border(geom, a_form):
    """With t = o_a - z_a*m_a != 0 the padded taps would contribute t*m_w*sum(cw) if beta ignored the border; the bar
    catches that at border pixels and only there."""
    p = conv_problem(a_form, SYM, GEOMETRIES[geom], seed=7)
    _, err = _err(p, whole_k_beta=True)
    kh, kw, stride, padding, dilation, h, w = GEOMETRIES[geom]
    (sh, sw), (ph, pw), (dh, dw) = conv_pairs(stride, padding, dilation)
    assert err.max().item() > 1e-3
    # interior pixels (window fully inside) agree with the border-aware form
    ho, wo = err.shape[2], err.shape[3]
    oh = torch.arange(ho) * sh - ph
    ow = torch.arange(wo) * sw - pw
    inside_h = (oh >= 0) & (oh + dh * (kh - 1) < h)
    inside_w = (ow >= 0) & (ow + dw * (kw - 1) < w)
    interior = err[:, :, inside_h][:, :, :, inside_w]
    if interior.numel():
        assert interior.max().item() <= 1e-5


def test_integer_convolution_is_exact():
    g = torch.Generator().manual_seed(0)
    ca = torch.randint(128, 256, (2, 512, 6, 6), generator=g)
    cw = torch.randint(100, 128, (3, 512, 3, 3), generator=g)
    out = code_conv(ca, cw, 1.0, 0.0, 0.0, torch.ones(3), padding=1)
    want = torch.nn.functional.conv2d(ca.to(torch.int64).double(), cw.double(), padding=1)
    assert want.abs().max() > 2 ** 24                           # the s32 -> fp32 conversion rounds
    assert torch.equal(out, want.float())


@pytest.mark.parametrize("geom", sorted(GEOMETRIES))
def test_tapwise_exact_conv_equals_code_conv(geom):
    """exact_conv (one float64 matmul per filter tap, the border sums from tap validity; the GPU reference of the
    batch-128 cases) equals code_conv (float64 conv2d) bit for bit on 8-bit codes, for every geometry."""
    kh, kw, stride, padding, dilation, h, w = GEOMETRIES[geom]
    g = torch.Generator().manual_seed(len(geom))
    ca = torch.randint(0, 256, (2, 64, h, w), generator=g)
    cw = torch.randint(-127, 128, (5, 64, kh, kw), generator=g)
    kw_ = dict(stride=stride, padding=padding, dilation=dilation)
    acc = exact_conv_acc(ca, cw, **kw_)
    assert torch.equal(acc, F.conv2d(ca.double(), cw.double(), **kw_))
    m_w = torch.rand(5, generator=g) * 0.01 + 1e-3
    bias = torch.randn(5, generator=g)
    for relu in (False, True):
        args = (ca, cw, torch.tensor(0.0371), torch.tensor(-0.21), torch.tensor(3.0), m_w, bias)
        assert torch.equal(exact_conv(*args, relu=relu, **kw_), code_conv(*args, relu=relu, **kw_))


def test_python_entry_argument_checks_need_no_gpu():
    """qconv_prepare / qconv refuse CPU tensors and malformed shapes before any CUDA call."""
    from dlmc_quant_b200 import qgemm as Q
    from dlmc_quant_b200._lib import DlmcqError
    a = torch.zeros(1, 8, 8, 64, dtype=torch.uint8)
    w = torch.zeros(4, 3, 3, 64, dtype=torch.uint8)
    al, be = torch.ones(4), torch.zeros(256, 4)
    with pytest.raises(DlmcqError, match="CUDA"):
        Q.qconv(a, w, al, be, padding=1)
    with pytest.raises(DlmcqError, match="CUDA"):
        Q.qconv_prepare(w, (1.0, 0.0, 0, 15, AFFINE, 0.0), (1.0, -7, 7, SYM, 0.0))
    with pytest.raises(DlmcqError):
        Q._geom(1, 8, 8, 64, 4, 3, 3, stride=(1, 2, 3))


def test_enable_flag_selects_conv_layers_without_gpu():
    """Eligibility is decided from the module alone: with convolutions=False the set is exactly the 1x1 / Linear set."""
    from torch import nn
    from dlmc_quant_b200 import qgemm as Q
    ok = [nn.Conv2d(64, 32, 3, padding=1), nn.Conv2d(128, 32, 3, stride=2, padding=1), nn.Conv2d(64, 32, 1, stride=2),
          nn.Conv2d(64, 32, 3, padding=2, dilation=2), nn.Conv2d(64, 32, (1, 3), padding=(0, 1))]
    no = [nn.Conv2d(64, 32, 3, padding=1, groups=2), nn.Conv2d(3, 32, 7, stride=2, padding=3),
          nn.Conv2d(64, 32, 3, padding=1, padding_mode='reflect'), nn.Conv2d(96, 32, 3, padding=1),
          nn.Conv2d(64, 32, 3, stride=9), nn.Conv2d(64, 32, 1), nn.Conv2d(64, 32, 3, padding='same')]
    assert all(Q._conv_geometry_ok(m) for m in ok)
    assert not any(Q._conv_geometry_ok(m) for m in no)
    assert Q._geometry_ok(nn.Conv2d(64, 32, 1)) and not Q._geometry_ok(nn.Conv2d(64, 32, 3, padding=1))
