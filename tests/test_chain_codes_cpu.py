"""CPU tests of the chained code layer: every refusal of dlmcq_qgemm_codes / dlmcq_qconv_codes is returned before any
CUDA call, and the host-side parts of the eligibility decision (fuse.chain_spec, qgemm.output_shape) need no device."""
import ctypes

import pytest
import torch
from torch import nn


@pytest.fixture(scope="module")
def lib():
    from dlmc_quant_b200 import _lib, build
    build.build()
    return _lib


def test_chain_entries_refuse_without_gpu(lib):
    h = lib.lib()
    EINVAL, EALIGN, EUNSUPPORTED = -1, -2, -5
    one, odd = ctypes.c_void_p(4096), ctypes.c_void_p(4100)    # never dereferenced: every call fails validation first
    u4 = lib.QParams(lib.FORM_AFFINE, 0, 15, 0.0, one, one)

    def tail(qp=u4, rm=one, rv=one, inter=lib.F32, enc=0):
        t = lib.BnqTail(one, one, rm, rv, 1e-5, 1, inter, ctypes.pointer(qp) if qp is not None else None, enc)
        return ctypes.byref(t)

    def gemm(m=256, n=64, k=64, enc=0, a=one, w=one, out=one, alpha=one, t=None):
        return h.dlmcq_qgemm_codes(a, w, alpha, one, out, m, n, k, enc, 0, tail() if t is None else t, None)

    def conv(geom=None, enc=0, a=one, out=one, t=None, alpha=one):
        g = geom or lib.ConvGeom(2, 8, 8, 64, 64, 3, 3, 1, 1, 1, 1, 1, 1, 1)
        return h.dlmcq_qconv_codes(a, one, alpha, one, out, ctypes.byref(g), enc, 0, tail() if t is None else t, None)

    for f in (gemm, conv):
        assert f(t=ctypes.cast(None, ctypes.POINTER(lib.BnqTail))) == EINVAL                       # no tail
        assert f(t=tail(rm=None)) == EINVAL and f(t=tail(rv=None)) == EINVAL                        # running buffers
        assert f(t=tail(qp=None)) == EINVAL
        assert f(t=tail(qp=lib.QParams(lib.FORM_A1, 0, 15, 0.0, one, one))) == EINVAL              # not AFFINE
        assert f(t=tail(qp=lib.QParams(lib.FORM_AFFINE, 0, 15, 0.0, None, one))) == EINVAL         # no scale
        assert f(t=tail(enc=5)) == EINVAL and f(enc=5) == EINVAL                                    # unknown encodings
        assert f(t=tail(inter=7)) == EINVAL                                                         # unknown dtype
        assert f(t=tail(qp=lib.QParams(lib.FORM_AFFINE, 0, 255, 0.0, one, one), enc=1)) == EUNSUPPORTED
        assert f(t=tail(qp=lib.QParams(lib.FORM_AFFINE, -128, 255, 0.0, one, one))) == EUNSUPPORTED
        assert f(alpha=None) == EINVAL
        assert f(out=odd) == EALIGN and f(a=odd) == EALIGN
    assert gemm(n=72) == EUNSUPPORTED and gemm(n=8) == EUNSUPPORTED                                 # n % 16 != 0
    assert gemm(k=40) == EUNSUPPORTED                                                                # k % 16 (qgemm)
    assert gemm(m=-1) == EINVAL and gemm(n=0) == EINVAL
    assert gemm(m=0) == 0                                                                            # empty
    assert gemm(out=None) == EINVAL
    assert conv(geom=lib.ConvGeom(2, 8, 8, 64, 72, 3, 3, 1, 1, 1, 1, 1, 1, 1)) == EUNSUPPORTED      # n % 16 != 0
    assert conv(geom=lib.ConvGeom(2, 8, 8, 48, 64, 3, 3, 1, 1, 1, 1, 1, 1, 1)) == EUNSUPPORTED      # cin % 64 (qconv)
    assert conv(geom=lib.ConvGeom(0, 8, 8, 64, 64, 3, 3, 1, 1, 1, 1, 1, 1, 1)) == EINVAL            # batch 0 (qconv)
    assert conv(out=None) == EINVAL


def _switched(mod, conv):
    from dlmc_quant_b200 import qgemm as Q
    mod.__dict__['_code_gemm'] = Q._CodeGemmState(Q.QGEMM_I8, conv)
    return mod


def test_output_shape_of_switched_layers():
    from dlmc_quant_b200 import qgemm as Q
    assert Q.output_shape(_switched(nn.Conv2d(64, 128, 1), False), (4, 64, 14, 14)) == (4, 128, 14, 14)
    assert Q.output_shape(_switched(nn.Conv2d(128, 128, 3, 2, 1), True), (4, 128, 56, 56)) == (4, 128, 28, 28)
    assert Q.output_shape(_switched(nn.Conv2d(64, 64, (3, 5), (1, 2), (2, 0), (2, 1)), True), (2, 64, 9, 11)) == \
        (2, 64, 9, 4)
    assert Q.output_shape(_switched(nn.Linear(256, 48), False), (7, 3, 256)) == (7, 3, 48)


def test_chain_spec_declines_without_a_qualifying_site():
    """Each of these declines before it would need a device: no consumer, a BatchNorm in training mode or without
    running statistics, and a producer that is not switched to the code path."""
    from dlmc_quant_b200 import fuse
    prod, cons = nn.Conv2d(64, 64, 1), nn.Conv2d(64, 64, 3, padding=1)
    bn = nn.BatchNorm2d(64).eval()
    dev = torch.device("cpu")
    assert fuse.chain_spec(prod, (2, 64, 8, 8), torch.float32, dev, bn, None) is None
    assert fuse.chain_spec(prod, (2, 64, 8, 8), torch.float32, dev, nn.BatchNorm2d(64).train(), cons) is None
    assert fuse.chain_spec(prod, (2, 64, 8, 8), torch.float32, dev,
                           nn.BatchNorm2d(64, track_running_stats=False).eval(), cons) is None
    assert fuse.chain_spec(prod, (2, 64, 8, 8), torch.float32, dev, bn, cons) is None         # producer not switched


@pytest.fixture
def qualifying(monkeypatch):
    """The device-dependent predicates of chain_spec accept: what is left is its shape and layout logic."""
    from dlmc_quant_b200 import fuse
    from dlmc_quant_b200 import qgemm as Q
    monkeypatch.setattr(Q, "_code_state", lambda *a, **k: object())
    monkeypatch.setattr(fuse, "_consumer_q", lambda *a, **k: (None, None))
    monkeypatch.setattr(Q, "code_input_spec", lambda *a, **k: (0, 1.0))
    return fuse


def test_chain_spec_layout_of_the_producer_output(qualifying):
    """Only outputs that `fusable` would take in the two-kernel chain: a Conv2d's channels-last [B, n, Ho, Wo] or a
    Linear's [rows, n], with BatchNorm over those n channels and n % 16 == 0."""
    spec = qualifying.chain_spec
    dev, f32 = torch.device("cpu"), torch.float32
    lin, cons = _switched(nn.Linear(64, 64), False), nn.Linear(64, 32)
    assert spec(lin, (8, 64), f32, dev, nn.BatchNorm1d(64).eval(), cons) == (0, 1.0)
    # a Linear on a 4-D input writes a contiguous [B, C, H, n]: BatchNorm2d normalises C, the tensor is not fusable
    assert spec(lin, (8, 16, 5, 64), f32, dev, nn.BatchNorm2d(16).eval(), cons) is None
    assert spec(lin, (8, 16, 5, 64), f32, dev, nn.BatchNorm2d(64).eval(), cons) is None
    assert spec(lin, (7, 3, 64), f32, dev, nn.BatchNorm1d(64).eval(), cons) is None          # 3-D: not [rows, C]
    assert spec(lin, (8, 64), f32, dev, nn.BatchNorm1d(32).eval(), cons) is None              # other channel count
    c1 = _switched(nn.Conv2d(64, 64, 1), False)
    c3 = _switched(nn.Conv2d(64, 80, 3, 2, 1), True)
    assert spec(c1, (2, 64, 8, 8), f32, dev, nn.BatchNorm2d(64).eval(), cons) == (0, 1.0)
    assert spec(c3, (2, 64, 9, 9), torch.bfloat16, dev, nn.BatchNorm2d(80).eval(), cons) == (0, 1.0)
    assert spec(c3, (2, 64, 9, 9), f32, dev, nn.BatchNorm2d(64).eval(), cons) is None         # BN over other channels
    assert spec(_switched(nn.Conv2d(64, 72, 1), False), (2, 64, 8, 8), f32, dev, nn.BatchNorm2d(72).eval(),
                cons) is None                                                                   # n % 16 != 0
    half = nn.BatchNorm2d(64).eval()
    half.running_var = half.running_var.half()
    assert spec(c1, (2, 64, 8, 8), f32, dev, half, cons) is None                              # fp32 buffers only


def test_bnq_tail_refuses_host_tensors():
    from dlmc_quant_b200 import qgemm as Q
    from dlmc_quant_b200._lib import DlmcqError
    z = torch.zeros(64)
    with pytest.raises(DlmcqError):
        Q.bnq_tail(z, z, torch.ones(1), torch.zeros(1), 0, 15, 0.1)
