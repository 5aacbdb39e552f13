"""CPU tests of dlmcq_bnq_forward_codes: every refusal is returned before any CUDA call (no GPU here)."""
import ctypes

import pytest


@pytest.fixture(scope="module")
def lib():
    from dlmc_quant_b200 import _lib, build
    build.build()
    return _lib


def test_bnq_forward_codes_refusals_without_gpu(lib):
    h = lib.lib()
    EINVAL, EALIGN, EUNSUPPORTED = -1, -2, -5
    one = ctypes.c_void_p(4096)                     # never dereferenced: every call below fails validation first
    odd = ctypes.c_void_p(4100)
    scale = ctypes.c_void_p(4096)
    eval_relu = lib.BnqDesc(64, 64, lib.F32, lib.BNQ_RELU, 1e-5, 0.1)
    u4 = lib.QParams(lib.FORM_AFFINE, 0, 15, 0.0, scale, scale)

    def f(desc=eval_relu, qp=u4, enc=0, x=one, codes=one, a=None, idn=None):
        return h.dlmcq_bnq_forward_codes(x, idn, one, one, one, one, one, one, a, codes, ctypes.byref(desc),
                                         ctypes.byref(qp) if qp is not None else None, enc, one, 1 << 20, None)
    train = lib.BnqDesc(64, 64, lib.F32, lib.BNQ_TRAINING | lib.BNQ_RELU, 1e-5, 0.1)
    assert f(desc=train) == EUNSUPPORTED                                               # codes have no backward
    assert f(codes=None) == EINVAL
    assert f(qp=None) == EINVAL
    assert f(qp=lib.QParams(lib.FORM_A1, 0, 15, 0.0, scale, scale)) == EINVAL          # not FORM_AFFINE
    assert f(qp=lib.QParams(lib.FORM_AFFINE, 0, 15, 0.0, None, scale)) == EINVAL       # no scale
    assert f(enc=7) == EINVAL                                                          # unknown encoding
    assert f(qp=lib.QParams(lib.FORM_AFFINE, 0, 255, 0.0, scale, scale), enc=1) == EUNSUPPORTED   # 8 bits in e4m3
    assert f(qp=lib.QParams(lib.FORM_AFFINE, -200, 7, 0.0, scale, scale), enc=0) == EUNSUPPORTED
    assert f(qp=lib.QParams(lib.FORM_AFFINE, -128, 255, 0.0, scale, scale), enc=0) == EUNSUPPORTED
    assert f(x=odd) == EALIGN
    assert f(codes=odd) == EALIGN
    assert f(a=odd) == EALIGN
    resid = lib.BnqDesc(64, 64, lib.F32, lib.BNQ_RESIDUAL, 1e-5, 0.1)
    assert f(desc=resid) == EINVAL                                                     # residual flag without identity
    assert f(desc=lib.BnqDesc(64, 6, lib.F32, 0, 1e-5, 0.1)) == EUNSUPPORTED           # channels % 4 != 0
    assert f(desc=lib.BnqDesc(0, 64, lib.F32, 0, 1e-5, 0.1)) == 0                      # empty: nothing to do
