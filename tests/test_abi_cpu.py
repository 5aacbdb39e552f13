"""CPU tests of the drop-in boundary: libdlmcq.so builds, loads, and exports exactly the entry
points include/dlmcq.h declares (no compute calls - there is no GPU here)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "dlmcq.h")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(dlmcq_[a-z0-9_]+)\s*\(", src)))


@pytest.fixture(scope="module")
def libpath():
    from dlmc_quant_b200 import build
    return build.build()


def test_header_declares_entry_points():
    names = declared_symbols()
    assert "dlmcq_fq_forward" in names and "dlmcq_fq_backward" in names and len(names) >= 25


def test_library_exports_every_declared_symbol(libpath):
    h = ctypes.CDLL(libpath)
    missing = [n for n in declared_symbols() if not hasattr(h, n)]
    assert not missing, f"declared in dlmcq.h but not exported: {missing}"


def test_ctypes_table_matches_header(libpath):
    from dlmc_quant_b200 import _lib
    assert sorted(_lib.SIGNATURES) == declared_symbols()
    h = _lib.lib()
    assert h.dlmcq_version() == 100
    assert h.dlmcq_status_string(0) == b"ok"
    assert h.dlmcq_status_string(-3) == b"workspace too small"


def test_workspace_query_needs_no_gpu(libpath):
    from dlmc_quant_b200 import _lib
    h = _lib.lib()
    base = h.dlmcq_workspace_bytes(None)
    assert base >= 256 + 2048 * 80 * 4          # 80 sweep partials per CTA fit
    lay = _lib.Layout(64, 2048, 49, 0)
    assert h.dlmcq_workspace_bytes(ctypes.byref(lay)) >= 256 + 64 * 2048 * 16
    ctx = ctypes.c_void_p()
    assert h.dlmcq_host_ctx_create(ctypes.byref(ctx), 12345) == -1          # chunk must be a multiple of 8
    assert h.dlmcq_host_ctx_synchronize(None) == -1 and h.dlmcq_host_ctx_destroy(None) == 0


def test_sweep_channel_plan_needs_no_gpu(libpath):
    """The channel sweep's warps per row for the shapes the GPU tests use to reach 1, 2, 4 and 8 warps per row
    (tests/test_gpu_rootq_obs.py), and the CTA count and shared memory that follow from it.  Without a device the SM
    count is 148, a B200's."""
    from dlmc_quant_b200 import _lib
    h = _lib.lib()
    for ch, inner, wpr in ((96, 100, 1), (96, 300, 2), (96, 700, 4), (96, 2304, 8),
                           (6, 100, 1), (6, 300, 2), (6, 700, 4), (6, 1100, 8)):
        it = _lib.SweepItem(channels=ch, inner=inner)
        assert h.dlmcq_obs_sweep_channel_plan(ctypes.byref(it), ch) == 0
        assert (it.wpr, it.staged) == (wpr, 1), (ch, inner)
        assert it.ctas == (ch * wpr + 7) // 8 and it.smem_bytes == (8 // wpr) * it.row_floats * 4, (ch, inner)


def test_argument_validation_without_gpu(libpath):
    """Bad arguments are rejected before any CUDA call is made."""
    from dlmc_quant_b200 import _lib
    h = _lib.lib()
    lay = _lib.Layout(1, 1, 16, 0)
    qp = _lib.QParams(1, 0, 15, 0.0, None, None)
    assert h.dlmcq_fq_forward(None, None, None, ctypes.byref(lay), ctypes.byref(qp), None) == -1
    bad = _lib.Layout(1, 0, 16, 0)
    assert h.dlmcq_fq_forward(None, None, None, ctypes.byref(bad), ctypes.byref(qp), None) == -1


def test_code_gemm_argument_validation_without_gpu(libpath):
    """The integer-code GEMM entries refuse what they cannot compute exactly - before any CUDA call."""
    from dlmc_quant_b200 import _lib
    h = _lib.lib()
    EINVAL, EALIGN, EUNSUPPORTED = -1, -2, -5
    one = ctypes.c_void_p(4096)                     # never dereferenced: every call below fails validation first
    odd = ctypes.c_void_p(4100)
    f = lambda *a: h.dlmcq_qgemm(*a)                # noqa: E731  (a, w, alpha, beta, out, m, n, k, enc, a_signed, relu, dtype, stream)
    assert f(one, one, one, one, one, -1, 8, 16, 0, 0, 0, 0, None) == EINVAL
    assert f(one, one, one, one, one, 4, 8, 16, 7, 0, 0, 0, None) == EINVAL            # unknown operand encoding
    assert f(one, one, one, one, one, 4, 8, 16, 0, 0, 0, 3, None) == EINVAL            # unknown output dtype
    assert f(one, one, one, one, one, 0, 8, 16, 0, 0, 0, 0, None) == 0                 # empty problem
    assert f(None, one, one, one, one, 4, 8, 16, 0, 0, 0, 0, None) == EINVAL
    assert f(odd, one, one, one, one, 4, 8, 16, 0, 0, 0, 0, None) == EALIGN            # TMA needs 16-byte aligned bases
    assert f(one, one, one, one, one, 4, 8, 24, 0, 0, 0, 0, None) == EUNSUPPORTED      # ... and a 16-byte row pitch
    scale = ctypes.c_void_p(4096)
    act = _lib.QParams(1, 0, 15, 0.0, scale, None)
    wt = _lib.QParams(3, -7, 7, 0.0, scale, None)
    g = lambda a, w, ch=8, enc=0: h.dlmcq_qgemm_prepare(one, 8, 16, enc, ctypes.byref(a), ctypes.byref(w), ch, None, one, one, None)  # noqa: E731
    assert g(act, _lib.QParams(1, -7, 7, 0.0, scale, scale)) == EUNSUPPORTED           # weight offset: product does not factor
    assert g(act, _lib.QParams(2, 0, 15, 0.0, scale, None)) == EUNSUPPORTED            # zero-point weights
    assert g(act, wt, ch=3) == EINVAL                                                  # scales: n or 1 entries
    assert g(_lib.QParams(2, 0, 255, 0.0, scale, scale), wt, enc=1) == EUNSUPPORTED    # 8-bit codes are not e4m3 integers
    assert g(act, _lib.QParams(3, 0, 255, 0.0, scale, None)) == EUNSUPPORTED           # B operand is int8
    lay = _lib.Layout(1, 1, 16, 0)
    c = lambda qp, enc: h.dlmcq_codes_forward(one, one, ctypes.byref(lay), ctypes.byref(qp), enc, None)  # noqa: E731
    assert c(act, 5) == EINVAL
    assert c(_lib.QParams(2, 0, 255, 0.0, scale, None), 1) == EUNSUPPORTED
    assert c(_lib.QParams(3, -200, 7, 0.0, scale, None), 0) == EUNSUPPORTED
    empty = _lib.Layout(1, 1, 0, 0)
    assert h.dlmcq_codes_forward(None, None, ctypes.byref(empty), ctypes.byref(act), 0, None) == 0


def test_code_gemm_prepare_refuses_inexact_accumulation(libpath):
    """dlmcq_qgemm_prepare / dlmcq_qconv_prepare refuse a K whose partial sums can leave the accumulator's exact range:
    K * max|a| * max|w| above 2^24 for e4m3 (fp32 accumulators), above 2^31 - 1 for the integer kind (s32) - before
    any CUDA call.  (The accepted side of each bound runs on the GPU: tests/qgemm_cases.py, tests/qconv_cases.py.)"""
    from dlmc_quant_b200 import _lib
    from dlmc_quant_b200 import qgemm as Q
    h = _lib.lib()
    EUNSUPPORTED = -5
    one = ctypes.c_void_p(4096)
    qp = lambda form, lo, hi: _lib.QParams(form, lo, hi, 0.0, one, one if form != 3 else None)  # noqa: E731
    gemm = lambda k, enc, act, wt: h.dlmcq_qgemm_prepare(one, 8, k, enc, ctypes.byref(act), ctypes.byref(wt), 8, None,  # noqa: E731
                                                          one, one, None)

    def conv(kh, kw, cin, enc, act, wt):
        g = Q._geom(1, 1, 1, cin, 8, kh, kw)
        return h.dlmcq_qconv_prepare(one, ctypes.byref(g), enc, ctypes.byref(act), ctypes.byref(wt), 8, None, one, one,
                                     None)
    e4_a, e4_w = qp(1, 0, 16), qp(3, -16, 16)
    assert 65536 * 16 * 16 == 2 ** 24
    assert gemm(65552, 1, e4_a, e4_w) == EUNSUPPORTED
    assert gemm(2 ** 20, 1, qp(2, 0, 15), qp(3, -8, 7)) == EUNSUPPORTED              # 2^20 * 15 * 8 > 2^24
    assert gemm(139824, 1, qp(1, 0, 15), qp(3, -8, 7)) == EUNSUPPORTED               # 4-bit codes: K <= 139810
    assert gemm(66320, 0, qp(2, 0, 255), qp(3, -127, 127)) == EUNSUPPORTED           # 8-bit codes: K <= 66311
    assert gemm(2 ** 40, 0, qp(2, 0, 15), qp(3, -7, 7)) == EUNSUPPORTED
    assert gemm(132112, 0, qp(3, -127, 127), qp(3, -128, 127)) == EUNSUPPORTED       # max|w| = 128, not 127
    assert conv(3, 3, 7296, 1, e4_a, e4_w) == EUNSUPPORTED                           # K = 65664 > 2^16
    assert conv(1, 1, 65600, 1, e4_a, e4_w) == EUNSUPPORTED
    assert conv(3, 3, 7424, 0, qp(2, 0, 255), qp(3, -127, 127)) == EUNSUPPORTED       # K = 66816
    assert conv(7, 7, 1408, 0, qp(2, 0, 255), qp(3, -127, 127)) == EUNSUPPORTED       # K = 68992
    # the Python mirror of the bound, at its edges
    assert Q.accumulator_exact(Q.QGEMM_E4M3, 65536, 0, 16, -16, 16)
    assert not Q.accumulator_exact(Q.QGEMM_E4M3, 65537, 0, 16, -16, 16)
    assert Q.accumulator_exact(Q.QGEMM_I8, 66311, 0, 255, -127, 127)
    assert not Q.accumulator_exact(Q.QGEMM_I8, 66312, 0, 255, -127, 127)
    assert Q.accumulator_exact(Q.QGEMM_I8, 131071, -128, 127, -128, 127)
    assert not Q.accumulator_exact(Q.QGEMM_I8, 131073, -128, 127, -128, 127)


def test_code_gemm_encoding_follows_the_accumulator_bound():
    """enable_code_gemm picks e4m3 only while K * max|a| * max|w| <= 2^24, the integer kind while it is <= 2^31 - 1,
    and leaves a layer on its original path when neither accumulates its K exactly; a layer switched to an explicit
    encoding that cannot hold its K keeps its original path too."""
    import copy
    import torch
    from dlmc_quant_b200 import quantize_model
    from dlmc_quant_b200.qgemm import QGEMM_E4M3, QGEMM_I8, enable_code_gemm
    nn = torch.nn

    def quantised(bits, *layers):
        net = nn.Sequential(*layers)
        cfg = {"weight": {"enable": True, "type": "minmax_channel", "args": {"n_bits": bits, "signed": True, "ch_axis": 0}},
               "input": {"enable": True, "type": "minmax_tensor", "args": {"n_bits": bits, "signed": False}},
               "exclude_layers": [], "override_options": [], "momentum": 0.1}
        quantize_model(net, copy.deepcopy(cfg), None)
        return net
    # 4-bit codes: max|a| = 15, max|w| = 7 -> e4m3 up to K = 159783
    net4 = quantised(4, nn.Linear(159776, 1), nn.Linear(159792, 1), nn.Conv2d(17792, 1, 3, padding=1))
    assert (net4[0].in_min_val, net4[0].in_max_val, net4[0].wt_min_val, net4[0].wt_max_val) == (0, 15, -7, 7)
    assert enable_code_gemm(net4, convolutions=True) == ["0", "1", "2"]
    assert [net4[i].__dict__["_code_gemm"].encoding for i in range(3)] == [QGEMM_E4M3, QGEMM_I8, QGEMM_I8]
    # 8-bit codes: max|a| = 255, max|w| = 127 -> the integer kind up to K = 66311, then no exact encoding
    net8 = quantised(8, nn.Linear(66304, 1), nn.Linear(66320, 1), nn.Conv2d(7424, 1, 3, padding=1))
    assert (net8[0].in_min_val, net8[0].in_max_val, net8[0].wt_min_val, net8[0].wt_max_val) == (0, 255, -127, 127)
    assert enable_code_gemm(net8, convolutions=True) == ["0"]
    assert net8[0].__dict__["_code_gemm"].encoding == QGEMM_I8
    assert all("_code_gemm" not in net8[i].__dict__ and "forward" not in net8[i].__dict__ for i in (1, 2))
    # explicit encodings: the state refuses what the prepare entry would refuse, so the layer keeps its path
    for net, enc in ((quantised(4, nn.Linear(159792, 1)), QGEMM_E4M3), (quantised(8, nn.Linear(66320, 1)), QGEMM_I8)):
        assert enable_code_gemm(net, enc) == ["0"]
        st = net[0].__dict__["_code_gemm"]
        assert st.refresh(net[0], net[0].__dict__["_code_gemm_forms"]) is False and st.usable is False


def test_code_gemm_module_switch_is_host_logic():
    """enable_code_gemm / disable_code_gemm: which layers qualify (Linear with K % 16 == 0, stride-1 1x1 Conv2d) and
    that switching is reversible - no device needed."""
    import copy
    import torch
    from dlmc_quant_b200 import quantize_model
    from dlmc_quant_b200.qgemm import disable_code_gemm, enable_code_gemm
    nn = torch.nn
    net = nn.Sequential(nn.Conv2d(16, 32, 1), nn.Conv2d(32, 32, 3, padding=1), nn.Conv2d(32, 64, 1, stride=2),
                        nn.Conv2d(64, 64, 1, groups=2), nn.Conv2d(64, 48, 1, bias=False), nn.Flatten(),
                        nn.Linear(48, 10), nn.Linear(10, 4))
    cfg = {"weight": {"enable": True, "type": "minmax_channel", "args": {"n_bits": 4, "signed": True, "ch_axis": 0}},
           "input": {"enable": True, "type": "minmax_tensor", "args": {"n_bits": 4, "signed": False}},
           "exclude_layers": [], "override_options": [], "momentum": 0.1}
    quantize_model(net, copy.deepcopy(cfg), None)
    stock = {n: m.forward.__func__ for n, m in net.named_modules() if hasattr(m, "qconfig")}
    assert enable_code_gemm(net) == ["0", "4", "6"]          # 3x3, strided, grouped convs and K = 10 keep the library path
    assert enable_code_gemm(net) == []                       # idempotent
    assert net[0].__dict__["_code_gemm"].encoding == 1       # 4-bit codes: e4m3 operands
    disable_code_gemm(net)
    assert all("_code_gemm" not in m.__dict__ and "forward" not in m.__dict__ for m in net.modules())
    assert {n: m.forward.__func__ for n, m in net.named_modules() if hasattr(m, "qconfig")} == stock
    net8 = nn.Sequential(nn.Linear(32, 8))
    cfg8 = copy.deepcopy(cfg)
    cfg8["weight"]["args"]["n_bits"] = cfg8["input"]["args"]["n_bits"] = 8
    quantize_model(net8, cfg8, None)
    enable_code_gemm(net8)
    assert net8[0].__dict__["_code_gemm"].encoding == 0      # 8-bit codes need the integer kind


def test_product_path_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from dlmc_quant_b200 import functional as F
    from dlmc_quant_b200._lib import DlmcqError
    with pytest.raises(DlmcqError):
        F.fq_forward(torch.zeros(8), torch.ones(1), None, 0, 15, 1)


def test_product_never_imports_oracle():
    """The oracle is test infrastructure: nothing under dlmc_quant_b200/ may reference it."""
    pkg = os.path.join(ROOT, "dlmc_quant_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.replace("no oracle", ""), f"{f} mentions the oracle"
