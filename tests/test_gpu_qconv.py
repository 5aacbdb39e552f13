"""GPU parity tests of the convolution on the integer codes: csrc/qgemm_kernels.cu qconv_kernel (TMA im2col ->
tcgen05.mma -> TMEM, implicit GEMM over channels-last codes) through the C ABI (dlmcq_qconv_prepare / dlmcq_qconv) and
the module switch enable_code_gemm(model, convolutions=True).

The cases live in tests/qconv_cases.py and run in a child process (a wedged TMA / tcgen05 pipeline traps and poisons
the CUDA context).  Bars: bit-exact against tests/qconv_oracle.py::code_conv for both operand encodings; <= 1e-5 of
conv2d(|y_a|, |y_w|) against the reference's F.conv2d of the fake-quantised tensors in float64; module outputs within
2e-5 of the output's magnitude of the layer's own fake-quant + strict-fp32 cuDNN path."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def report():
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "qconv_cases.py")], capture_output=True, text=True,
                       timeout=900, env=env, cwd=ROOT)
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert lines, f"case runner produced no report (rc {p.returncode}):\n{p.stdout[-2000:]}\n{p.stderr[-4000:]}"
    return json.loads(lines[-1])


def _failed(report, prefix):
    return {k: v.get("error") for k, v in report["cases"].items() if k.startswith(prefix) and not v["ok"]}


def test_case_runner_covered_every_family(report):
    names = list(report["cases"])
    for prefix in ("raw_i8_", "raw_e4m3_", "pipe_i8_", "pipe_e4m3_", "module_", "fallback_", "errors"):
        assert any(n.startswith(prefix) for n in names), prefix
    assert len(names) >= 70


def test_integer_kind_conv_is_bit_exact(report):
    """kind::i8: every geometry, Cin 64 (64-byte swizzle) / 128 / 192 / 256, ragged pixels and n, scalar and bf16
    epilogues, ReLU, signed and 8-bit codes, tiles across image boundaries, more tiles than SMs."""
    assert not _failed(report, "raw_i8_"), _failed(report, "raw_i8_")


def test_e4m3_kind_conv_is_bit_exact(report):
    assert not _failed(report, "raw_e4m3_"), _failed(report, "raw_e4m3_")


def test_worst_case_accumulators_are_exact(report):
    """Saturated, one-sign biased and cancelling codes at the ResNet-50 3x3 layers' K on both kinds, at K = 65088
    with |code| = 16 on e4m3 and at K = 66240 with 8-bit codes on the integer kind: bit-exact, and each case reached
    the magnitude it was built for."""
    acc = {k: v for k, v in report["cases"].items() if k.startswith("acc_")}
    assert len(acc) == 30, sorted(acc)
    assert not _failed(report, "acc_"), _failed(report, "acc_")
    for name, c in acc.items():
        assert c["peak_abs_partial_sum"] >= c["max_abs_acc"] > 0, (name, c)
        if "saturated" in name:                                  # interior pixels see every tap
            hi_a, hi_w = (255, 127) if "8bit" in name else (16, 16) if "k65088" in name else (15, 7)
            assert c["max_abs_acc"] == c["K"] * hi_a * hi_w, (name, c)
    assert acc["acc_e4m3_saturated_k65088"]["max_abs_acc"] > 2 ** 24 - 2 ** 17
    assert acc["acc_i8_8bit_saturated_k66240"]["max_abs_acc"] > 2 ** 31 - 2 ** 22


def test_codes_prepare_conv_pipeline(report):
    """fp32 / bf16 x -> codes_forward -> qconv_prepare -> qconv: bit-exact vs the oracle, <= 1e-5 vs the reference."""
    assert not _failed(report, "pipe_"), _failed(report, "pipe_")


def test_module_switch(report):
    """QBase 4-bit and FSPTQ 8-bit 3x3 / strided layers, NCHW and channels-last inputs, ResNet-50 layer by layer,
    CUDA-graph capture; autograd keeps the differentiable path."""
    assert not _failed(report, "module_"), _failed(report, "module_")


def test_ineligible_layers_keep_their_path_and_errors(report):
    bad = {**_failed(report, "fallback_"), **_failed(report, "errors")}
    assert not bad, bad
