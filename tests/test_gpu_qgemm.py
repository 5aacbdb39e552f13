"""GPU parity tests of the integer-code layer product (SURVEY.md 8f row f2, consumer side): csrc/qgemm_kernels.cu
through the C ABI (dlmcq_codes_forward / dlmcq_qgemm_prepare / dlmcq_qgemm) and the module switch
dlmc_quant_b200.qgemm.enable_code_gemm.

The cases live in tests/qgemm_cases.py and run in a child process: the GEMM is a TMA + tcgen05 pipeline whose failure
mode is a trap (watchdog) that poisons the CUDA context - it must not take the rest of this suite with it.

Bars: the code bytes equal dlmcq_fq_forward's codes BIT FOR BIT; the GEMM equals oracle/restate.py::code_gemm (exact
integer dot product, then the two documented fp32 roundings) BIT FOR BIT for both operand encodings; against the
reference expression itself (product of the two fake-quantised tensors, float64) the relative error is <= 1e-5."""
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
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "qgemm_cases.py")], capture_output=True, text=True,
                       timeout=600, env=env, cwd=ROOT)
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert lines, f"case runner produced no report (rc {p.returncode}):\n{p.stdout[-2000:]}\n{p.stderr[-4000:]}"
    return json.loads(lines[-1])


def _failed(report, prefix):
    return {k: v.get("error") for k, v in report["cases"].items() if k.startswith(prefix) and not v["ok"]}


def test_case_runner_covered_every_family(report):
    names = list(report["cases"])
    for prefix in ("raw_i8_", "raw_e4m3_", "pipe_i8_", "pipe_e4m3_", "module_", "errors"):
        assert any(n.startswith(prefix) for n in names), prefix
    assert len(names) >= 40


def test_integer_kind_gemm_is_bit_exact(report):
    """tcgen05.mma kind::i8 (u8|s8 x s8 -> s32): full / ragged M, N, K tiles, K < one swizzle atom, 4-bit and 8-bit
    codes, signed activations, ReLU and bf16 epilogues."""
    assert not _failed(report, "raw_i8_"), _failed(report, "raw_i8_")


def test_e4m3_kind_gemm_is_bit_exact(report):
    """tcgen05.mma kind::f8f6f4 on e4m3-encoded codes, fp32 accumulators."""
    assert not _failed(report, "raw_e4m3_"), _failed(report, "raw_e4m3_")


def test_worst_case_accumulators_are_exact(report):
    """Saturated, one-sign biased and cancelling codes at the ResNet-50 3x3 layers' K on both kinds, at K = 65520
    with |code| = 16 on e4m3 (partial sums up to 2^24) and at K = 66304 with 8-bit codes on the integer kind (up to
    2^31 - 1): bit-exact, and each case reached the magnitude it was built for."""
    acc = {k: v for k, v in report["cases"].items() if k.startswith("acc_")}
    assert len(acc) == 36, sorted(acc)
    assert not _failed(report, "acc_"), _failed(report, "acc_")
    for name, c in acc.items():
        assert c["peak_abs_partial_sum"] >= c["max_abs_acc"] > 0, (name, c)
        if "saturated" in name:
            hi_a, hi_w = (255, 127) if "8bit" in name else (16, 16) if "k65520" in name else (15, 7)
            assert c["max_abs_acc"] == c["K"] * hi_a * hi_w, (name, c)
    assert acc["acc_e4m3_saturated_k65520"]["max_abs_acc"] > 2 ** 24 - 2 ** 13
    assert acc["acc_i8_8bit_saturated_k66304"]["max_abs_acc"] > 2 ** 31 - 2 ** 19
    assert acc["acc_e4m3_biased_k65520"]["peak_abs_partial_sum"] > 2 ** 23


def test_codes_prepare_gemm_pipeline(report):
    """x, w -> code bytes (== the fake-quant kernels' codes) -> alpha / beta from device qparams -> GEMM: bit-exact
    against the integer oracle, <= 1e-5 relative against the reference product in float64, for the AFFINE, ZP, A1
    and SYM activation forms with per-channel / per-tensor AFFINE and SYM weights."""
    assert not _failed(report, "pipe_"), _failed(report, "pipe_")


def test_module_switch_and_argument_errors(report):
    """enable_code_gemm on quantize_model'd Linear / 1x1 Conv2d layers (QBase 4-bit, FSPTQ 8-bit; channels-last and
    NCHW inputs): eval output equals the fake-quant + library path to 2e-5 of the output's magnitude; autograd calls
    keep the differentiable path; bad shapes are refused loudly."""
    bad = {**_failed(report, "module_"), **_failed(report, "errors")}
    assert not bad, bad
