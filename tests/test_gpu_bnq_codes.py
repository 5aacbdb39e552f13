"""GPU tests of the inference hand-off from the fused BatchNorm producer to the code GEMM: dlmcq_bnq_forward_codes
(csrc/bnq_kernels.cu) and its wiring (fuse.py: bn_act_into / bn_add_act, qgemm.py: code_input_spec / forward_codes).

The cases live in tests/bnq_codes_cases.py and run in a child process: the consumer side is a TMA + tcgen05 pipeline
whose failure mode is a trap that poisons the CUDA context - it must not take the rest of this suite with it.

Bars, all bit for bit: the codes equal dlmcq_codes_forward of the same call's plain output, and the plain output and
statistics equal dlmcq_bnq_forward's; whole models give the same logits whether the producer hands over codes or every
consumer quantises the fused plain output itself."""
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
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "bnq_codes_cases.py")], capture_output=True,
                       text=True, timeout=1200, env=env, cwd=ROOT)
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert lines, f"case runner produced no report (rc {p.returncode}):\n{p.stdout[-2000:]}\n{p.stderr[-4000:]}"
    return json.loads(lines[-1])


def _failed(report, prefix):
    return {k: v.get("error") for k, v in report["cases"].items() if k.startswith(prefix) and not v["ok"]}


def test_case_runner_covered_every_family(report):
    names = list(report["cases"])
    for prefix in ("raw_f32_", "raw_bf16_", "raw_r50_f32_", "raw_r50_bf16_", "raw_generic_values_",
                   "raw_generic_tiny_scale_", "model_r50_", "model_r18", "other_linear_", "fallback_unswitched",
                   "fallback_unusable", "fallback_train_autograd", "toggles", "graph"):
        assert any(n.startswith(prefix) for n in names), prefix
    assert len(names) >= 100


def test_raw_entry_codes_are_bit_identical(report):
    """fp32 / bf16, with and without residual and ReLU, I8 (4-bit and 8-bit unsigned, 4-bit signed) and E4M3 (4-bit
    unsigned, 5-bit signed), ragged row counts and every ResNet-50 batch-128 BatchNorm site shape."""
    assert not _failed(report, "raw_f32_"), _failed(report, "raw_f32_")
    assert not _failed(report, "raw_bf16_"), _failed(report, "raw_bf16_")
    assert not _failed(report, "raw_r50_"), _failed(report, "raw_r50_")


def test_raw_entry_generic_path(report):
    """NaN, +-inf, |x| > 2^20 in the input and a scale outside the fast-division domain."""
    assert not _failed(report, "raw_generic_"), _failed(report, "raw_generic_")


def test_resnet_logits_identical_and_codes_handed_over(report):
    """ResNet-50 W4A4 eval (auto encoding, forced I8, and 1x1 layers only) and ResNet-18: same logits as the consumers
    quantising the plain output; 47 sites (31 with 1x1 layers only) take codes from their producer and the stride-2
    downsample convolutions run on the code path."""
    bad = {**_failed(report, "model_")}
    assert not bad, bad
    r50 = report["cases"]["model_r50_convolutions"]
    assert r50["codes_from_producer"] == 47 and r50["layers_on_code_path"] == 53
    assert report["cases"]["model_r50_pointwise_only"]["codes_from_producer"] == 31


def test_batchnorm1d_linear_consumers(report):
    assert not _failed(report, "other_"), _failed(report, "other_")


def test_fallbacks_toggles_and_graph_capture(report):
    """Unswitched / unusable consumers, train mode and autograd hand over a_q as fuse alone does; switch order,
    disable_code_gemm, unfuse() and CUDA-graph replay change nothing."""
    bad = {**_failed(report, "fallback_"), **_failed(report, "toggles"), **_failed(report, "graph")}
    assert not bad, bad
