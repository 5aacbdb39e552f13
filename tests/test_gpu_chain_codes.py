"""GPU tests of the chained code layer: dlmcq_qgemm_codes / dlmcq_qconv_codes (csrc/qgemm_kernels.cu, the code GEMM
epilogue running eval BatchNorm -> ReLU -> the next layer's input quantizer) and its wiring (fuse.chain_spec,
qgemm.forward_codes with a tail).

The cases live in tests/chain_codes_cases.py and run in a child process: the kernel is a TMA + tcgen05 pipeline whose
failure mode is a trap that poisons the CUDA context - it must not take the rest of this suite with it.

Bars, byte for byte: the chained codes equal the two-kernel chain they replace (the layer output, then the fused
BatchNorm producer's codes) and, on a small subset, an independent restatement; whole models give the same logits with
the chain on and off."""
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
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "chain_codes_cases.py")], capture_output=True,
                       text=True, timeout=1800, env=env, cwd=ROOT)
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert lines, f"case runner produced no report (rc {p.returncode}):\n{p.stdout[-2000:]}\n{p.stderr[-4000:]}"
    return json.loads(lines[-1])


def _failed(report, prefix):
    return {k: v.get("error") for k, v in report["cases"].items() if k.startswith(prefix) and not v["ok"]}


def test_case_runner_covered_every_family(report):
    names = list(report["cases"])
    for prefix in ("raw_r50_conv1_", "raw_r50_conv2_", "raw_gemm_ragged_", "raw_gemm_n144_", "raw_conv_n80_",
                   "raw_conv_c192_", "raw_generic_bn_", "raw_generic_tiny_scale_", "raw_generic_acc_bound_",
                   "restate_gemm", "restate_conv", "model_r50", "model_r18", "stack_conv_", "stack_linear_",
                   "fallback_consumer_per_channel", "fallback_linear_4d_batchnorm2d", "tail_refusals", "fallback_",
                   "toggles", "graph"):
        assert any(n.startswith(prefix) for n in names), prefix
    assert len(names) >= 100


def test_raw_entries_match_the_two_kernel_chain(report):
    """Every ResNet-50 batch-128 chained-site geometry (1x1 conv1 GEMMs, 3x3 conv2 convolutions at stride 1 and 2),
    I8 / E4M3 producers and consumers (also mixed), fp32 / bf16 layer outputs, ReLU on and off, unsigned 4- / 8-bit and
    signed 4-bit consumer ranges, ragged m, n = 80 / 144, padded borders, 64-channel chunks."""
    bad = {**_failed(report, "raw_r50_"), **_failed(report, "raw_gemm_"), **_failed(report, "raw_conv_")}
    assert not bad, bad


def test_raw_entries_generic_path(report):
    """BatchNorm constants outside the packed path's domain (gamma 0 / negative, running_var near 0 and huge, NaN mean,
    |beta| > 2^20), a consumer scale outside the fast-division domain, accumulators at the encodings' bounds."""
    assert not _failed(report, "raw_generic_"), _failed(report, "raw_generic_")


def test_independent_restatement_and_folding_control(report):
    bad = _failed(report, "restate_")
    assert not bad, bad
    assert all(report["cases"][k]["folded_codes_differ"] > 0 for k in ("restate_gemm", "restate_conv"))


def test_models_identical_with_the_chain_on_and_off(report):
    """ResNet-50 (32 chained sites; 53 -> 21 layer calls with an fp32 output; the fused BatchNorm code pass at the 15
    residual sites only; 0 chained with 1x1 layers only) and ResNet-18 (8 chained sites), W4A4 eval."""
    bad = _failed(report, "model_")
    assert not bad, bad
    r50 = report["cases"]["model_r50"]
    assert r50["chained"] == 32 and r50["layer_calls_plain_on"] == 21 and r50["layer_calls_plain_off"] == 53
    assert r50["bnq_codes_on"] == 15
    assert report["cases"]["model_r50_pointwise_only"]["chained"] == 0
    assert report["cases"]["model_r18"]["chained"] == 8


def test_sequential_stacks_fallbacks_toggles_and_graph(report):
    bad = {**_failed(report, "stack_"), **_failed(report, "fallback_"), **_failed(report, "toggles"),
           **_failed(report, "graph"), **_failed(report, "tail_refusals")}
    assert not bad, bad
