"""GPU parity tests of the layer product on the integer codes at ResNet-50 batch-128 sizes: every convolution
enable_code_gemm(convolutions=True) switches (dlmcq_qconv) and every stride-1 1x1 convolution (dlmcq_qgemm), both
operand encodings, fp32 and bf16 outputs; and a switched FSPTQ model given an empty batch.

The cases live in tests/qcode_resnet_cases.py and run in a child process (a wedged TMA / tcgen05 pipeline traps and
poisons the CUDA context).  Bars: bit-exact against tests/qconv_oracle.py::exact_conv (exact integer convolution on the
GPU, the kernels' two fp32 roundings); fp32 outputs within 1e-5 of conv2d(|y_a|, |y_w|) of the reference's F.conv2d of
the fake-quantised tensors in float64."""
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
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "qcode_resnet_cases.py")], capture_output=True,
                       text=True, timeout=900, env=env, cwd=ROOT)
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert lines, f"case runner produced no report (rc {p.returncode}):\n{p.stdout[-2000:]}\n{p.stderr[-4000:]}"
    return json.loads(lines[-1])


def _failed(report, prefix):
    return {k: v.get("error") for k, v in report["cases"].items() if k.startswith(prefix) and not v["ok"]}


def test_case_runner_covered_every_shape(report):
    names = list(report["cases"])
    assert sum(n.startswith("conv_") for n in names) == 10
    assert sum(n.startswith("pointwise_") for n in names) == 12
    assert "module_fsptq_empty_batch" in names


def test_resnet50_convolutions_at_batch_128_are_bit_exact(report):
    """3x3 stride 1 / 2 and strided 1x1 layers through dlmcq_qconv (up to 3136 M tiles, about 21 per persistent CTA)."""
    assert not _failed(report, "conv_"), _failed(report, "conv_")


def test_resnet50_pointwise_layers_at_batch_128_are_bit_exact(report):
    """The stride-1 1x1 layers through dlmcq_qgemm on the [B*H*W, Cin] matrix of the channels-last codes."""
    assert not _failed(report, "pointwise_"), _failed(report, "pointwise_")


def test_switched_layers_accept_an_empty_batch(report):
    assert not _failed(report, "module_"), _failed(report, "module_")
