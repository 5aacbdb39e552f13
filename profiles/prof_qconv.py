"""The convolution on the integer codes (csrc/qgemm_kernels.cu qconv_kernel: TMA im2col -> tcgen05.mma -> TMEM,
implicit GEMM over channels-last one-byte codes) on the ResNet-50 layers `enable_code_gemm(convolutions=True)` adds -
its 16 3x3 convolutions (three of them stride 2) and its three stride-2 1x1 downsample convolutions - at batch 128,
channels-last, W4A4 codes, beside the library path the reference takes (cuDNN on the fake-quantised fp32 tensor, TF32
as torch enables by default, and strict fp32).  Then whole-model ResNet-50 W4A4 eval images/s for four arms.

Per layer shape (count = how many of ResNet-50's layers have it): CUDA-event time of 20 calls after 5 warm-ups;
algorithmic bytes  qconv: B*H*W*Cin (codes) + n*K (weight codes) + B*Ho*Wo*n*4 (fp32 out; bf16: *2), K = kh*kw*Cin;
cuDNN: the same with 4-byte activations and weights; qconv bytes / time against the copy peak measured in this run
(device-to-device copy of 2 GiB: read + write bytes / time).  Working sets below 100 MB are flagged `l2_resident`
(L2 is 126 MB).  `codes_us` is the separate x -> code pass.  Full-size check: qconv (activation offset != 0, so the
border rule is live) vs strict-fp32 cuDNN on the dequantised tensors within 1e-5 of conv2d(|y_a|, |y_w|).

    python profiles/prof_qconv.py [batch] > profiles/r03_prof_qconv.jsonl"""
import copy
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as TF

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from dlmc_quant_b200 import qgemm as Q  # noqa: E402

# (H = W of the input, Cin, Cout, k, stride, padding, count) of torchvision ResNet-50's layers the convolution kernel
# serves; batch 128
SHAPES = [(56, 64, 64, 3, 1, 1, 3), (56, 128, 128, 3, 2, 1, 1), (28, 128, 128, 3, 1, 1, 3), (28, 256, 256, 3, 2, 1, 1),
          (14, 256, 256, 3, 1, 1, 5), (14, 512, 512, 3, 2, 1, 1), (7, 512, 512, 3, 1, 1, 2),
          (56, 256, 512, 1, 2, 0, 1), (28, 512, 1024, 1, 2, 0, 1), (14, 1024, 2048, 1, 2, 0, 1)]


def timeit(fn, iters=20, warm=5):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / iters * 1e3      # us


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else "unknown"


def copy_peak_gbs():
    a = torch.empty(1 << 31, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    us = timeit(lambda: b.copy_(a), 10, 3)
    del a, b
    return 2 * (1 << 31) / us * 1e-3


def run_layer(batch, hw, cin, cout, k, stride, pad, peak):
    dev = torch.device("cuda")
    g = torch.Generator(device="cuda").manual_seed(hw * 1000 + cin + k)
    ho = (hw + 2 * pad - k) // stride + 1
    ca = torch.randint(0, 16, (batch, hw, hw, cin), device=dev, generator=g, dtype=torch.uint8)
    cw = torch.randint(-7, 8, (cout, k, k, cin), device=dev, generator=g, dtype=torch.int8)
    s_a, o_a = 0.11, 0.05
    s_w = torch.rand(cout, device=dev, generator=g) * 0.01 + 0.002
    act = (torch.tensor([s_a], device=dev), torch.tensor([o_a], device=dev), 0, 15, 0, 0.0)     # A1: y = c*s + o
    alpha, beta = Q.qconv_prepare(cw.view(torch.uint8), act, (s_w, -7, 7, 3, 0.0))
    wb = cw.view(torch.uint8)
    out32 = torch.empty(batch, ho, ho, cout, device=dev)
    out16 = torch.empty(batch, ho, ho, cout, device=dev, dtype=torch.bfloat16)
    kw = dict(stride=stride, padding=pad)
    m, kk = batch * ho * ho, k * k * cin
    rec = {"layer": f"{k}x{k}/s{stride} {cin}->{cout} @{hw}x{hw}", "m": m, "k": kk, "n": cout}
    rec["qconv_f32_us"] = timeit(lambda: Q.qconv(ca, wb, alpha, beta, out=out32, **kw))
    rec["qconv_bf16_us"] = timeit(lambda: Q.qconv(ca, wb, alpha, beta, out=out16, out_dtype=torch.bfloat16, **kw))
    a_bytes = batch * hw * hw * cin
    by32, by16 = a_bytes + cout * kk + m * cout * 4, a_bytes + cout * kk + m * cout * 2
    rec["qconv_bytes_f32"] = by32
    rec["qconv_f32_gbs"] = by32 / rec["qconv_f32_us"] * 1e-3
    rec["qconv_bf16_gbs"] = by16 / rec["qconv_bf16_us"] * 1e-3
    rec["qconv_f32_frac_of_copy_peak"] = rec["qconv_f32_gbs"] / peak
    rec["qconv_bf16_frac_of_copy_peak"] = rec["qconv_bf16_gbs"] / peak
    rec["tops"] = 2.0 * m * cout * kk / rec["qconv_f32_us"] * 1e-6
    rec["l2_resident"] = by32 < 100e6
    x = (ca.float() * s_a + o_a).permute(0, 3, 1, 2)                  # NCHW view of channels-last fp32 storage
    w = (cw.float() * s_w[:, None, None, None]).permute(0, 3, 1, 2)  # channels-last weight
    torch.backends.cudnn.allow_tf32 = True
    rec["cudnn_tf32_us"] = timeit(lambda: TF.conv2d(x, w, **kw))
    torch.backends.cudnn.allow_tf32 = False
    rec["cudnn_fp32_us"] = timeit(lambda: TF.conv2d(x, w, **kw))
    rec["cudnn_bytes"] = a_bytes * 4 + cout * kk * 4 + m * cout * 4
    rec["speedup_vs_cudnn_tf32"] = rec["cudnn_tf32_us"] / rec["qconv_f32_us"]
    xs = x.contiguous(memory_format=torch.channels_last)
    sc, of = torch.tensor([s_a], device=dev), torch.tensor([o_a], device=dev)
    rec["codes_us"] = timeit(lambda: Q.codes_forward(xs, sc, of, 0, 15, 0))
    ref = TF.conv2d(x, w, **kw)
    mag = TF.conv2d(x.abs(), w.abs(), **kw)
    torch.backends.cudnn.allow_tf32 = True
    got = Q.qconv(ca, wb, alpha, beta, **kw).permute(0, 3, 1, 2)
    rec["max_err_over_bound"] = float(((got - ref).abs() / mag.clamp_min(1e-30)).max())
    rec["property_ok"] = rec["max_err_over_bound"] <= 1e-5
    return rec


def whole_model(batch, steps=20):
    import torchvision
    from dlmc_quant_b200 import quantize_model
    from dlmc_quant_b200.qgemm import enable_code_gemm
    cfg = {"weight": {"enable": True, "type": "minmax_channel", "args": {"n_bits": 4, "signed": True, "ch_axis": 0}},
           "input": {"enable": True, "type": "minmax_tensor", "args": {"n_bits": 4, "signed": False}},
           "exclude_layers": [], "override_options": [], "momentum": 0.1}
    x = torch.randn(batch, 3, 224, 224, device="cuda").contiguous(memory_format=torch.channels_last)
    res = {"model": f"torchvision resnet50 W4A4 (QBase, minmax observers), eval / no_grad, channels_last, batch {batch}, "
                    "fp32 tensors, cuDNN TF32 (torch default)", "timing": f"CUDA events, {steps} forwards after 3 warm-ups"}
    for arm in ("fp32", "quantize_model", "code_gemm_pointwise", "code_gemm_convolutions"):
        torch.manual_seed(2333)
        model = torchvision.models.resnet50().cuda().to(memory_format=torch.channels_last)
        if arm != "fp32":
            quantize_model(model, copy.deepcopy(cfg), None)
        model.eval()
        with torch.no_grad():
            model(x[:8])
            switched = None
            if arm.startswith("code_gemm"):
                switched = len(enable_code_gemm(model, convolutions=arm.endswith("convolutions")))
            for _ in range(3):
                model(x)
            torch.cuda.synchronize()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(steps):
                model(x)
            t1.record()
            torch.cuda.synchronize()
        ms = t0.elapsed_time(t1) / steps
        res[arm] = {"images_per_s": round(batch / ms * 1e3, 1), "ms_per_forward": round(ms, 3)}
        if switched is not None:
            res[arm]["layers_switched"] = switched
            res[arm]["layers_that_used_it"] = sum(1 for m_ in model.modules()
                                                  if getattr(m_.__dict__.get("_code_gemm"), "usable", False))
        del model
        torch.cuda.empty_cache()
    return res


def main():
    batch = int(sys.argv[1]) if len(sys.argv) > 1 else 128
    peak = copy_peak_gbs()
    print(json.dumps({"device": torch.cuda.get_device_name(0), "card": card(), "copy_peak_gbs": round(peak, 1),
                      "batch": batch}), flush=True)
    for hw, cin, cout, k, stride, pad, count in SHAPES:
        try:
            rec = run_layer(batch, hw, cin, cout, k, stride, pad, peak)
            rec["count"] = count
        except Exception as e:  # noqa: BLE001
            rec = {"shape": [hw, cin, cout, k, stride], "error": f"{type(e).__name__}: {e}"[:300]}
        print(json.dumps({k_: (round(v, 4) if isinstance(v, float) else v) for k_, v in rec.items()}), flush=True)
        torch.cuda.empty_cache()
    try:
        print(json.dumps({"whole_model": whole_model(batch)}), flush=True)
    except Exception as e:  # noqa: BLE001
        print(json.dumps({"whole_model": "error", "error": f"{type(e).__name__}: {e}"[:300]}), flush=True)


if __name__ == "__main__":
    main()
