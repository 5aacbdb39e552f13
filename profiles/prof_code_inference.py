"""BatchNorm (+ identity) + ReLU + the next layer's activation codes at inference: the fused producer writing the codes
(dlmcq_bnq_forward_codes) against the two compositions it replaces, at the eight ResNet-50 batch-128 BatchNorm site
shapes, channels-last fp32; then whole-model ResNet-50 W4A4 eval images/s for four arms.

Per site, CUDA-event time of 20 calls after 5 warm-ups (profiles/prof_qconv.py timeit) of
  codes_us       : the codes pass (x [+ identity] -> codes [+ the plain a at residual sites]);
  fused_aq_us    : the fused fp32 a_q pass (dlmcq_bnq_forward) + codes_forward(a_q) - what the consumer did before;
  cudnn_us       : cuDNN batch_norm (+ identity add) + in-place ReLU + codes_forward.
Algorithmic bytes of the codes pass: rows*C*(4 [x] + 1 [codes]) plain, rows*C*(4 + 4 + 4 + 1) residual (x, identity,
a, codes); its rate against the device-to-device copy peak measured in the same run.  Every working set but the two
smallest is larger than the 126 MB L2.

    python profiles/prof_code_inference.py > profiles/r03_prof_code_inference.jsonl"""
import copy
import ctypes as C
import json
import math
import os
import sys

import torch
import torch.nn.functional as TF

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
from prof_qconv import card, copy_peak_gbs, timeit  # noqa: E402

from dlmc_quant_b200 import _lib  # noqa: E402
from dlmc_quant_b200 import functional as F  # noqa: E402
from dlmc_quant_b200 import qgemm as Q  # noqa: E402
from dlmc_quant_b200.fuse import _bnq_ws  # noqa: E402

BATCH = 128
SITES = [(56, 64), (56, 256), (28, 128), (28, 512), (14, 256), (14, 1024), (7, 512), (7, 2048)]   # (H = W, C)
CFG = {"weight": {"enable": True, "type": "minmax_channel", "args": {"n_bits": 4, "signed": True, "ch_axis": 0}},
       "input": {"enable": True, "type": "minmax_tensor", "args": {"n_bits": 4, "signed": False}},
       "exclude_layers": [], "override_options": [], "momentum": 0.1}


def run_site(hw, ch, resid, peak):
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(hw * 10000 + ch)
    rows = BATCH * hw * hw
    x = torch.randn(BATCH, ch, hw, hw, generator=g, device=dev).contiguous(memory_format=torch.channels_last)
    idn = torch.randn_like(x).contiguous(memory_format=torch.channels_last) if resid else None
    gamma, beta = torch.rand(ch, device=dev) + 0.5, torch.randn(ch, device=dev) * 0.3
    rmean, rvar = torch.randn(ch, device=dev) * 0.2, torch.rand(ch, device=dev) + 0.5
    scale, offset = torch.tensor([0.2], device=dev), torch.tensor([0.0], device=dev)
    lo, hi, enc = 0, 15, Q.QGEMM_E4M3
    gq = 1 / math.sqrt(x.numel() * hi)
    desc = _lib.BnqDesc(rows, ch, _lib.F32, _lib.BNQ_RELU | (_lib.BNQ_RESIDUAL if resid else 0), 1e-5, 0.1)
    qp = _lib.QParams(_lib.FORM_AFFINE, lo, hi, gq, scale.data_ptr(), offset.data_ptr())
    ws, nws = _bnq_ws(dev, desc)
    stats = torch.empty(2, ch, device=dev)
    a = torch.empty_like(x) if resid else None
    aq = torch.empty_like(x)
    codes = torch.empty_like(x, dtype=torch.uint8)
    h = _lib.lib()

    def codes_pass():
        _lib.check(h.dlmcq_bnq_forward_codes(F._ptr(x), F._ptr(idn), F._ptr(gamma), F._ptr(beta), F._ptr(rmean),
                                             F._ptr(rvar), stats.data_ptr(), stats.data_ptr() + 4 * ch, F._ptr(a),
                                             F._ptr(codes), C.byref(desc), C.byref(qp), enc, F._ptr(ws), nws,
                                             F._stream_ptr()))

    def fused_aq():
        _lib.check(h.dlmcq_bnq_forward(F._ptr(x), F._ptr(idn), F._ptr(gamma), F._ptr(beta), F._ptr(rmean),
                                       F._ptr(rvar), stats.data_ptr(), stats.data_ptr() + 4 * ch, F._ptr(a),
                                       F._ptr(aq), C.byref(desc), C.byref(qp), F._ptr(ws), nws, F._stream_ptr()))
        Q.codes_forward(aq, scale, offset, lo, hi, _lib.FORM_AFFINE, gq, encoding=enc)

    def cudnn():
        z = TF.batch_norm(x, rmean, rvar, gamma, beta, False, 0.1, 1e-5)
        if resid:
            z += idn
        z = torch.relu_(z)
        Q.codes_forward(z, scale, offset, lo, hi, _lib.FORM_AFFINE, gq, encoding=enc)

    rec = {"site": f"{'residual' if resid else 'plain'} {BATCH}x{hw}x{hw}x{ch}", "rows": rows, "C": ch}
    rec["codes_us"] = timeit(codes_pass)
    rec["fused_aq_us"] = timeit(fused_aq)
    rec["cudnn_us"] = timeit(cudnn)
    n = rows * ch
    rec["codes_bytes"] = n * (4 + 4 + 4 + 1 if resid else 4 + 1)
    rec["codes_gbs"] = rec["codes_bytes"] / rec["codes_us"] * 1e-3
    rec["codes_frac_of_copy_peak"] = rec["codes_gbs"] / peak
    rec["speedup_vs_fused_aq"] = rec["fused_aq_us"] / rec["codes_us"]
    rec["speedup_vs_cudnn"] = rec["cudnn_us"] / rec["codes_us"]
    return rec


def whole_model(batch, steps=20):
    import torchvision
    from dlmc_quant_b200 import fuse, quantize_model
    from dlmc_quant_b200.qgemm import enable_code_gemm
    x = torch.randn(batch, 3, 224, 224, device="cuda").contiguous(memory_format=torch.channels_last)
    res = {"model": f"torchvision resnet50 W4A4 (QBase, minmax observers), eval / no_grad, channels_last, batch {batch}, "
                    "fp32 tensors, cuDNN TF32 (torch default)", "timing": f"CUDA events, {steps} forwards after 3 warm-ups"}
    for arm in ("fp32", "quantize_model", "code_gemm_convolutions", "fuse_and_code_gemm_convolutions"):
        torch.manual_seed(2333)
        model = torchvision.models.resnet50().cuda().to(memory_format=torch.channels_last)
        if arm != "fp32":
            quantize_model(model, copy.deepcopy(CFG), None)
        model.eval()
        with torch.no_grad():
            model(x[:8])
            if arm.startswith("fuse"):
                fuse.fuse_bn_act_quant(model)
            if "code_gemm" in arm:
                enable_code_gemm(model, convolutions=True)
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
        del model
        torch.cuda.empty_cache()
    return res


def main():
    peak = copy_peak_gbs()
    print(json.dumps({"device": torch.cuda.get_device_name(0), "card": card(), "copy_peak_gbs": round(peak, 1),
                      "batch": BATCH}), flush=True)
    for hw, ch in SITES:
        for resid in (False, True):
            try:
                rec = run_site(hw, ch, resid, peak)
            except Exception as e:  # noqa: BLE001
                rec = {"site": [hw, ch, resid], "error": f"{type(e).__name__}: {e}"[:300]}
            print(json.dumps({k: (round(v, 4) if isinstance(v, float) else v) for k, v in rec.items()}), flush=True)
            torch.cuda.empty_cache()
    try:
        print(json.dumps({"whole_model": whole_model(BATCH)}), flush=True)
    except Exception as e:  # noqa: BLE001
        print(json.dumps({"whole_model": "error", "error": f"{type(e).__name__}: {e}"[:300]}), flush=True)


if __name__ == "__main__":
    main()
