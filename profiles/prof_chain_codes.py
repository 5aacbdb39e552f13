"""Layer in codes, layer out codes at inference: the code GEMM / implicit-GEMM convolution writing the next layer's codes
from its epilogue (dlmcq_qgemm_codes / dlmcq_qconv_codes) against the two kernels it replaces, at every distinct
ResNet-50 batch-128 chained-site geometry (conv1 -> bn1 -> relu -> conv2, conv2 -> bn2 -> relu -> conv3), channels-last,
I8 operands, fp32 layer output; then whole-model ResNet-50 W4A4 eval images/s with fuse_bn_act_quant +
enable_code_gemm(convolutions=True), the chain on and off (fuse.chain_spec patched out), alternated in one run.

Per site, CUDA-event time of 20 calls after 5 warm-ups (profiles/prof_qconv.py timeit) of
  two_kernel_us : qgemm / qconv with an fp32 output + dlmcq_bnq_forward_codes (eval prepare + apply);
  chained_us    : the chained entry.
Algorithmic bytes: two-kernel m*K + n*K + 9*m*n (fp32 out written and read, codes written), chained m*K + n*K + m*n
(K = kh*kw*Cin; the im2col re-reads of the convolution are not counted); the chained rate against the
device-to-device copy peak measured in the same run.

    python profiles/prof_chain_codes.py > profiles/r03_prof_chain_codes.jsonl"""
import copy
import ctypes as C
import json
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
from prof_qconv import card, copy_peak_gbs, timeit  # noqa: E402

from dlmc_quant_b200 import _lib  # noqa: E402
from dlmc_quant_b200 import functional as F  # noqa: E402
from dlmc_quant_b200 import qgemm as Q  # noqa: E402
from dlmc_quant_b200.fuse import _bnq_ws  # noqa: E402

BATCH = 128
CFG = {"weight": {"enable": True, "type": "minmax_channel", "args": {"n_bits": 4, "signed": True, "ch_axis": 0}},
       "input": {"enable": True, "type": "minmax_tensor", "args": {"n_bits": 4, "signed": False}},
       "exclude_layers": [], "override_options": [], "momentum": 0.1}
# (name, input hw, cin, n, kernel, stride): conv1 1x1 (GEMM) and conv2 3x3 pad 1 sites
SITES = [("conv1", 56, 64, 64, 1, 1), ("conv1", 56, 256, 64, 1, 1), ("conv1", 56, 256, 128, 1, 1),
         ("conv1", 28, 512, 128, 1, 1), ("conv1", 28, 512, 256, 1, 1), ("conv1", 14, 1024, 256, 1, 1),
         ("conv1", 14, 1024, 512, 1, 1), ("conv1", 7, 2048, 512, 1, 1),
         ("conv2", 56, 64, 64, 3, 1), ("conv2", 56, 128, 128, 3, 2), ("conv2", 28, 128, 128, 3, 1),
         ("conv2", 28, 256, 256, 3, 2), ("conv2", 14, 256, 256, 3, 1), ("conv2", 14, 512, 512, 3, 2),
         ("conv2", 7, 512, 512, 3, 1)]


def run_site(name, hw, cin, n, k, stride, peak):
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(0)
    a = torch.randint(0, 16, (BATCH, hw, hw, cin), generator=g, device=dev).to(torch.uint8)
    w = (torch.randint(-7, 8, (n, k, k, cin), generator=g, device=dev) & 0xFF).to(torch.uint8)
    alpha = torch.rand(n, generator=g, device=dev) * 0.02 + 0.005
    gamma, bbeta = torch.rand(n, generator=g, device=dev) + 0.5, torch.randn(n, generator=g, device=dev) * 0.3
    rmean, rvar = torch.randn(n, generator=g, device=dev) * 0.2, torch.rand(n, generator=g, device=dev) + 0.5
    scale, offset = torch.tensor([2.5 / 15], device=dev), torch.tensor([0.07], device=dev)
    if k == 1:
        a2, w2 = a.view(-1, cin), w.view(n, cin)
        beta = torch.randn(n, generator=g, device=dev)
        layer = lambda: Q.qgemm(a2, w2, alpha, beta)                                       # noqa: E731
        y = layer()
    else:
        beta = torch.randn(16 ** 2, n, generator=g, device=dev)
        layer = lambda: Q.qconv(a, w, alpha, beta, stride, 1)                              # noqa: E731
        y = layer()
    m = y.numel() // n
    gq = 1 / math.sqrt(y.numel() * 15)
    desc = _lib.BnqDesc(m, n, _lib.F32, _lib.BNQ_RELU, 1e-5, 0.1)
    qp = _lib.QParams(_lib.FORM_AFFINE, 0, 15, gq, scale.data_ptr(), offset.data_ptr())
    st = torch.empty(2, n, device=dev)
    codes = torch.empty(m, n, dtype=torch.uint8, device=dev)
    ws, nws = _bnq_ws(dev, desc)

    def two_kernel():
        yy = layer()
        _lib.check(_lib.lib().dlmcq_bnq_forward_codes(
            F._ptr(yy), None, F._ptr(gamma), F._ptr(bbeta), F._ptr(rmean), F._ptr(rvar), st.data_ptr(),
            st.data_ptr() + 4 * n, None, F._ptr(codes), C.byref(desc), C.byref(qp), 0, F._ptr(ws), nws,
            F._stream_ptr()))
    t = Q.bnq_tail(rmean, rvar, scale, offset, 0, 15, gq, gamma, bbeta, 1e-5, True, torch.float32, 0)
    if k == 1:
        chained = lambda: Q.qgemm_codes(a2, w2, alpha, beta, t)                            # noqa: E731
    else:
        chained = lambda: Q.qconv_codes(a, w, alpha, beta, t, stride, 1)                   # noqa: E731
    two_kernel()
    same = bool(torch.equal(chained().view(-1, n), codes))
    us_two, us_chain = timeit(two_kernel), timeit(chained)
    kk = k * k * cin
    b_two, b_chain = m * kk + n * kk + 9 * m * n, m * kk + n * kk + m * n
    return {"site": name, "hw": hw, "cin": cin, "n": n, "k": k, "stride": stride, "m": m, "identical": same,
            "two_kernel_us": us_two, "chained_us": us_chain, "speedup": us_two / us_chain,
            "two_kernel_bytes": b_two, "chained_bytes": b_chain,
            "chained_gbs": b_chain / us_chain * 1e-3, "chained_of_copy_peak": b_chain / us_chain * 1e-3 / peak}


def whole_model(batch, rounds=3, steps=20):
    import torchvision
    from dlmc_quant_b200 import fuse, quantize_model
    torch.manual_seed(2333)
    x = torch.randn(batch, 3, 224, 224, device="cuda").contiguous(memory_format=torch.channels_last)
    model = torchvision.models.resnet50().cuda().to(memory_format=torch.channels_last)
    quantize_model(model, copy.deepcopy(CFG), None)
    model.eval()
    orig = fuse.chain_spec
    arms = {"chain_on": orig, "chain_off": lambda *a, **k: None}
    times = {a: [] for a in arms}
    with torch.no_grad():
        model(x[:8])
        fuse.fuse_bn_act_quant(model)
        Q.enable_code_gemm(model, convolutions=True)
        try:
            for arm, fn in arms.items():
                fuse.chain_spec = fn
                for _ in range(3):
                    model(x)
            ref, same = None, True
            for _ in range(rounds):
                for arm, fn in arms.items():                       # alternated: on, off, on, off, ...
                    fuse.chain_spec = fn
                    torch.cuda.synchronize()
                    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    t0.record()
                    for _ in range(steps):
                        y = model(x)
                    t1.record()
                    torch.cuda.synchronize()
                    times[arm].append(t0.elapsed_time(t1) / steps)
                    ref = y if ref is None else ref
                    same = same and bool(torch.equal(ref, y))
        finally:
            fuse.chain_spec = orig
    res = {"logits_identical": same}
    for arm, ms in times.items():
        best = min(ms)
        res[arm] = {"images_per_s": round(batch / best * 1e3, 1), "ms_per_forward": [round(v, 3) for v in ms]}
    return res


def main():
    peak = copy_peak_gbs()
    print(json.dumps({"device": torch.cuda.get_device_name(0), "card": card(), "copy_peak_gbs": round(peak, 1),
                      "batch": BATCH}), flush=True)
    for site in SITES:
        try:
            rec = run_site(*site, peak)
        except Exception as e:  # noqa: BLE001
            rec = {"site": list(site), "error": f"{type(e).__name__}: {e}"[:300]}
        print(json.dumps({k: (round(v, 4) if isinstance(v, float) else v) for k, v in rec.items()}), flush=True)
        torch.cuda.empty_cache()
    try:
        print(json.dumps({"whole_model": whole_model(BATCH)}), flush=True)
    except Exception as e:  # noqa: BLE001
        print(json.dumps({"whole_model": "error", "error": f"{type(e).__name__}: {e}"[:300]}), flush=True)


if __name__ == "__main__":
    main()
