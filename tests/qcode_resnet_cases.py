"""Case runner for the layer product on the integer codes at ResNet-50 batch-128 sizes, executed in its OWN process by
tests/test_gpu_qcode_resnet.py for the same reason as tests/qgemm_cases.py: a wedged tcgen05 / TMA pipeline traps and a
trap poisons the CUDA context.  Prints one JSON report on the last line.

Every convolution enable_code_gemm(convolutions=True) switches (profiles/prof_qconv.py SHAPES: 3x3 stride 1 / 2 and
the strided 1x1 projections, through dlmcq_qconv) and every stride-1 1x1 convolution (bench.py R50_POINTWISE, through
dlmcq_qgemm on the [B*H*W, Cin] matrix), at batch 128: at these sizes a persistent CTA walks about 20 tiles and the TMEM
double buffer and the operand ring wrap their barrier phases many times.  Codes come from codes_forward on a
post-ReLU-like activation with a non-zero offset (A1 or AFFINE form: the border rule of beta is live) and per-channel
SYM weights.  Bars, for both operand encodings and fp32 / bf16 outputs:
  * bit-exact against tests/qconv_oracle.py::exact_conv (exact integer convolution as float64 matmuls per filter tap on
    the GPU, the kernels' two fp32 roundings);
  * fp32 output within 1e-5 of conv2d(|y_a|, |y_w|) (+ |bias|) of F.conv2d of the fake-quantised tensors in float64."""
import copy
import json
import os
import sys
import time
import traceback

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as TF  # noqa: E402

from oracle import restate as R  # noqa: E402
from tests.qconv_oracle import A1, AFFINE, SYM, conv_epilogue, exact_conv_acc, valid_tap_wsum  # noqa: E402

I8, E4M3 = 0, 1
BATCH = 128
# (H = W, Cin, Cout, k, stride, padding, layers of this shape in ResNet-50): profiles/prof_qconv.py SHAPES
CONV_SHAPES = [(56, 64, 64, 3, 1, 1, 3), (56, 128, 128, 3, 2, 1, 1), (28, 128, 128, 3, 1, 1, 3),
               (28, 256, 256, 3, 2, 1, 1), (14, 256, 256, 3, 1, 1, 5), (14, 512, 512, 3, 2, 1, 1),
               (7, 512, 512, 3, 1, 1, 2), (56, 256, 512, 1, 2, 0, 1), (28, 512, 1024, 1, 2, 0, 1),
               (14, 1024, 2048, 1, 2, 0, 1)]
# (H = W, Cin, Cout, layers): bench.py R50_POINTWISE, stride-1 1x1
POINTWISE_SHAPES = [(56, 64, 64, 1), (56, 64, 256, 4), (56, 256, 64, 2), (56, 256, 128, 1), (28, 128, 512, 4),
                    (28, 512, 128, 3), (28, 512, 256, 1), (14, 256, 1024, 6), (14, 1024, 256, 5), (14, 1024, 512, 1),
                    (7, 512, 2048, 3), (7, 2048, 512, 2)]


def _decode(code_bytes, encoding):
    if encoding == E4M3:
        return code_bytes.view(torch.float8_e4m3fn).float()
    return code_bytes.float()                                 # unsigned activation codes / callers view int8 weights


def case_layer(hw, cin, cout, k, stride, pad, a_form, seed):
    """One ResNet-50 layer at batch 128 on the code path, both encodings, fp32 and bf16 outputs."""
    from dlmc_quant_b200 import functional as F
    from dlmc_quant_b200 import qgemm as Q
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.relu(torch.randn(BATCH, cin, hw, hw, generator=g, device=dev)).contiguous(memory_format=torch.channels_last)
    w = (torch.randn(cout, k, k, cin, generator=g, device=dev) * 0.05).contiguous()     # [n, kh, kw, Cin]
    bias = torch.randn(cout, generator=g, device=dev)
    a_lo, a_hi, w_lo, w_hi = 0, 15, -7, 7
    s_a = (x.max() / a_hi * 0.9).reshape(1)
    off = torch.tensor([0.11 if a_form == AFFINE else 0.03], device=dev)
    s_w = w.abs().amax(dim=(1, 2, 3)) / w_hi + 1e-6
    g_a = R.lsq_g(x.numel(), a_hi) if a_form == AFFINE else 0.0
    m_a = R.grad_scale(s_a.cpu(), g_a).detach() if a_form == AFFINE else s_a.cpu()
    # the fake-quantised tensors and their codes (dlmcq_fq_forward: the reference chain, tests/test_gpu_fq.py)
    qa, ca = F.fq_forward(x, s_a, off, a_lo, a_hi, a_form, g_a, want_codes=True)
    qw, cw = F.fq_forward(w, s_w, None, w_lo, w_hi, SYM, 0.0, ch_axis=0, want_codes=True)
    cw_nchw, qw_nchw = cw.permute(0, 3, 1, 2), qw.permute(0, 3, 1, 2)
    conv = dict(stride=stride, padding=pad)
    acc = exact_conv_acc(ca, cw_nchw, **conv)
    want = conv_epilogue(acc, valid_tap_wsum(cw_nchw, hw, hw, **conv), m_a, off.cpu(), torch.zeros(1), s_w, bias)
    want = want.permute(0, 2, 3, 1)                                              # [B, Ho, Wo, n], contiguous storage
    ref = TF.conv2d(qa.double(), qw_nchw.double(), bias.double(), **conv).permute(0, 2, 3, 1)
    mag = TF.conv2d(qa.double().abs(), qw_nchw.double().abs(), bias.double().abs(), **conv).permute(0, 2, 3, 1)
    del qa, qw
    pointwise = k == 1 and stride == 1
    worst = 0.0
    for enc in (I8, E4M3):
        a_codes = Q.codes_forward(x, s_a, off, a_lo, a_hi, a_form, g_a, encoding=enc)
        w_codes = Q.codes_forward(w, s_w, None, w_lo, w_hi, SYM, 0.0, ch_axis=0, encoding=enc)
        assert torch.equal(_decode(a_codes, enc), ca), "activation code bytes differ from dlmcq_fq_forward's codes"
        wi = w_codes.view(torch.int8).float() if enc == I8 else _decode(w_codes, enc)
        assert torch.equal(wi, cw), "weight code bytes differ from dlmcq_fq_forward's codes"
        act = (s_a, off, a_lo, a_hi, a_form, g_a)
        wt = (s_w, w_lo, w_hi, SYM, 0.0)
        a_nhwc = a_codes.permute(0, 2, 3, 1)
        if pointwise:
            alpha, beta = Q.qgemm_prepare(w_codes.reshape(cout, cin), act, wt, bias, enc)
        else:
            alpha, beta = Q.qconv_prepare(w_codes, act, wt, bias, enc)
        for out_dtype in (torch.float32, torch.bfloat16):
            if pointwise:
                out = Q.qgemm(a_nhwc.reshape(-1, cin), w_codes.reshape(cout, cin), alpha, beta, out_dtype=out_dtype,
                              encoding=enc).view(BATCH, hw, hw, cout)
            else:
                out = Q.qconv(a_nhwc, w_codes, alpha, beta, out_dtype=out_dtype, encoding=enc, **conv)
            torch.cuda.synchronize()
            exp = want if out_dtype == torch.float32 else want.to(torch.bfloat16)
            if not torch.equal(out, exp):
                bad = out.float() != exp.float()
                idx = bad.nonzero()[0].tolist()
                raise AssertionError(f"encoding {enc} {out_dtype}: {int(bad.sum())} of {bad.numel()} differ from the "
                                     f"exact reference; first at {idx}: got {out[tuple(idx)].item()} "
                                     f"want {exp[tuple(idx)].item()}")
            if out_dtype == torch.float32:
                err = ((out.double() - ref).abs() / mag.clamp_min(1e-30)).max().item()
                assert err <= 1e-5, f"encoding {enc}: {err:.3e} of conv2d(|y_a|, |y_w|) vs the reference conv"
                worst = max(worst, err)
    return {"K": k * k * cin, "outputs": int(want.numel()), "max_abs_acc": int(acc.abs().max().item()),
            "rel_err_vs_reference_fp64": worst}


def case_empty_batch():
    """A switched FSPTQ 3x3 convolution (qconv) and 1x1 convolution (qgemm) given batch 0 return the empty
    [0, n, Ho, Wo] of their original path."""
    from dlmc_quant_b200 import quantize_model
    from dlmc_quant_b200.qgemm import enable_code_gemm
    torch.manual_seed(4)
    nn = torch.nn
    net = nn.Sequential(nn.Conv2d(64, 64, 3, stride=2, padding=1), nn.ReLU(), nn.Conv2d(64, 48, 1)).cuda()
    cfg = {"weight": {"enable": True, "type": "minmax_channel", "args": {"n_bits": 8, "signed": True, "ch_axis": 0}},
           "input": {"enable": True, "type": "minmax_tensor", "args": {"n_bits": 8, "signed": False}},
           "exclude_layers": [], "override_options": [], "momentum": 0.1}
    quantize_model(net, copy.deepcopy(cfg), None, quantization_type="FSPTQ")
    net = net.to(memory_format=torch.channels_last).eval()
    # post-ReLU input: the observer's minimum is 0, so the FSPTQ zero-point is an integer and the layer is served
    x = torch.relu(torch.randn(3, 64, 11, 9)).cuda().contiguous(memory_format=torch.channels_last)
    with torch.no_grad():
        net(x)
        want = net(x[:0])
        assert enable_code_gemm(net, convolutions=True) == ["0", "2"]
        full = net(x)
        assert all(net[i].__dict__["_code_gemm"].usable for i in (0, 2)), "a layer fell back to its original path"
        got = net(x[:0])
    torch.cuda.synchronize()
    assert tuple(want.shape) == (0, 48, 6, 5) and got.shape == want.shape and got.dtype == want.dtype
    assert full.shape == (3, 48, 6, 5)
    return {}


def build_cases():
    cases = []
    for i, (hw, cin, cout, k, stride, pad, _) in enumerate(CONV_SHAPES):
        form = AFFINE if i % 2 == 0 else A1
        cases.append((f"conv_{hw}x{hw}_{cin}to{cout}_{k}x{k}_stride{stride}", case_layer,
                      dict(hw=hw, cin=cin, cout=cout, k=k, stride=stride, pad=pad, a_form=form, seed=100 + i)))
    for i, (hw, cin, cout, _) in enumerate(POINTWISE_SHAPES):
        form = A1 if i % 2 == 0 else AFFINE
        cases.append((f"pointwise_{hw}x{hw}_{cin}to{cout}", case_layer,
                      dict(hw=hw, cin=cin, cout=cout, k=1, stride=1, pad=0, a_form=form, seed=200 + i)))
    cases.append(("module_fsptq_empty_batch", case_empty_batch, {}))
    return cases


def main(argv):
    only = argv[1] if len(argv) > 1 else ""
    report = {"cases": {}, "device": torch.cuda.get_device_name(0)}
    dead = False
    t_all = time.time()
    for name, fn, kw in build_cases():
        if only and only not in name:
            continue
        if dead:
            report["cases"][name] = {"ok": False, "error": "skipped: the CUDA context died in an earlier case"}
            continue
        t0 = time.time()
        try:
            extra = fn(**kw)
            torch.cuda.synchronize()
            report["cases"][name] = {"ok": True, "s": round(time.time() - t0, 3), **(extra or {})}
        except Exception as e:  # noqa: BLE001
            msg = f"{type(e).__name__}: {e}"
            report["cases"][name] = {"ok": False, "error": msg[:400], "trace": traceback.format_exc()[-600:]}
            try:
                torch.cuda.synchronize()
            except Exception:  # noqa: BLE001
                dead = True
        torch.cuda.empty_cache()
    report["passed"] = sum(1 for c in report["cases"].values() if c["ok"])
    report["failed"] = sum(1 for c in report["cases"].values() if not c["ok"])
    report["s"] = round(time.time() - t_all, 1)
    print(json.dumps(report))
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv))
