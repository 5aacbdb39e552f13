"""Case runner for the convolution on the integer codes (csrc/qgemm_kernels.cu qconv_kernel: TMA im2col -> tcgen05 ->
TMEM), executed in its OWN process by tests/test_gpu_qconv.py for the same reason as tests/qgemm_cases.py: a wedged
pipeline traps and a trap poisons the CUDA context.  Prints one JSON report on the last line.

Checked against tests/qconv_oracle.py::code_conv (exact integer convolution, the border rule for beta, the kernels'
two fp32 roundings: BIT-EXACT) and ::conv_reference (F.conv2d of the fake-quantised tensors in float64: 1e-5 of
conv2d(|y_a|, |y_w|)); module cases against the layer's own fake-quant + cuDNN path in strict fp32 (2e-5 of the
output's magnitude)."""
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

from tests.qconv_oracle import A1, AFFINE, GEOMETRIES, SYM, ZP, code_conv, conv_problem, conv_reference  # noqa: E402
from tests.qgemm_cases import PATTERNS, act_codes_of, blocked_acc, wt_codes_of  # noqa: E402

I8, E4M3 = 0, 1


def _bytes_of(codes_int, encoding):
    if encoding == I8:
        return (codes_int.to(torch.int64) & 0xFF).to(torch.uint8)
    return codes_int.to(torch.float32).to(torch.float8_e4m3fn).view(torch.uint8)


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def _assert_equal(got, want, what):
    if not torch.equal(got, want):
        bad = got.float() != want.float()
        idx = bad.nonzero()[0].tolist()
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} differ; first at {idx}: "
                             f"got {got[tuple(idx)].item()} want {want[tuple(idx)].item()}")


def case_raw(geom, encoding, batch=2, cin=64, n=40, a_signed=False, relu=False, bf16=False, zp=False, seed=0,
             a_hi=15, w_hi=7, pattern="random"):
    """codes of a pattern (tests/qgemm_cases.py PATTERNS; the weights' K order is the kernel's (r, s, c)) ->
    qconv_prepare (A1 offset or ZP zero-point activation, per-channel SYM weight) -> qconv vs code_conv, bit for bit.
    The worst-case patterns report K, the largest |acc| and the largest |partial sum| of the exact accumulation."""
    from dlmc_quant_b200 import qgemm as Q
    kh, kw, stride, padding, dilation, h, w = geom
    g = torch.Generator().manual_seed(seed)
    a_lo = -a_hi if a_signed else 0
    report = {}
    if pattern == "random":
        ca = torch.randint(a_lo, a_hi + 1, (batch, cin, h, w), generator=g)
        cw = torch.randint(-w_hi, w_hi + 1, (n, cin, kh, kw), generator=g)
    else:
        ca = act_codes_of(pattern, (batch, cin, h, w), a_hi, a_signed, g)
        cw_k = wt_codes_of(pattern, n, kh * kw * cin, w_hi, g)                 # [n, K], K = (r, s, c)
        cw = cw_k.reshape(n, kh, kw, cin).permute(0, 3, 1, 2).contiguous()
        cols = torch.nn.functional.unfold(ca.double(), (kh, kw), dilation=dilation, padding=padding, stride=stride)
        cols = cols.reshape(batch, cin, kh, kw, -1).permute(0, 4, 2, 3, 1).reshape(-1, kh * kw * cin)
        acc, peak = blocked_acc(cols, cw_k)
        report.update(K=kh * kw * cin, max_abs_acc=int(acc.abs().max().item()), peak_abs_partial_sum=int(peak))
    s_a = torch.tensor([0.0371])
    off = torch.tensor([3.0 if zp else -0.21])
    s_w = (torch.rand(n, generator=g) * 0.01 + 1e-3)
    bias = torch.randn(n, generator=g)
    act = (s_a.cuda(), off.cuda(), a_lo, a_hi, ZP if zp else A1, 0.0)
    wt = (s_w.cuda(), -w_hi, w_hi, SYM, 0.0)
    wc = _bytes_of(_nhwc(cw), encoding).cuda()
    alpha, beta = Q.qconv_prepare(wc, act, wt, bias.cuda(), encoding)
    out = Q.qconv(_bytes_of(_nhwc(ca), encoding).cuda(), wc, alpha, beta, stride, padding, dilation, relu=relu,
                  out_dtype=torch.bfloat16 if bf16 else torch.float32, a_signed=a_signed, encoding=encoding)
    torch.cuda.synchronize()
    want = code_conv(ca, cw, s_a, torch.zeros(1) if zp else off, off if zp else torch.zeros(1), s_w, bias,
                     stride=stride, padding=padding, dilation=dilation, relu=relu)
    want = _nhwc(want)
    if bf16:
        want = want.to(torch.bfloat16)
    _assert_equal(out.cpu(), want, "vs code_conv")
    return {"pixels": out.shape[0] * out.shape[1] * out.shape[2], "n": n, **report}


def case_pipeline(geom, a_form, w_form, encoding, dtype=torch.float32, cin=64, n=48, n_bits=4, a_signed=False,
                  per_channel=True, seed=0):
    """x, w -> codes_forward -> qconv_prepare -> qconv: bit-exact vs code_conv on the oracle's codes, <= 1e-5 vs the
    reference's F.conv2d of the fake-quantised tensors in float64."""
    from dlmc_quant_b200 import qgemm as Q
    p = conv_problem(a_form, w_form, geom, cin=cin, n=n, n_bits=n_bits, a_signed=a_signed, per_channel=per_channel,
                     seed=seed)
    x = p["x"]
    if dtype == torch.bfloat16:                                # the reference sees the bf16 input's values
        x = x.to(torch.bfloat16)
        p = conv_problem(a_form, w_form, geom, cin=cin, n=n, n_bits=n_bits, a_signed=a_signed, per_channel=per_channel,
                         seed=seed)
        from oracle import restate as R
        xf = x.float()
        a_lo, a_hi = p["a_range"]
        if a_form == AFFINE:
            p["qa"], p["ca"] = R.fq_affine(xf, p["s_a"], p["off"], a_lo, a_hi, p["g_a"]), R.fq_affine_codes(xf, p["s_a"], p["off"], a_lo, a_hi, p["g_a"])
        elif a_form == ZP:
            p["qa"], p["ca"] = R.fq_zp(xf, p["s_a"], p["off"], a_lo, a_hi), R.fq_zp_codes(xf, p["s_a"], p["off"], a_lo, a_hi)
        elif a_form == A1:
            p["qa"], p["ca"] = R.emulate_a1(xf, p["s_a"], p["off"], a_lo, a_hi), R.codes_a1(xf, p["s_a"], p["off"], a_lo, a_hi)
        else:
            p["qa"], p["ca"] = R.fq_sym(xf, p["s_a"], a_lo, a_hi), R.fq_sym_codes(xf, p["s_a"], a_lo, a_hi)
        p["qa"], p["ca"] = p["qa"].detach(), p["ca"].detach()
    a_lo, a_hi = p["a_range"]
    w_lo, w_hi = p["w_range"]
    off = None if p["off"] is None else p["off"].cuda()
    xc = x.cuda().contiguous(memory_format=torch.channels_last)
    a_codes = Q.codes_forward(xc, p["s_a"].cuda(), off, a_lo, a_hi, a_form, p["g_a"], encoding=encoding)
    w_nhwc = p["w"].permute(0, 2, 3, 1).contiguous().cuda()
    w_codes = Q.codes_forward(w_nhwc, p["s_w"].cuda(), None, w_lo, w_hi, w_form, p["g_w"],
                              ch_axis=0 if per_channel else None, encoding=encoding)
    alpha, beta = Q.qconv_prepare(w_codes, (p["s_a"].cuda(), off, a_lo, a_hi, a_form, p["g_a"]),
                                  (p["s_w"].cuda(), w_lo, w_hi, w_form, p["g_w"]), p["bias"].cuda(), encoding)
    out = Q.qconv(a_codes.permute(0, 2, 3, 1), w_codes, alpha, beta, a_signed=a_lo < 0, encoding=encoding,
                  **p["conv"]).cpu()
    want = _nhwc(code_conv(p["ca"], p["cw"], p["m_a"], p["o_a"], p["z_a"], p["m_w"], p["bias"], **p["conv"]))
    _assert_equal(out, want, "vs code_conv")
    ref, mag = conv_reference(p["qa"], p["qw"], p["bias"], **p["conv"])
    err = ((out.permute(0, 3, 1, 2).double() - ref).abs() / mag.clamp_min(1e-30)).max().item()
    assert err <= 1e-5, f"vs the reference conv: {err:.3e}"
    return {"rel_err_vs_reference_fp64": err}


def _quantised(net, family):
    from dlmc_quant_b200 import quantize_model
    bits, kind = (4, None) if family == "qbase" else (8, "FSPTQ")
    cfg = {"weight": {"enable": True, "type": "minmax_channel", "args": {"n_bits": bits, "signed": True, "ch_axis": 0}},
           "input": {"enable": True, "type": "minmax_tensor", "args": {"n_bits": bits, "signed": False}},
           "exclude_layers": [], "override_options": [], "momentum": 0.1}
    if kind:
        quantize_model(net, copy.deepcopy(cfg), None, quantization_type=kind)
    else:
        quantize_model(net, copy.deepcopy(cfg), None)
    return net


def case_module(conv_kw, family, encoding=None, channels_last=True, cin=64, seed=0):
    """enable_code_gemm(convolutions=True): eval forward of the code path vs the layer's own fake-quant path."""
    from dlmc_quant_b200.qgemm import enable_code_gemm
    torch.manual_seed(seed)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    net = _quantised(torch.nn.Sequential(torch.nn.Conv2d(cin, 72, **conv_kw)).cuda(), family)
    # QBase: a float offset (min = 0.1) enters beta and the border rule; FSPTQ: integral zero-point
    x = (torch.relu(torch.randn(4, cin, 13, 11)) + (0.1 if family == "qbase" else 0.0)).cuda()
    if channels_last:
        x = x.contiguous(memory_format=torch.channels_last)
        net = net.to(memory_format=torch.channels_last)
    net.eval()
    with torch.no_grad():
        net(x)
        want = net(x)
        assert enable_code_gemm(net) == [], "the layer is not a 1x1 / Linear layer"
        names = enable_code_gemm(net, encoding, convolutions=True)
        assert names == ["0"], names
        got = net(x)
        st = net[0].__dict__["_code_gemm"]
        assert st.usable and st.conv, "the layer fell back to its original path"
    torch.cuda.synchronize()
    assert got.shape == want.shape
    err = (got.float() - want.float()).abs().max().item() / max(want.abs().max().item(), 1e-30)
    assert err <= 2e-5, f"code path vs fake-quant path: {err:.3e} of the output's magnitude"
    y = net(x.clone().requires_grad_(True))
    assert y.grad_fn is not None, "autograd call left the differentiable path"
    return {"max_err_over_output_scale": err}


def case_fallback(kind):
    """Layers the kernel does not serve keep their original path, bit for bit."""
    from dlmc_quant_b200.qgemm import enable_code_gemm
    torch.manual_seed(2)
    nn = torch.nn
    family = "qbase"
    x = torch.rand(2, 64, 10, 10).cuda() + 0.2
    if kind == "groups":
        mod = nn.Conv2d(64, 64, 3, padding=1, groups=2)
    elif kind == "stem":
        mod, x = nn.Conv2d(3, 64, 7, stride=2, padding=3), torch.rand(2, 3, 32, 32).cuda()
    elif kind == "reflect":
        mod = nn.Conv2d(64, 32, 3, padding=1, padding_mode="reflect")
    else:                                                       # FSPTQ with a fractional zero-point
        mod, family, x = nn.Conv2d(64, 32, 3, padding=1), "fsptq", torch.rand(2, 64, 10, 10).cuda() + 0.37
    net = _quantised(nn.Sequential(mod).cuda(), family)
    net.eval()
    with torch.no_grad():
        want = net(x)
        names = enable_code_gemm(net, convolutions=True)
        got = net(x)
    if kind == "zero_point":
        assert names == ["0"] and net[0].__dict__["_code_gemm"].usable is False
        assert float(net[0].in_offset) != round(float(net[0].in_offset)), "test premise: fractional zero-point"
    else:
        assert names == [], names
    assert torch.equal(got, want)
    return {}


def case_resnet_layers():
    """Quantised torchvision ResNet-50: convolutions=True switches every 3x3 and strided layer besides the 34 of the
    default; each switched layer matches the library path on its in-model input within 2e-5 of its output's magnitude;
    the default switch is unchanged."""
    import torchvision
    from dlmc_quant_b200.qgemm import enable_code_gemm
    torch.manual_seed(11)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    net = torchvision.models.resnet50().cuda().to(memory_format=torch.channels_last)
    _quantised(net, "qbase")
    net.eval()
    x = torch.randn(3, 3, 96, 96).cuda().contiguous(memory_format=torch.channels_last)
    seen = {}
    with torch.no_grad():
        net(x)
        hooks = [m.register_forward_hook(lambda mod, inp, out, n=n: seen.__setitem__(n, (mod, inp[0].clone(), out.clone())))
                 for n, m in net.named_modules() if isinstance(m, (torch.nn.Conv2d, torch.nn.Linear))]
        net(x)
        for h in hooks:
            h.remove()
        names = enable_code_gemm(net, convolutions=True)
        assert len(names) >= 53, len(names)
        conv_names = [n for n in names if net.get_submodule(n).__dict__["_code_gemm"].conv]
        worst, worst_name = 0.0, None
        for n in names:
            mod, inp, want = seen[n]
            got = mod(inp)
            assert mod.__dict__["_code_gemm"].usable, f"{n} fell back to the library path"
            assert got.shape == want.shape
            err = float((got.float() - want.float()).abs().max() / want.abs().max().clamp_min(1e-30))
            if err > worst:
                worst, worst_name = err, n
        assert worst <= 2e-5, f"{worst_name}: {worst:.3e} of the layer's output magnitude"
    net2 = _quantised(torchvision.models.resnet50().cuda(), "qbase")
    default = enable_code_gemm(net2)
    assert default == [n for n in names if n not in conv_names] and len(default) == 34, default
    return {"layers": len(names), "conv_layers": len(conv_names), "worst_layer": worst_name,
            "worst_err_over_output_scale": worst}


def case_cuda_graph():
    """A switched 3x3 layer is capturable after one warm forward; replays equal the eager code path bit for bit."""
    from dlmc_quant_b200.qgemm import enable_code_gemm
    torch.manual_seed(5)
    nn = torch.nn
    net = nn.Sequential(nn.Conv2d(64, 64, 3, padding=1), nn.ReLU(), nn.Conv2d(64, 128, 3, stride=2, padding=1),
                        nn.ReLU()).cuda().to(memory_format=torch.channels_last)
    _quantised(net, "qbase")
    net.eval()
    xs = [torch.rand(3, 64, 12, 12).cuda().contiguous(memory_format=torch.channels_last) + 0.1 for _ in range(3)]
    with torch.no_grad():
        net(xs[0])
        assert enable_code_gemm(net, convolutions=True) == ["0", "2"]
        eager = [net(x).clone() for x in xs]
        static_x = xs[0].clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            net(static_x)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            static_y = net(static_x)
        for x, want in zip(xs, eager):
            static_x.copy_(x)
            graph.replay()
            torch.cuda.synchronize()
            assert torch.equal(static_y, want), "graph replay differs from the eager code path"
    return {}


def case_errors():
    """Unsupported geometry / alignment is refused with the documented status before any launch."""
    import ctypes as C
    from dlmc_quant_b200 import _lib
    from dlmc_quant_b200 import qgemm as Q
    EINVAL, EALIGN, EUNSUPPORTED = -1, -2, -5
    h = _lib.lib()
    a = torch.zeros(2 * 8 * 8 * 64 + 16, dtype=torch.uint8).cuda()
    w = torch.zeros(4 * 9 * 64, dtype=torch.uint8).cuda()
    al = torch.ones(4).cuda()
    be = torch.zeros(256 * 4).cuda()
    out = torch.empty(2 * 8 * 8 * 4).cuda()

    def run(ptr_a=None, **kw):
        g = Q._geom(2, 8, 8, 64, 4, 3, 3, 1, 1, 1)
        for k, v in kw.items():
            setattr(g, k, v)
        return h.dlmcq_qconv(C.c_void_p(ptr_a or a.data_ptr()), C.c_void_p(w.data_ptr()), C.c_void_p(al.data_ptr()),
                             C.c_void_p(be.data_ptr()), C.c_void_p(out.data_ptr()), C.byref(g), 0, 0, 0, 0, None)
    got = {"groups": run(groups=2), "cin_96": run(cin=96), "stride_9": run(stride_h=9), "pad_200": run(pad_w=200),
           "corner": run(h=300, dil_h=100, pad_h=1), "unaligned": run(ptr_a=a.data_ptr() + 1), "no_output": run(h=1, pad_h=0),
           "negative_pad": run(pad_h=-1), "huge": run(batch=1 << 20, h=4096, w=4096, pad_h=1)}
    want = {"groups": EUNSUPPORTED, "cin_96": EUNSUPPORTED, "stride_9": EUNSUPPORTED, "pad_200": EUNSUPPORTED,
            "corner": EUNSUPPORTED, "unaligned": EALIGN, "no_output": EINVAL, "negative_pad": EINVAL,
            "huge": EUNSUPPORTED}
    assert got == want, got
    assert run() == 0
    # the accumulator bound of qconv_prepare (K = kh*kw*Cin): accepted at K * 16 * 16 = 2^24 (e4m3) and at the largest
    # Cin of 8-bit 3x3 codes below 2^31 - 1 (integer kind), refused one channel block above
    act = lambda hi: (torch.ones(1).cuda(), torch.zeros(1).cuda(), 0, hi, A1, 0.0)  # noqa: E731
    for enc, a_hi, w_hi, taps, cin_ok in ((E4M3, 16, 16, 1, 65536), (I8, 255, 127, 3, 7360)):
        for cin, ok in ((cin_ok, True), (cin_ok + 64, False)):
            try:
                Q.qconv_prepare(torch.zeros(4, taps, taps, cin, dtype=torch.uint8).cuda(), act(a_hi),
                                (al, -w_hi, w_hi, SYM, 0.0), None, enc)
                accepted = True
            except _lib.DlmcqError as e:
                assert "unsupported" in str(e), e
                accepted = False
            assert accepted == ok, (enc, cin)
    torch.cuda.synchronize()
    return {}


def build_cases():
    cases = []
    for enc, tag in ((I8, "i8"), (E4M3, "e4m3")):
        for name in sorted(GEOMETRIES):
            cases.append((f"raw_{tag}_{name}", case_raw, dict(geom=GEOMETRIES[name], encoding=enc, seed=len(name))))
        g33 = (3, 3, 1, 1, 1, 14, 14)
        cases.append((f"raw_{tag}_cin128_zp", case_raw, dict(geom=g33, encoding=enc, cin=128, n=64, zp=True)))
        cases.append((f"raw_{tag}_cin256_stride2", case_raw, dict(geom=(3, 3, 2, 1, 1, 15, 13), encoding=enc, cin=256,
                                                                   n=136)))
        cases.append((f"raw_{tag}_cin192_ragged_n", case_raw, dict(geom=g33, encoding=enc, cin=192, n=130)))
        cases.append((f"raw_{tag}_scalar_epilogue", case_raw, dict(geom=g33, encoding=enc, n=30)))
        cases.append((f"raw_{tag}_bf16_relu", case_raw, dict(geom=g33, encoding=enc, n=72, relu=True, bf16=True)))
        cases.append((f"raw_{tag}_bf16_scalar", case_raw, dict(geom=g33, encoding=enc, n=36, bf16=True)))
        cases.append((f"raw_{tag}_signed", case_raw, dict(geom=g33, encoding=enc, a_signed=True, a_hi=7)))
        # 392 tiles over 148 SMs: persistent walk, both TMEM buffers reused; 28x28 planes: tiles straddle images
        cases.append((f"raw_{tag}_persistent", case_raw, dict(geom=(3, 3, 1, 1, 1, 28, 28), encoding=enc, batch=32,
                                                               cin=128, n=256)))
    # n = 1 (scalar epilogue, one-row beta table), n = 2048 (16 N tiles), a single output pixel, batch 1 below one tile
    for enc, tag in ((I8, "i8"), (E4M3, "e4m3")):
        cases.append((f"raw_{tag}_n1", case_raw, dict(geom=GEOMETRIES["3x3_pad1"], encoding=enc, n=1)))
        cases.append((f"raw_{tag}_n2048", case_raw, dict(geom=GEOMETRIES["3x3_pad1_stride2"], encoding=enc, n=2048)))
        cases.append((f"raw_{tag}_one_output_pixel", case_raw, dict(geom=(3, 3, 1, 0, 1, 3, 3), encoding=enc, batch=1,
                                                                     cin=128, n=96)))
        cases.append((f"raw_{tag}_batch1_below_one_tile", case_raw, dict(geom=(3, 3, 1, 1, 1, 9, 11), encoding=enc,
                                                                          batch=1, n=72)))
    # worst-case accumulators (tests/qgemm_cases.py PATTERNS): the ResNet-50 3x3 layers' K = 9 * 64 ... 9 * 512 on
    # both kinds; e4m3 with |code| = 16 at K = 9 * 7232 (K * 256 just below 2^24); 8-bit codes on the integer kind at
    # K = 9 * 7360 (K * 255 * 127 just below 2^31 - 1)
    g_acc = (3, 3, 1, 1, 1, 12, 11)
    for pattern in PATTERNS[1:]:
        for enc, tag in ((I8, "i8"), (E4M3, "e4m3")):
            for cin in (64, 128, 256, 512):
                cases.append((f"acc_{tag}_{pattern}_k{9 * cin}", case_raw,
                              dict(geom=g_acc, encoding=enc, cin=cin, n=64, pattern=pattern, seed=cin)))
        cases.append((f"acc_e4m3_{pattern}_k{9 * 7232}", case_raw,
                      dict(geom=g_acc, encoding=E4M3, cin=7232, n=64, a_hi=16, w_hi=16, pattern=pattern)))
        cases.append((f"acc_i8_8bit_{pattern}_k{9 * 7360}", case_raw,
                      dict(geom=g_acc, encoding=I8, cin=7360, n=64, a_hi=255, w_hi=127, pattern=pattern)))
    cases.append(("raw_i8_8bit_signed", case_raw, dict(geom=(3, 3, 1, 1, 1, 9, 9), encoding=I8, cin=512, n=64,
                                                       a_signed=True, a_hi=127, w_hi=127)))
    cases.append(("raw_i8_8bit", case_raw, dict(geom=(3, 3, 1, 1, 1, 7, 7), encoding=I8, cin=512, n=64, a_hi=255,
                                                w_hi=127)))
    for enc, tag in ((I8, "i8"), (E4M3, "e4m3")):
        for name in ("3x3_pad1", "3x3_pad1_stride2", "1x1_stride2", "5x5_pad2", "3x3_dilation2"):
            cases.append((f"pipe_{tag}_affine_{name}", case_pipeline, dict(geom=GEOMETRIES[name], a_form=AFFINE,
                                                                          w_form=AFFINE, encoding=enc)))
        cases.append((f"pipe_{tag}_zp_sym", case_pipeline, dict(geom=GEOMETRIES["3x3_pad1"], a_form=ZP, w_form=SYM,
                                                                encoding=enc, cin=128)))
        cases.append((f"pipe_{tag}_a1_sym_per_tensor", case_pipeline, dict(geom=GEOMETRIES["1x3"], a_form=A1,
                                                                           w_form=SYM, encoding=enc, per_channel=False)))
        cases.append((f"pipe_{tag}_sym_signed", case_pipeline, dict(geom=GEOMETRIES["3x1"], a_form=SYM, w_form=SYM,
                                                                    encoding=enc, a_signed=True)))
        cases.append((f"pipe_{tag}_affine_bf16", case_pipeline, dict(geom=GEOMETRIES["3x3_pad1"], a_form=AFFINE,
                                                                     w_form=SYM, encoding=enc, dtype=torch.bfloat16)))
    cases.append(("pipe_i8_zp_8bit", case_pipeline, dict(geom=GEOMETRIES["3x3_pad1_stride2"], a_form=ZP, w_form=SYM,
                                                         encoding=I8, n_bits=8, cin=128)))
    for fam in ("qbase", "fsptq"):
        cases.append((f"module_{fam}_3x3", case_module, dict(conv_kw=dict(kernel_size=3, padding=1), family=fam)))
        cases.append((f"module_{fam}_3x3_stride2_nchw", case_module, dict(conv_kw=dict(kernel_size=3, stride=2, padding=1),
                                                                           family=fam, channels_last=False, cin=128)))
        cases.append((f"module_{fam}_1x1_stride2", case_module, dict(conv_kw=dict(kernel_size=1, stride=2), family=fam)))
    cases.append(("module_qbase_i8_3x3_nchw", case_module, dict(conv_kw=dict(kernel_size=3, padding=1), family="qbase",
                                                                encoding=I8, channels_last=False)))
    for kind in ("groups", "stem", "reflect", "zero_point"):
        cases.append((f"fallback_{kind}", case_fallback, dict(kind=kind)))
    cases.append(("module_resnet50_every_switched_layer", case_resnet_layers, {}))
    cases.append(("module_cuda_graph_capture", case_cuda_graph, {}))
    cases.append(("errors", case_errors, {}))
    return cases


def main(argv):
    only = argv[1] if len(argv) > 1 else ""
    report = {"cases": {}, "device": torch.cuda.get_device_name(0)}
    dead = False
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
    report["passed"] = sum(1 for c in report["cases"].values() if c["ok"])
    report["failed"] = sum(1 for c in report["cases"].values() if not c["ok"])
    print(json.dumps(report))
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv))
