"""Case runner for the integer-code GEMM (csrc/qgemm_kernels.cu), executed in its OWN process by
tests/test_gpu_qgemm.py: a tcgen05 / TMA pipeline that wedges traps (the kernels carry a watchdog) and a trap poisons the
CUDA context, which must not take the rest of the GPU suite with it.  Prints one JSON report on the last line.

Checked against oracle/restate.py::code_gemm (the factored product, every fp32 rounding where the kernels round:
BIT-EXACT) and ::layer_product_reference (the reference's F.linear / 1x1 F.conv2d on the fake-quantised tensors in
float64: relative tolerance 1e-5 of sum_k |y_a*y_w|, the north star's floating-point bound)."""
import json
import os
import sys
import time
import traceback

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from oracle import restate as R  # noqa: E402

A1, AFFINE, ZP, SYM = 0, 1, 2, 3
I8, E4M3 = 0, 1


def _bytes_of(codes_int, encoding):
    """integer-valued tensor -> the operand bytes of the chosen encoding (host-side construction for raw GEMM cases)."""
    if encoding == I8:
        return (codes_int.to(torch.int64) & 0xFF).to(torch.uint8)
    return codes_int.to(torch.float32).to(torch.float8_e4m3fn).view(torch.uint8)


PATTERNS = ("random", "saturated", "biased", "cancel")
TAIL = 48                                    # trailing K entries of the "cancel" pattern: codes +-1, then one 0


def act_codes_of(pattern, shape, a_hi, a_signed, g):
    """Activation codes of a pattern: "random" draws the whole range; "saturated" is a_hi everywhere; "biased" and
    "cancel" draw the upper half [a_hi // 2 + 1, a_hi] (positive: one sign, so the running sum only grows)."""
    if pattern == "random":
        return torch.randint(-a_hi if a_signed else 0, a_hi + 1, shape, generator=g)
    if pattern == "saturated":
        return torch.full(shape, a_hi, dtype=torch.int64)
    return torch.randint(a_hi // 2 + 1, a_hi + 1, shape, generator=g)


def wt_codes_of(pattern, n, k, w_hi, g):
    """[n, k] weight codes of a pattern, K in accumulation order: "saturated" is -w_hi everywhere (|acc| = K * max|a| *
    max|w|, negative); "biased" draws [w_hi // 2 + 1, w_hi] (odd increments: a constant would add multiples of 32 per
    MMA step and hide a short accumulator); "cancel" is biased positive over the first half of K, negative over the
    second, then TAIL - 1 entries of +-1 and one 0, so the exact result is small but needs every bit up to the
    running sum's peak."""
    if pattern == "random":
        return torch.randint(-w_hi, w_hi + 1, (n, k), generator=g)
    if pattern == "saturated":
        return torch.full((n, k), -w_hi, dtype=torch.int64)
    cw = torch.randint(w_hi // 2 + 1, w_hi + 1, (n, k), generator=g)
    if pattern == "cancel":
        body = k - TAIL
        cw[:, body // 2:body] *= -1
        cw[:, body:] = torch.randint(0, 2, (n, TAIL), generator=g) * 2 - 1
        cw[:, -1] = 0
    return cw


def blocked_acc(ca, cw, step=16, chunk=64):
    """acc = ca [m, K] @ cw [n, K]^T accumulated in K order, one K block of `step` at a time (float64: every partial
    sum is an integer below 2^53, so exact), and the largest |partial sum| at any block boundary."""
    m, k = ca.shape
    n = cw.shape[0]
    a, w = ca.to(torch.float64), cw.to(torch.float64)
    acc = torch.zeros(m, n, dtype=torch.float64)
    peak = 0.0
    for k0 in range(0, k, step * chunk):
        k1 = min(k, k0 + step * chunk)
        nb = (k1 - k0) // step
        blocks = torch.einsum("mbs,nbs->bmn", a[:, k0:k1].reshape(m, nb, step), w[:, k0:k1].reshape(n, nb, step))
        run = acc + blocks.cumsum(0)
        peak = max(peak, run.abs().max().item())
        acc = run[-1]
    return acc, peak


def case_raw_gemm(m, n, k, encoding, a_signed, relu=False, bf16=False, seed=0, a_hi=15, w_hi=7, pattern="random"):
    """codes of a pattern -> dlmcq_qgemm vs the integer oracle, bit for bit.  The worst-case patterns report K, the
    largest |acc| and the largest |partial sum| of the exact accumulation in K order."""
    from dlmc_quant_b200 import qgemm as Q
    g = torch.Generator().manual_seed(seed)
    ca = act_codes_of(pattern, (m, k), a_hi, a_signed, g)
    cw = wt_codes_of(pattern, n, k, w_hi, g)
    if pattern == "cancel":
        ca[:, k - TAIL:] = 1                  # the tail adds an odd sum of +-1
    alpha = (torch.rand(n, generator=g) * 0.01 + 1e-3).float()
    beta = torch.randn(n, generator=g).float()
    out = Q.qgemm(_bytes_of(ca, encoding).cuda(), _bytes_of(cw, encoding).cuda(), alpha.cuda(), beta.cuda(), relu=relu,
                  out_dtype=torch.bfloat16 if bf16 else torch.float32, a_signed=a_signed, encoding=encoding)
    torch.cuda.synchronize()
    report = {"elements": m * n}
    if pattern == "random":
        acc = ca @ cw.t()
    else:
        acc, peak = blocked_acc(ca, cw)
        report.update(K=k, max_abs_acc=int(acc.abs().max().item()), peak_abs_partial_sum=int(peak))
    want = acc.to(torch.float32) * alpha + beta
    if relu:
        want = torch.relu(want)
    if bf16:
        want = want.to(torch.bfloat16)
    got = out.cpu()
    if not torch.equal(got, want):
        bad = (got.float() != want.float())
        idx = bad.nonzero()[0].tolist()
        raise AssertionError(f"{int(bad.sum())} of {bad.numel()} differ; first at {idx}: got {got[tuple(idx)].item()} "
                             f"want {want[tuple(idx)].item()}")
    return report


def _mult(form, scale, g):
    """dequantisation multiplier of a form (fp32, as fq_math.cuh::make_params)."""
    if form == AFFINE:
        return R.grad_scale(scale, g).detach()
    return scale


def case_pipeline(m, n, k, a_form, w_form, encoding, n_bits_a=4, n_bits_w=4, a_signed=False, per_channel=True, bias=True,
                  seed=0):
    """x, w -> codes_forward -> qgemm_prepare -> qgemm, against (1) the integer oracle on the SAME codes bit for bit
    and (2) the reference's product of the two fake-quantised tensors in float64."""
    from dlmc_quant_b200 import functional as F
    from dlmc_quant_b200 import qgemm as Q
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(m, k, generator=g)
    if not a_signed:
        x = torch.relu(x) + 0.05 * torch.rand(m, k, generator=g)
    w = torch.randn(n, k, generator=g) * 0.05
    a_lo, a_hi = R.qrange(a_signed, n_bits_a)
    w_lo, w_hi = R.qrange(True, n_bits_w)
    s_a = (x.abs().max() / a_hi * 0.9).reshape(1).float()
    if a_form == ZP:
        off_a = torch.tensor([3.0 if not a_signed else 0.0])
    elif a_form in (A1, AFFINE):
        off_a = torch.tensor([0.03 if not a_signed else -0.02])
    else:
        off_a = None
    s_w = (w.abs().amax(dim=1) / w_hi + 1e-6).float() if per_channel else (w.abs().max() / w_hi).reshape(1).float()
    g_a = R.lsq_g(x.numel(), a_hi) if a_form == AFFINE else 0.0
    g_w = R.lsq_g(w.numel(), w_hi) if w_form == AFFINE else 0.0
    b = torch.randn(n, generator=g) if bias else None

    xc, wc = x.cuda(), w.cuda()
    a_codes = Q.codes_forward(xc, s_a.cuda(), None if off_a is None else off_a.cuda(), a_lo, a_hi, a_form, g_a,
                              encoding=encoding)
    w_codes = Q.codes_forward(wc, s_w.cuda(), None, w_lo, w_hi, w_form, g_w, ch_axis=0 if per_channel else None,
                              encoding=encoding)
    # (0) the bytes are the codes of the fake-quant kernels
    fa = F.fq_forward(xc, s_a.cuda(), None if off_a is None else off_a.cuda(), a_lo, a_hi, a_form, g_a, want_codes=True,
                      want_y=False)
    fw = F.fq_forward(wc, s_w.cuda(), None, w_lo, w_hi, w_form, g_w, ch_axis=0 if per_channel else None,
                      want_codes=True, want_y=False)

    def ints(bytes_, signed):
        if encoding == E4M3:
            return bytes_.view(torch.float8_e4m3fn).float()
        return bytes_.view(torch.int8).float() if signed else bytes_.float()
    assert torch.equal(ints(a_codes, a_lo < 0), fa), "activation code bytes differ from dlmcq_fq_forward's codes"
    assert torch.equal(ints(w_codes, True), fw), "weight code bytes differ from dlmcq_fq_forward's codes"

    alpha, beta = Q.qgemm_prepare(w_codes, (s_a.cuda(), None if off_a is None else off_a.cuda(), a_lo, a_hi, a_form, g_a),
                                  (s_w.cuda(), w_lo, w_hi, w_form, g_w), None if b is None else b.cuda(), encoding)
    out = Q.qgemm(a_codes, w_codes, alpha, beta, a_signed=a_lo < 0, encoding=encoding)
    torch.cuda.synchronize()

    # (1) integer oracle on the same codes
    m_a = _mult(a_form, s_a, g_a)
    m_w = _mult(w_form, s_w, g_w)
    o_a = off_a if a_form in (A1, AFFINE) else torch.zeros(1)
    z_a = off_a if a_form == ZP else torch.zeros(1)
    want = R.code_gemm(fa.cpu(), fw.cpu(), m_a, o_a, z_a, m_w, b)
    got = out.cpu()
    if not torch.equal(got, want):
        bad = got != want
        idx = bad.nonzero()[0].tolist()
        raise AssertionError(f"vs integer oracle: {int(bad.sum())} of {bad.numel()} differ; first at {idx}: "
                             f"got {got[tuple(idx)].item()} want {want[tuple(idx)].item()}")
    # (2) the reference expression: product of the fake-quantised tensors (oracle chain), float64
    if a_form == AFFINE:
        qa = R.fq_affine(x, s_a, off_a, a_lo, a_hi, g_a)
    elif a_form == ZP:
        qa = R.fq_zp(x, s_a, off_a, a_lo, a_hi)
    elif a_form == A1:
        qa = R.emulate_a1(x, s_a, off_a, a_lo, a_hi)
    else:
        qa = R.fq_sym(x, s_a, a_lo, a_hi)
    sw = s_w.reshape(-1, 1) if per_channel else s_w
    qw = R.fq_affine(w, sw, torch.zeros(1), w_lo, w_hi, g_w) if w_form == AFFINE else R.fq_sym(w, sw, w_lo, w_hi)
    ref = R.layer_product_reference(qa.detach(), qw.detach(), b)
    mag = qa.detach().double().abs() @ qw.detach().double().abs().t() + (0 if b is None else b.double().abs())
    err = ((got.double() - ref).abs() / mag.clamp_min(1e-30)).max().item()
    assert err <= 1e-5, f"vs the reference product: relative error {err:.3e} > 1e-5"
    return {"rel_err_vs_reference_fp64": err}


def case_module(kind, family, encoding, channels_last=True, seed=0):
    """quantize_model + enable_code_gemm: eval forward of the code path vs the module's own fake-quant path."""
    import copy
    from dlmc_quant_b200 import quantize_model
    from dlmc_quant_b200.qgemm import enable_code_gemm
    torch.manual_seed(seed)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    nn = torch.nn
    if kind == "conv":
        net = nn.Sequential(nn.Conv2d(64, 96, 1, bias=True)).cuda()
        # QBase: a float offset (min = 0.1) is part of the factorisation; FSPTQ: its zero-point must be integral
        x = (torch.relu(torch.randn(6, 64, 9, 7)) + (0.1 if family == "qbase" else 0.0)).cuda()
        if channels_last:
            x = x.contiguous(memory_format=torch.channels_last)
            net = net.to(memory_format=torch.channels_last)
    else:
        net = nn.Sequential(nn.Linear(128, 40)).cuda()
        x = torch.relu(torch.randn(3, 5, 128)).cuda()
    if family == "qbase":
        cfg = {"weight": {"enable": True, "type": "minmax_channel", "args": {"n_bits": 4, "signed": True, "ch_axis": 0}},
               "input": {"enable": True, "type": "minmax_tensor", "args": {"n_bits": 4, "signed": False}},
               "exclude_layers": [], "override_options": [], "momentum": 0.1}
        quantize_model(net, copy.deepcopy(cfg), None)
    else:
        cfg = {"weight": {"enable": True, "type": "minmax_channel", "args": {"n_bits": 8, "signed": True, "ch_axis": 0}},
               "input": {"enable": True, "type": "minmax_tensor", "args": {"n_bits": 8, "signed": False}},
               "exclude_layers": [], "override_options": [], "momentum": 0.1}
        quantize_model(net, copy.deepcopy(cfg), None, quantization_type="FSPTQ")
    net.eval()
    with torch.no_grad():
        want = net(x)                                       # initialises the observers, reference path
        want = net(x)
        names = enable_code_gemm(net, encoding)
        assert names, "no layer was switched to the code path"
        got = net(x)
        st = net[0].__dict__["_code_gemm"]
        assert st.usable, "the layer fell back to its original path"
    torch.cuda.synchronize()
    assert got.shape == want.shape
    scale = want.abs().max().item()
    err = (got.float() - want.float()).abs().max().item() / max(scale, 1e-30)
    assert err <= 2e-5, f"code path vs fake-quant path: {err:.3e} of the output's magnitude"
    # under autograd the layer must keep its differentiable path
    y = net(x.clone().requires_grad_(True))
    assert y.grad_fn is not None
    return {"max_err_over_output_scale": err, "switched": names}


def case_fractional_zp():
    """FSPTQ adds the observer's offset as a zero-point (FSPTQuant/base.py:108-109); when it is not an integer the
    clamped codes are not integers either, the product does not factor, and the layer must keep its original path."""
    import copy
    from dlmc_quant_b200 import quantize_model
    from dlmc_quant_b200.qgemm import enable_code_gemm
    torch.manual_seed(3)
    net = torch.nn.Sequential(torch.nn.Linear(64, 24)).cuda()
    cfg = {"weight": {"enable": True, "type": "minmax_channel", "args": {"n_bits": 8, "signed": True, "ch_axis": 0}},
           "input": {"enable": True, "type": "minmax_tensor", "args": {"n_bits": 8, "signed": False}},
           "exclude_layers": [], "override_options": [], "momentum": 0.1}
    quantize_model(net, copy.deepcopy(cfg), None, quantization_type="FSPTQ")
    net.eval()
    x = (torch.rand(10, 64) + 0.37).cuda()
    with torch.no_grad():
        want = net(x)
        assert float(net[0].in_offset) != round(float(net[0].in_offset)), "test premise: fractional zero-point"
        assert enable_code_gemm(net) == ["0"]
        got = net(x)
    assert net[0].__dict__["_code_gemm"].usable is False
    assert torch.equal(got, want)
    return {}


def case_resnet_layers():
    """Every layer of a quantised torchvision ResNet-50 that enable_code_gemm switches, on the input it sees inside the
    model (captured on the strict-fp32 library path): code path vs library path, layer by layer, 2e-5 of the layer's
    output magnitude.  (Whole-model logits are not a parity measure for a 4-bit network: one flipped code is 1/15 of a
    layer's range and 50 untrained layers amplify it - bench.py reports them beside the TF32 path for scale.)"""
    import copy
    import torchvision
    from dlmc_quant_b200 import quantize_model
    from dlmc_quant_b200.qgemm import enable_code_gemm
    torch.manual_seed(11)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    cfg = {"weight": {"enable": True, "type": "minmax_channel", "args": {"n_bits": 4, "signed": True, "ch_axis": 0}},
           "input": {"enable": True, "type": "minmax_tensor", "args": {"n_bits": 4, "signed": False}},
           "exclude_layers": [], "override_options": [], "momentum": 0.1}
    net = torchvision.models.resnet50().cuda().to(memory_format=torch.channels_last)
    quantize_model(net, copy.deepcopy(cfg), None)
    net.eval()
    x = torch.randn(3, 3, 96, 96).cuda().contiguous(memory_format=torch.channels_last)
    seen = {}
    with torch.no_grad():
        net(x)                                              # observers
        hooks = [m.register_forward_hook(lambda mod, inp, out, n=n: seen.__setitem__(n, (mod, inp[0].clone(), out.clone())))
                 for n, m in net.named_modules() if isinstance(m, (torch.nn.Conv2d, torch.nn.Linear))]
        net(x)
        for h in hooks:
            h.remove()
        names = enable_code_gemm(net)
        assert len(names) >= 34, names
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
    return {"layers": len(names), "worst_layer": worst_name, "worst_err_over_output_scale": worst}


def case_golden():
    """tests/golden/qgemm.npz - the eval-mode outputs of the UNMODIFIED reference's QLinear / 1x1 QConv2d / FSPTQ layers:
    the device pipeline (codes_forward -> qgemm_prepare -> qgemm, both operand encodings where the codes fit) equals the
    integer oracle bit for bit and the reference's layer output to 1e-5 of sum_k |y_a*y_w| (+ |bias|)."""
    from dlmc_quant_b200 import qgemm as Q
    from tests import golden_io
    from tests.qgemm_golden import Problem
    worst, runs = 0.0, 0
    for name, case in sorted(golden_io.load("qgemm").items()):
        p = Problem(case)
        ca, cw, m_a, o_a, z_a, m_w = p.oracle()
        want = R.code_gemm(ca, cw, m_a, o_a, z_a, m_w, p.bias)
        encs = [I8] + ([E4M3] if max(p.a_hi, -p.a_lo, p.w_hi, -p.w_lo) <= 16 else [])
        off = p.off_a.cuda()
        for enc in encs:
            a_codes = Q.codes_forward(p.x.cuda(), p.s_a.cuda(), off, p.a_lo, p.a_hi, p.a_form, p.g_a, encoding=enc)
            w_codes = Q.codes_forward(p.w.cuda(), p.s_w.cuda(), None, p.w_lo, p.w_hi, p.w_form, p.g_w,
                                      ch_axis=0 if p.s_w.numel() > 1 else None, encoding=enc)
            alpha, beta = Q.qgemm_prepare(w_codes, (p.s_a.cuda(), off, p.a_lo, p.a_hi, p.a_form, p.g_a),
                                          (p.s_w.cuda(), p.w_lo, p.w_hi, p.w_form, p.g_w),
                                          None if p.bias is None else p.bias.cuda(), enc)
            got = Q.qgemm(a_codes, w_codes, alpha, beta, a_signed=p.a_lo < 0, encoding=enc).cpu()
            assert torch.equal(got, want), f"{name} (encoding {enc}): differs from the integer oracle"
            err = ((got.double() - p.y.double()).abs() / p.bound().clamp_min(1e-30)).max().item()
            assert err <= 1e-5, f"{name}: {err:.3e} vs the reference's layer output"
            worst, runs = max(worst, err), runs + 1
    return {"fixtures_x_encodings": runs, "worst_rel_err_vs_reference_layer_output": worst}


def case_codes_layouts():
    """dlmcq_codes_forward == the codes of dlmcq_fq_forward, byte for byte, on every path of the code kernels: fp32 and
    bf16, vector path with a ragged tail, unaligned views (scalar path), per-channel weights and activations,
    special values (NaN -> 0, +-inf clamp, -0), both encodings."""
    from dlmc_quant_b200 import functional as F
    from dlmc_quant_b200 import qgemm as Q
    g = torch.Generator().manual_seed(17)
    checked = 0
    for dtype in (torch.float32, torch.bfloat16):
        for enc in (I8, E4M3):
            for form, lo, hi, off in ((AFFINE, 0, 15, 0.04), (ZP, 0, 15, 3.0), (SYM, -7, 7, None), (A1, -7, 7, -0.01)):
                x = (torch.randn(4099 + 16 * 37, generator=g) * 2).to(dtype)
                x[:6] = torch.tensor([float("nan"), float("inf"), -float("inf"), -0.0, 0.0, 1e-30]).to(dtype)
                xc = x.cuda()
                s = torch.tensor([0.23]).cuda()
                o = None if off is None else torch.tensor([off]).cuda()
                gg = 1e-3 if form == AFFINE else 0.0
                for view in (xc, xc[1:], xc[:4096]):                      # aligned + ragged, unaligned, aligned exact
                    view = view if view.data_ptr() % 16 else view.contiguous()
                    want = F.fq_forward(view, s, o, lo, hi, form, gg, want_codes=True, want_y=False).float().nan_to_num(0.0)
                    got = Q.codes_forward(view, s, o, lo, hi, form, gg, encoding=enc)
                    gi = got.view(torch.float8_e4m3fn).float() if enc == E4M3 else (
                        got.view(torch.int8).float() if lo < 0 else got.float())
                    assert torch.equal(gi, want), (dtype, enc, form, view.shape)
                    checked += 1
            # per-channel: weights [C, K] (ch_axis 0) and activations [B, C, H, W] (ch_axis 1)
            for shape, ax in (((24, 50), 0), ((3, 8, 5, 5), 1)):
                t = (torch.randn(*shape, generator=g) * 0.1).to(dtype).cuda()
                c = shape[ax]
                sc = (torch.rand(c, generator=g) * 0.02 + 0.01).cuda()
                want = F.fq_forward(t, sc, None, -7, 7, SYM, 0.0, ch_axis=ax, want_codes=True, want_y=False).float()
                got = Q.codes_forward(t, sc, None, -7, 7, SYM, 0.0, ch_axis=ax, encoding=enc)
                gi = got.view(torch.float8_e4m3fn).float() if enc == E4M3 else got.view(torch.int8).float()
                assert torch.equal(gi, want), (dtype, enc, shape)
                checked += 1
    return {"comparisons": checked}


def case_cuda_graph():
    """The switched layers are capturable: after one warm forward (observers, weight codes, alpha / beta cached, kernel
    attributes set) a forward holds no host synchronisation, so torch.cuda.graph records it; replays on fresh inputs
    equal the eager code path bit for bit."""
    import copy
    from dlmc_quant_b200 import quantize_model
    from dlmc_quant_b200.qgemm import enable_code_gemm
    torch.manual_seed(5)
    nn = torch.nn
    net = nn.Sequential(nn.Conv2d(32, 64, 1), nn.ReLU(), nn.Conv2d(64, 48, 1, bias=False), nn.ReLU(),
                        nn.AdaptiveAvgPool2d(1), nn.Flatten(), nn.Linear(48, 16)).cuda().to(memory_format=torch.channels_last)
    cfg = {"weight": {"enable": True, "type": "minmax_channel", "args": {"n_bits": 4, "signed": True, "ch_axis": 0}},
           "input": {"enable": True, "type": "minmax_tensor", "args": {"n_bits": 4, "signed": False}},
           "exclude_layers": [], "override_options": [], "momentum": 0.1}
    quantize_model(net, copy.deepcopy(cfg), None)
    net.eval()
    xs = [torch.rand(5, 32, 10, 10).cuda().contiguous(memory_format=torch.channels_last) for _ in range(3)]
    with torch.no_grad():
        net(xs[0])
        assert enable_code_gemm(net) == ["0", "2", "6"]
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
    from dlmc_quant_b200 import qgemm as Q
    from dlmc_quant_b200._lib import DlmcqError
    a = torch.zeros(16, 24, dtype=torch.uint8).cuda()
    w = torch.zeros(8, 24, dtype=torch.uint8).cuda()
    al = torch.ones(8).cuda()
    try:
        Q.qgemm(a, w, al, al)
    except DlmcqError as e:
        assert "unsupported" in str(e)
    else:
        raise AssertionError("k % 16 != 0 was accepted")
    empty = Q.qgemm(torch.zeros(0, 32, dtype=torch.uint8).cuda(), torch.zeros(8, 32, dtype=torch.uint8).cuda(), al, al)
    assert empty.shape == (0, 8)
    # the accumulator bound of qgemm_prepare: accepted at K * max|a| * max|w| = 2^24 (e4m3) and at the largest K of
    # 8-bit codes below 2^31 - 1 (integer kind), refused one K block above
    act = lambda hi: (torch.ones(1).cuda(), torch.zeros(1).cuda(), 0, hi, A1, 0.0)  # noqa: E731
    for enc, a_hi, w_hi, k_ok in ((E4M3, 16, 16, 65536), (I8, 255, 127, 66304)):
        for k, ok in ((k_ok, True), (k_ok + 16, False)):
            try:
                Q.qgemm_prepare(torch.zeros(8, k, dtype=torch.uint8).cuda(), act(a_hi), (al, -w_hi, w_hi, SYM, 0.0),
                                None, enc)
                accepted = True
            except DlmcqError as e:
                assert "unsupported" in str(e), e
                accepted = False
            assert accepted == ok, (enc, k)
    torch.cuda.synchronize()
    return {}


def build_cases():
    cases = []
    raw_shapes = [(128, 128, 128), (256, 128, 512), (128, 256, 128), (100, 72, 64), (300, 200, 208), (1, 16, 16),
                  (401, 1000, 2048), (4096, 64, 256), (129, 129, 144), (512, 512, 4096),
                  (128 * 150 + 7, 384, 96),          # 453 tiles: every persistent CTA walks several, both TMEM buffers reused
                  (128 * 148 * 2, 128, 640)]         # exactly two tiles per CTA, the operand ring wraps inside a tile
    for enc in (I8, E4M3):
        tag = "i8" if enc == I8 else "e4m3"
        for (m, n, k) in raw_shapes:
            cases.append((f"raw_{tag}_{m}x{n}x{k}", case_raw_gemm, dict(m=m, n=n, k=k, encoding=enc, a_signed=False)))
        cases.append((f"raw_{tag}_signed", case_raw_gemm, dict(m=200, n=136, k=320, encoding=enc, a_signed=True, a_hi=7)))
        cases.append((f"raw_{tag}_relu_bf16", case_raw_gemm, dict(m=257, n=96, k=128, encoding=enc, a_signed=False,
                                                                    relu=True, bf16=True)))
        cases.append((f"raw_{tag}_bf16_scalar_stores", case_raw_gemm, dict(m=300, n=100, k=160, encoding=enc, a_signed=False,
                                                                            bf16=True)))
        cases.append((f"raw_{tag}_relu", case_raw_gemm, dict(m=130, n=130, k=256, encoding=enc, a_signed=False, relu=True)))
    # 8-bit codes need the integer kind; K = 8192 keeps |acc| far beyond 2^24 so the s32 -> f32 rounding is exercised
    cases.append(("raw_i8_8bit", case_raw_gemm, dict(m=256, n=128, k=8192, encoding=I8, a_signed=False, a_hi=255, w_hi=127)))
    cases.append(("raw_i8_8bit_signed", case_raw_gemm, dict(m=64, n=48, k=1024, encoding=I8, a_signed=True, a_hi=127,
                                                            w_hi=127)))
    # worst-case accumulators: the ResNet-50 3x3 layers' K (9 * 64 ... 9 * 512) and 2048 with 4-bit codes on both
    # kinds; e4m3 at K = 65520 on its extreme codes (|code| = 16: K * 16 * 16 just below 2^24); the integer kind with
    # 8-bit codes at the largest multiple of 16 with K * 255 * 127 <= 2^31 - 1
    for pattern in PATTERNS[1:]:
        for enc, tag in ((I8, "i8"), (E4M3, "e4m3")):
            for k in (576, 1152, 2048, 2304, 4608):
                cases.append((f"acc_{tag}_{pattern}_k{k}", case_raw_gemm,
                              dict(m=136, n=144, k=k, encoding=enc, a_signed=False, pattern=pattern, seed=k)))
        cases.append((f"acc_e4m3_{pattern}_k65520", case_raw_gemm,
                      dict(m=128, n=128, k=65520, encoding=E4M3, a_signed=False, a_hi=16, w_hi=16, pattern=pattern)))
        cases.append((f"acc_i8_8bit_{pattern}_k66304", case_raw_gemm,
                      dict(m=128, n=128, k=66304, encoding=I8, a_signed=False, a_hi=255, w_hi=127, pattern=pattern)))
    for enc in (I8, E4M3):
        tag = "i8" if enc == I8 else "e4m3"
        cases.append((f"pipe_{tag}_affine", case_pipeline, dict(m=300, n=72, k=256, a_form=AFFINE, w_form=AFFINE, encoding=enc)))
        cases.append((f"pipe_{tag}_zp_sym", case_pipeline, dict(m=260, n=130, k=192, a_form=ZP, w_form=SYM, encoding=enc)))
        cases.append((f"pipe_{tag}_a1_sym_per_tensor", case_pipeline, dict(m=64, n=40, k=128, a_form=A1, w_form=SYM,
                                                                            encoding=enc, per_channel=False, bias=False)))
        cases.append((f"pipe_{tag}_sym_signed_act", case_pipeline, dict(m=96, n=24, k=64, a_form=SYM, w_form=SYM, encoding=enc,
                                                                         a_signed=True)))
    cases.append(("pipe_i8_zp_8bit", case_pipeline, dict(m=200, n=64, k=512, a_form=ZP, w_form=SYM, encoding=I8, n_bits_a=8,
                                                         n_bits_w=8)))
    for enc in (I8, E4M3):
        tag = "i8" if enc == I8 else "e4m3"
        cases.append((f"module_{tag}_conv_qbase", case_module, dict(kind="conv", family="qbase", encoding=enc)))
        cases.append((f"module_{tag}_linear_qbase", case_module, dict(kind="linear", family="qbase", encoding=enc)))
    cases.append(("module_auto_encoding_conv_qbase", case_module, dict(kind="conv", family="qbase", encoding=None)))
    cases.append(("module_i8_conv_fsptq_8bit", case_module, dict(kind="conv", family="fsptq", encoding=I8)))
    cases.append(("module_i8_linear_fsptq_8bit", case_module, dict(kind="linear", family="fsptq", encoding=I8)))
    cases.append(("module_i8_conv_nchw_qbase", case_module, dict(kind="conv", family="qbase", encoding=I8, channels_last=False)))
    cases.append(("module_fsptq_fractional_zero_point_keeps_reference_path", case_fractional_zp, {}))
    cases.append(("module_resnet50_every_switched_layer", case_resnet_layers, {}))
    cases.append(("module_cuda_graph_capture", case_cuda_graph, {}))
    cases.append(("codes_forward_every_path", case_codes_layouts, {}))
    cases.append(("golden_reference_layer_outputs", case_golden, {}))
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
