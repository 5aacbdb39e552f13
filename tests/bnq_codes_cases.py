"""Case runner for the fused BatchNorm producer that writes the consumer's integer codes (dlmcq_bnq_forward_codes) and its
wiring into the code GEMM (fuse.py + qgemm.py), executed in its OWN process by tests/test_gpu_bnq_codes.py: the consumer
side is a tcgen05 / TMA pipeline whose failure mode is a trap that poisons the CUDA context.  Prints one JSON report on
the last line.

Bars, all bit for bit:
  * raw entry: codes_out == dlmcq_codes_forward(a) with a the same call's plain output; a_out and save_mean /
    save_invstd == those of dlmcq_bnq_forward on identical inputs;
  * models: the producer handing codes to the code GEMM gives the same logits as every consumer quantising the fused
    plain output itself with codes_forward (fuse._consumer_q disabled); fallbacks give the same outputs as fuse alone;
    switch order, disable_code_gemm / unfuse() and CUDA-graph replay change nothing."""
import copy
import ctypes as C
import json
import math
import os
import sys
import time
import traceback

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

I8, E4M3 = 0, 1
# (rows, C) of every BatchNorm site of torchvision ResNet-50 at batch 128
R50_SITES = [(128 * 56 * 56, 64), (128 * 56 * 56, 256), (128 * 28 * 28, 128), (128 * 28 * 28, 512),
             (128 * 14 * 14, 256), (128 * 14 * 14, 1024), (128 * 7 * 7, 512), (128 * 7 * 7, 2048)]
CFG = {"weight": {"enable": True, "type": "minmax_channel", "args": {"n_bits": 4, "signed": True, "ch_axis": 0}},
       "input": {"enable": True, "type": "minmax_tensor", "args": {"n_bits": 4, "signed": False}},
       "exclude_layers": [], "override_options": [], "momentum": 0.1}


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int16)


def _same(a, b, what):
    if not torch.equal(_bits(a), _bits(b)) if a.is_floating_point() else not torch.equal(a, b):
        bad = (_bits(a) != _bits(b)) if a.is_floating_point() else (a != b)
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} differ")


def raw_case(rows, ch, dtype, resid, relu, enc, lo, hi, special=None, seed=0):
    from dlmc_quant_b200 import _lib
    from dlmc_quant_b200 import functional as F
    from dlmc_quant_b200 import qgemm as Q
    from dlmc_quant_b200.fuse import _bnq_ws
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(seed)
    x = (torch.randn(rows, ch, generator=g, device=dev) * 2).to(dtype)
    idn = (torch.randn(rows, ch, generator=g, device=dev)).to(dtype) if resid else None
    gamma = torch.rand(ch, generator=g, device=dev) + 0.5
    beta = torch.randn(ch, generator=g, device=dev) * 0.3
    rmean = torch.randn(ch, generator=g, device=dev) * 0.2
    rvar = torch.rand(ch, generator=g, device=dev) + 0.5
    scale = torch.tensor([2.5 / max(hi, 1)], device=dev)
    offset = torch.tensor([0.07], device=dev)
    if special == "values":
        flat = x.view(-1)
        n = flat.numel()
        idx = torch.randperm(n, generator=g, device=dev)[: max(8, n // 50)]
        vals = torch.tensor([float("nan"), float("inf"), -float("inf"), 3.0e6, -2.0e6, 2.0 ** 21],
                            device=dev).to(dtype)
        flat[idx] = vals[torch.arange(idx.numel(), device=dev) % vals.numel()]
    if special == "tiny_scale":
        scale = torch.tensor([2.0 ** -45], device=dev)            # outside the fast-division domain
    gq = 1 / math.sqrt(rows * ch * hi)
    flags = (2 if relu else 0) | (4 if resid else 0)
    desc = _lib.BnqDesc(rows, ch, F._dtype_code(x), flags, 1e-5, 0.1)
    qp = _lib.QParams(_lib.FORM_AFFINE, lo, hi, gq, scale.data_ptr(), offset.data_ptr())
    a1, a2 = torch.empty_like(x), torch.empty_like(x)
    st1, st2 = torch.empty(2, ch, device=dev), torch.empty(2, ch, device=dev)
    codes = torch.empty(rows, ch, dtype=torch.uint8, device=dev)
    h = _lib.lib()
    ws, nws = _bnq_ws(dev, desc)
    s = F._stream_ptr()
    _lib.check(h.dlmcq_bnq_forward_codes(F._ptr(x), F._ptr(idn), F._ptr(gamma), F._ptr(beta), F._ptr(rmean),
                                         F._ptr(rvar), st1.data_ptr(), st1.data_ptr() + 4 * ch, F._ptr(a1),
                                         F._ptr(codes), C.byref(desc), C.byref(qp), enc, F._ptr(ws), nws, s))
    _lib.check(h.dlmcq_bnq_forward(F._ptr(x), F._ptr(idn), F._ptr(gamma), F._ptr(beta), F._ptr(rmean), F._ptr(rvar),
                                   st2.data_ptr(), st2.data_ptr() + 4 * ch, F._ptr(a2), None, C.byref(desc), None,
                                   F._ptr(ws), nws, s))
    want = Q.codes_forward(a1, scale, offset, lo, hi, _lib.FORM_AFFINE, gq, encoding=enc)
    # codes alone (no plain output) must be the same bytes
    codes2 = torch.empty_like(codes)
    _lib.check(h.dlmcq_bnq_forward_codes(F._ptr(x), F._ptr(idn), F._ptr(gamma), F._ptr(beta), F._ptr(rmean),
                                         F._ptr(rvar), st1.data_ptr(), st1.data_ptr() + 4 * ch, None,
                                         F._ptr(codes2), C.byref(desc), C.byref(qp), enc, F._ptr(ws), nws, s))
    torch.cuda.synchronize()
    _same(a1, a2, "plain output vs dlmcq_bnq_forward")
    _same(st1, st2, "save_mean / save_invstd vs dlmcq_bnq_forward")
    _same(codes, want, "codes vs dlmcq_codes_forward(a)")
    _same(codes2, want, "codes without a plain output vs dlmcq_codes_forward(a)")
    return {"distinct_codes": int(torch.unique(codes).numel())}


def _resnet(kind, batch=32, seed=2333):
    import torchvision
    from dlmc_quant_b200 import quantize_model
    torch.manual_seed(seed)
    m = torchvision.models.resnet50() if kind == "r50" else torchvision.models.resnet18()
    m = m.cuda().to(memory_format=torch.channels_last)
    quantize_model(m, copy.deepcopy(CFG), None)
    x = torch.randn(batch, 3, 224 if kind == "r50" else 96, 224 if kind == "r50" else 96,
                    device="cuda").contiguous(memory_format=torch.channels_last)
    m.eval()
    with torch.no_grad():
        m(x)                                                      # lazy observer init
    return m, x


class _Count:
    """Counts the stand-alone activation code passes (qgemm.codes_forward on an input) and records which modules ran on
    the code path (qgemm.forward_codes)."""

    def __init__(self, Q):
        self.Q, self.codes, self.ran = Q, 0, []
        self.orig_codes, self.orig_fwd = Q.codes_forward, Q.forward_codes

    def __enter__(self):
        def codes(*a, **k):
            self.codes += 1
            return self.orig_codes(*a, **k)

        def fwd(mod, *a, **k):
            self.ran.append(mod)
            return self.orig_fwd(mod, *a, **k)
        self.Q.codes_forward, self.Q.forward_codes = codes, fwd
        return self

    def __exit__(self, *exc):
        self.Q.codes_forward, self.Q.forward_codes = self.orig_codes, self.orig_fwd


def _arms(m, x, convolutions=True, encoding=None):
    """(logits with codes handed over, logits with every consumer quantising the fused plain output, counters)."""
    from dlmc_quant_b200 import fuse
    from dlmc_quant_b200 import qgemm as Q
    fuse.fuse_bn_act_quant(m)
    Q.enable_code_gemm(m, encoding=encoding, convolutions=convolutions)
    with torch.no_grad():
        m(x)                                                      # weight codes, epilogue vectors
        with _Count(Q) as ca:
            ya = m(x)
        orig = fuse._consumer_q
        fuse._consumer_q = lambda *a, **k: None
        try:
            with _Count(Q) as cb:
                yb = m(x)
        finally:
            fuse._consumer_q = orig
    torch.cuda.synchronize()
    return ya, yb, ca, cb


def model_r50_case(convolutions=True, encoding=None):
    torch.backends.cudnn.deterministic = True
    m, x = _resnet("r50")
    ya, yb, ca, cb = _arms(m, x, convolutions, encoding)
    _same(ya, yb, "logits: codes from the producer vs codes_forward of the plain output")
    handed = cb.codes - ca.codes
    want = 47 if convolutions else 31
    assert handed == want, f"{handed} sites received codes from their producer, want {want}"
    assert len(ca.ran) == len(cb.ran), (len(ca.ran), len(cb.ran))
    if convolutions:
        ds = [m.layer2[0].downsample[0], m.layer3[0].downsample[0], m.layer4[0].downsample[0]]
        assert all(any(r is d for r in ca.ran) for d in ds), "a stride-2 downsample convolution left the code path"
        assert len(ca.ran) == 53, len(ca.ran)
    if encoding is not None:
        assert all(mod.__dict__["_code_gemm"].encoding == encoding for mod in ca.ran)
    return {"codes_from_producer": handed, "layers_on_code_path": len(ca.ran), "standalone_code_passes": ca.codes}


def model_r18_case():
    torch.backends.cudnn.deterministic = True
    m, x = _resnet("r18", batch=8)
    ya, yb, ca, cb = _arms(m, x)
    _same(ya, yb, "ResNet-18 logits")
    handed = cb.codes - ca.codes
    assert handed == 15, handed          # 8 x conv2 (bn1 -> conv2) + 7 x conv1 of the blocks after the first
    return {"codes_from_producer": handed}


def _seq(signed, relu, dtype):
    from dlmc_quant_b200 import quantize_model
    nn = torch.nn
    torch.manual_seed(5)
    layers = [nn.BatchNorm1d(256)] + ([nn.ReLU()] if relu else []) + [nn.Linear(256, 128)]
    net = nn.Sequential(*layers).cuda()
    cfg = copy.deepcopy(CFG)
    cfg["input"]["args"]["signed"] = signed
    quantize_model(net, cfg, None)
    with torch.no_grad():
        net[0].running_mean.normal_(0, 0.3)
        net[0].running_var.uniform_(0.5, 1.5)
    net.eval()
    x = (torch.randn(384, 256, device="cuda") * 2).to(dtype)
    with torch.no_grad():
        net(x.float())
    return net, x


def other_linear_case(signed, relu, dtype):
    from dlmc_quant_b200 import fuse
    from dlmc_quant_b200 import qgemm as Q
    net, x = _seq(signed, relu, dtype)
    q = net[-1]
    assert (q.in_min_val < 0) == signed
    fuse.fuse_bn_act_quant(net)
    assert Q.enable_code_gemm(net) == [str(len(net) - 1)]
    with torch.no_grad():
        net(x)
        with _Count(Q) as ca:
            ya = net(x)
        orig = fuse._consumer_q
        fuse._consumer_q = lambda *a, **k: None
        try:
            with _Count(Q) as cb:
                yb = net(x)
        finally:
            fuse._consumer_q = orig
    torch.cuda.synchronize()
    assert ca.codes == 0 and cb.codes == 1 and len(ca.ran) == 1, (ca.codes, cb.codes, len(ca.ran))
    _same(ya, yb, "BatchNorm1d -> QLinear output")
    return {}


def _fuse_only(m, x):
    from dlmc_quant_b200 import fuse
    h = fuse.fuse_bn_act_quant(m)
    with torch.no_grad():
        y = m(x)
    h.unfuse()
    return y


def fallback_unswitched_case():
    """conv2 (3x3) not switched without convolutions=True: bn1 hands it the fp32 a_q, exactly as fuse alone."""
    from dlmc_quant_b200 import fuse
    from dlmc_quant_b200 import qgemm as Q
    torch.backends.cudnn.deterministic = True
    m, x = _resnet("r50", batch=8)
    conv2 = m.layer1[0].conv2
    seen = []
    orig = conv2.forward_prequantized
    conv2.forward_prequantized = lambda aq: (seen.append(aq.dtype), orig(aq))[1]
    fuse.fuse_bn_act_quant(m)
    Q.enable_code_gemm(m)
    with torch.no_grad():
        m(x)
    assert seen and seen[-1] == torch.float32, seen
    return {}


def fallback_unusable_case():
    """A switched consumer with a non-zero weight offset is unusable: its producer hands over a_q as fuse alone does,
    and the outputs equal fuse alone's."""
    from dlmc_quant_b200 import fuse
    from dlmc_quant_b200 import qgemm as Q
    net, x = _seq(False, True, torch.float32)
    with torch.no_grad():
        net[-1].wt_offset.add_(0.01)                         # per-channel offsets, now non-zero
        want = _fuse_only(net, x)
        fuse.fuse_bn_act_quant(net)
        Q.enable_code_gemm(net)
        with _Count(Q) as c:
            got = net(x)
    torch.cuda.synchronize()
    assert net[-1].__dict__["_code_gemm"].usable is False and not c.ran
    _same(got, want, "unusable consumer vs fuse alone")
    return {}


def fallback_train_autograd_case():
    """Train mode and autograd: no codes, outputs equal fuse alone's."""
    from dlmc_quant_b200 import fuse
    from dlmc_quant_b200 import qgemm as Q
    torch.backends.cudnn.deterministic = True
    m, x = _resnet("r18", batch=4)
    ref = copy.deepcopy(m)
    fuse.fuse_bn_act_quant(m)
    Q.enable_code_gemm(m, convolutions=True)
    with _Count(Q) as c:
        y_grad = m(x)                                            # eval, autograd on
    want_grad = _fuse_only(ref, x)
    _same(y_grad.detach(), want_grad, "eval under autograd vs fuse alone")
    m.train()
    ref.train()
    m_state = copy.deepcopy(ref.state_dict())
    with torch.no_grad():
        y_train = m(x)
    ref.load_state_dict(m_state)
    want_train = _fuse_only(ref, x)
    torch.cuda.synchronize()
    assert not c.ran
    _same(y_train, want_train, "train mode vs fuse alone")
    return {}


def toggles_case():
    """Both switch orders give the same logits; disable_code_gemm restores fuse alone, unfuse() restores the code GEMM
    alone - bit for bit."""
    from dlmc_quant_b200 import fuse
    from dlmc_quant_b200 import qgemm as Q
    torch.backends.cudnn.deterministic = True
    m, x = _resnet("r50", batch=8)
    m2 = copy.deepcopy(m)
    fuse_only = _fuse_only(copy.deepcopy(m), x)
    c = copy.deepcopy(m)
    Q.enable_code_gemm(c, convolutions=True)
    with torch.no_grad():
        code_only = c(x)
    h1 = fuse.fuse_bn_act_quant(m)
    Q.enable_code_gemm(m, convolutions=True)
    Q.enable_code_gemm(m2, convolutions=True)
    h2 = fuse.fuse_bn_act_quant(m2)
    with torch.no_grad():
        y1, y2 = m(x), m2(x)
        _same(y1, y2, "fuse then enable vs enable then fuse")
        Q.disable_code_gemm(m)
        _same(m(x), fuse_only, "after disable_code_gemm vs fuse alone")
        h2.unfuse()
        _same(m2(x), code_only, "after unfuse() vs the code GEMM alone")
    del h1
    return {}


def graph_case():
    """One eval forward of the combined model captured in a CUDA graph after a warm-up: replay == eager."""
    from dlmc_quant_b200 import fuse
    from dlmc_quant_b200 import qgemm as Q
    torch.backends.cudnn.deterministic = True
    m, x = _resnet("r50", batch=8)
    fuse.fuse_bn_act_quant(m)
    Q.enable_code_gemm(m, convolutions=True)
    with torch.no_grad():
        eager = m(x)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            m(x)
        torch.cuda.current_stream().wait_stream(s)
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            out = m(x)
        gr.replay()
    torch.cuda.synchronize()
    _same(out, eager, "graph replay vs eager")
    return {}


def build_cases():
    cases = []
    combos = [(I8, 0, 15, True), (I8, 0, 255, True), (I8, -8, 7, False), (E4M3, 0, 15, True), (E4M3, -16, 15, False)]
    for dtype, dn in ((torch.float32, "f32"), (torch.bfloat16, "bf16")):
        for resid in (False, True):
            for enc, lo, hi, relu in combos:
                en = "i8" if enc == I8 else "e4m3"
                for rows, ch in ((37, 64), (162, 256)):
                    cases.append((f"raw_{dn}_{en}_{lo}_{hi}_{'res' if resid else 'plain'}_{rows}x{ch}", raw_case,
                                  dict(rows=rows, ch=ch, dtype=dtype, resid=resid, relu=relu, enc=enc, lo=lo, hi=hi)))
                if relu and hi == 15:
                    cases.append((f"raw_{dn}_{en}_{lo}_{hi}_{'res' if resid else 'plain'}_norelu_1000x128", raw_case,
                                  dict(rows=1000, ch=128, dtype=dtype, resid=resid, relu=False, enc=enc, lo=lo, hi=hi)))
        for i, (rows, ch) in enumerate(R50_SITES):
            for resid in (False, True):
                enc, lo, hi, relu = combos[(i + resid) % len(combos)]
                en = "i8" if enc == I8 else "e4m3"
                cases.append((f"raw_r50_{dn}_{en}_{lo}_{hi}_{'res' if resid else 'plain'}_{rows}x{ch}", raw_case,
                              dict(rows=rows, ch=ch, dtype=dtype, resid=resid, relu=relu, enc=enc, lo=lo, hi=hi,
                                   seed=i)))
        for special in ("values", "tiny_scale"):
            for enc, lo, hi, relu in combos:
                en = "i8" if enc == I8 else "e4m3"
                cases.append((f"raw_generic_{special}_{dn}_{en}_{lo}_{hi}", raw_case,
                              dict(rows=4099, ch=64, dtype=dtype, resid=True, relu=relu, enc=enc, lo=lo, hi=hi,
                                   special=special)))
    cases.append(("model_r50_convolutions", model_r50_case, {}))
    cases.append(("model_r50_pointwise_only", model_r50_case, dict(convolutions=False)))
    cases.append(("model_r50_forced_i8", model_r50_case, dict(encoding=I8)))
    cases.append(("model_r18", model_r18_case, {}))
    for signed, relu in ((False, True), (True, False)):
        for dtype, dn in ((torch.float32, "f32"), (torch.bfloat16, "bf16")):
            cases.append((f"other_linear_{'signed' if signed else 'unsigned'}_{dn}", other_linear_case,
                          dict(signed=signed, relu=relu, dtype=dtype)))
    cases.append(("fallback_unswitched", fallback_unswitched_case, {}))
    cases.append(("fallback_unusable", fallback_unusable_case, {}))
    cases.append(("fallback_train_autograd", fallback_train_autograd_case, {}))
    cases.append(("toggles", toggles_case, {}))
    cases.append(("graph", graph_case, {}))
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
