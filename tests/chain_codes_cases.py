"""Case runner for the chained code layer (dlmcq_qgemm_codes / dlmcq_qconv_codes: code GEMM or convolution -> eval
BatchNorm -> ReLU -> the next layer's input codes in one kernel) and its wiring (fuse.chain_spec, qgemm.forward_codes
with a tail), executed in its OWN process by tests/test_gpu_chain_codes.py: the kernel is a tcgen05 / TMA pipeline
whose failure mode is a trap that poisons the CUDA context.  Prints one JSON report on the last line.

Bars, all byte for byte / bit for bit:
  * raw entries == the two-kernel chain they replace: dlmcq_qgemm / dlmcq_qconv (out_dtype T) followed by
    dlmcq_bnq_forward_codes of that output;
  * on a small subset, == an independent restatement (oracle/restate.py::code_gemm, tests/qconv_oracle.py::code_conv,
    then the eval BatchNorm with restate.fma_f32 and an IEEE sqrt, then the restated AFFINE quantizer), and a variant
    with BatchNorm folded into alpha / beta differs (the test can see a folding);
  * models: the same logits with the chain on and off (fuse.chain_spec patched out), with the chained sites, the
    fp32-output layer calls and the fused BatchNorm code passes counted."""
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
CFG = {"weight": {"enable": True, "type": "minmax_channel", "args": {"n_bits": 4, "signed": True, "ch_axis": 0}},
       "input": {"enable": True, "type": "minmax_tensor", "args": {"n_bits": 4, "signed": False}},
       "exclude_layers": [], "override_options": [], "momentum": 0.1}
B = 128
# every distinct chained-site geometry of torchvision ResNet-50 at batch 128: conv1 (1x1, GEMM) as (m, k, n) and
# conv2 (3x3, pad 1) as (h, cin, stride); the first block of a stage reads the previous stage's resolution and width
R50_CONV1 = [(B * 56 * 56, 64, 64), (B * 56 * 56, 256, 64), (B * 56 * 56, 256, 128), (B * 28 * 28, 512, 128),
             (B * 28 * 28, 512, 256), (B * 14 * 14, 1024, 256), (B * 14 * 14, 1024, 512), (B * 7 * 7, 2048, 512)]
R50_CONV2 = [(56, 64, 1), (56, 128, 2), (28, 128, 1), (28, 256, 2), (14, 256, 1), (14, 512, 2), (7, 512, 1)]
# (producer encoding, consumer encoding, consumer lo, hi, relu): the consumer's range must fit its encoding
COMBOS = [(I8, I8, 0, 15, True), (E4M3, E4M3, 0, 15, True), (I8, E4M3, -16, 15, False), (E4M3, I8, 0, 255, True),
          (I8, I8, -8, 7, False), (E4M3, I8, -8, 7, True)]


def _same(a, b, what):
    if not torch.equal(a, b):
        bad = a != b
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} differ")


def _bytes(v, enc):
    if enc == I8:
        return (v.to(torch.int64) & 0xFF).to(torch.uint8)
    return v.to(torch.float32).to(torch.float8_e4m3fn).view(torch.uint8)


def _operands(shape_a, n, k_w, enc, g, pattern="random"):
    """Producer operands: activation codes (unsigned 4-bit, or unsigned 8-bit on I8), weight codes (signed 4-bit, or
    -16 .. 16 on E4M3 with pattern "saturated")."""
    dev = torch.device("cuda")
    a_hi = 15 if enc == E4M3 else 255 if pattern == "saturated" else 15
    w_hi = 16 if enc == E4M3 else 127
    if pattern == "saturated":
        ca = torch.full(shape_a, a_hi, dtype=torch.int64, device=dev)
        cw = torch.full(k_w, -w_hi if enc == E4M3 else -128, dtype=torch.int64, device=dev)
    else:
        ca = torch.randint(0, a_hi + 1, shape_a, generator=g, device=dev)
        cw = torch.randint(-7, 8, k_w, generator=g, device=dev)
    return ca, cw, _bytes(ca, enc), _bytes(cw, enc)


def _bn(n, g, special=None):
    dev = torch.device("cuda")
    gamma = torch.rand(n, generator=g, device=dev) + 0.5
    beta = torch.randn(n, generator=g, device=dev) * 0.3
    rmean = torch.randn(n, generator=g, device=dev) * 0.2
    rvar = torch.rand(n, generator=g, device=dev) + 0.5
    if special == "bn":
        gamma[0::7] = 0.0
        gamma[1::7] *= -1
        rvar[2::7] = 1e-30
        rvar[3::7] = 1e30
        rmean[4] = float("nan")
        beta[5::7] = 3.0e6                                       # constants outside the packed path's domain
    return gamma, beta, rmean, rvar


def _two_kernel(y, n, bn, relu, scale, offset, lo, hi, gq, enc_out):
    """dlmcq_bnq_forward_codes of the layer output y (rows x n, channels innermost): the chain being replaced."""
    from dlmc_quant_b200 import _lib
    from dlmc_quant_b200 import functional as F
    from dlmc_quant_b200.fuse import _bnq_ws
    gamma, beta, rmean, rvar = bn
    rows = y.numel() // n
    desc = _lib.BnqDesc(rows, n, F._dtype_code(y), 2 if relu else 0, 1e-5, 0.1)
    qp = _lib.QParams(_lib.FORM_AFFINE, lo, hi, gq, scale.data_ptr(), offset.data_ptr())
    st = torch.empty(2, n, device=y.device)
    codes = torch.empty(rows, n, dtype=torch.uint8, device=y.device)
    ws, nws = _bnq_ws(y.device, desc)
    _lib.check(_lib.lib().dlmcq_bnq_forward_codes(F._ptr(y), None, F._ptr(gamma), F._ptr(beta), F._ptr(rmean),
                                                  F._ptr(rvar), st.data_ptr(), st.data_ptr() + 4 * n, None,
                                                  F._ptr(codes), C.byref(desc), C.byref(qp), enc_out, F._ptr(ws), nws,
                                                  F._stream_ptr()))
    return codes


def _consumer(hi, g, special):
    dev = torch.device("cuda")
    scale = torch.tensor([2.5 / max(hi, 1)], device=dev)
    if special == "tiny_scale":
        scale = torch.tensor([2.0 ** -45], device=dev)              # outside the fast-division domain
    offset = torch.tensor([0.07], device=dev)
    return scale, offset


def raw_gemm_case(m, k, n, dtype, combo, special=None, seed=0, pattern="random"):
    from dlmc_quant_b200 import qgemm as Q
    enc_in, enc_out, lo, hi, relu = combo
    g = torch.Generator(device="cuda").manual_seed(seed)
    _, _, a, w = _operands((m, k), n, (n, k), enc_in, g, pattern)
    alpha = torch.rand(n, generator=g, device="cuda") * 0.02 + 0.005
    beta = torch.randn(n, generator=g, device="cuda")
    if pattern == "saturated":
        alpha.fill_(1.0)
        beta.zero_()
    bn = _bn(n, g, special)
    scale, offset = _consumer(hi, g, special)
    gq = 1 / math.sqrt(m * n * hi)
    y = Q.qgemm(a, w, alpha, beta, out_dtype=dtype, encoding=enc_in)
    want = _two_kernel(y, n, bn, relu, scale, offset, lo, hi, gq, enc_out)
    t = Q.bnq_tail(bn[2], bn[3], scale, offset, lo, hi, gq, bn[0], bn[1], 1e-5, relu, dtype, enc_out)
    got = Q.qgemm_codes(a, w, alpha, beta, t, encoding=enc_in)
    torch.cuda.synchronize()
    _same(got, want, "qgemm_codes vs qgemm + bnq_forward_codes")
    return {"distinct_codes": int(torch.unique(got).numel()), "max_abs_y": float(y.float().abs().nan_to_num().max())}


def raw_conv_case(batch, h, cin, n, stride, dtype, combo, ksize=3, pad=1, special=None, seed=0):
    from dlmc_quant_b200 import qgemm as Q
    enc_in, enc_out, lo, hi, relu = combo
    g = torch.Generator(device="cuda").manual_seed(seed)
    _, _, a, w = _operands((batch, h, h, cin), n, (n, ksize, ksize, cin), enc_in, g)
    alpha = torch.rand(n, generator=g, device="cuda") * 0.02 + 0.005
    beta = torch.randn((ksize + 1) ** 4, n, generator=g, device="cuda")     # every border class differs
    bn = _bn(n, g, special)
    scale, offset = _consumer(hi, g, special)
    y = Q.qconv(a, w, alpha, beta, stride, pad, out_dtype=dtype, encoding=enc_in)
    gq = 1 / math.sqrt(y.numel() * hi)
    want = _two_kernel(y, n, bn, relu, scale, offset, lo, hi, gq, enc_out).view(y.shape)
    t = Q.bnq_tail(bn[2], bn[3], scale, offset, lo, hi, gq, bn[0], bn[1], 1e-5, relu, dtype, enc_out)
    got = Q.qconv_codes(a, w, alpha, beta, t, stride, pad, encoding=enc_in)
    torch.cuda.synchronize()
    _same(got, want, "qconv_codes vs qconv + bnq_forward_codes")
    return {"distinct_codes": int(torch.unique(got).numel())}


def _restated_tail(v, bn, relu, scale, offset, lo, hi, gq, fold=False):
    """Eval BatchNorm with restate.fma_f32 and an IEEE sqrt, ReLU, then the restated AFFINE quantizer -> codes."""
    from oracle import restate as R
    gamma, beta, rmean, rvar = (t.cpu() for t in bn)
    invstd = torch.ones_like(rvar) / torch.sqrt(rvar + torch.tensor(1e-5, dtype=torch.float32))
    a = gamma * invstd
    z = R.fma_f32(v - rmean, a.expand_as(v), beta.expand_as(v))
    act = torch.relu(z) if relu else z
    return R.fq_affine_codes(act, scale.cpu(), offset.cpu(), lo, hi, gq)


def restate_case(conv):
    """A small GEMM (1x1) and a padded 3x3 convolution restated independently, byte for byte; then a producer with
    BatchNorm folded into alpha / beta must differ on the same inputs.  The inputs make a folding visible: a layer bias
    of ~100 that the running mean cancels (the unchained layer rounds v at |v| ~ 100 before subtracting), a steep
    gamma * invstd (~25) and an 8-bit consumer."""
    from dlmc_quant_b200 import qgemm as Q
    from oracle import restate as R
    from tests import qconv_oracle as O
    g = torch.Generator(device="cuda").manual_seed(11)
    n, lo, hi, relu = 64, 0, 255, True
    m_a, o_a = torch.tensor(0.0625), torch.tensor(0.11)
    m_w = torch.rand(n, generator=g, device="cuda").cpu() * 0.01 + 0.004
    bias = (torch.rand(n, generator=g, device="cuda") + 99.5).cpu()
    if conv:
        ca, cw, a, w = _operands((4, 12, 12, 64), n, (n, 3, 3, 64), I8, g)
        v = O.code_conv(ca.cpu().permute(0, 3, 1, 2), cw.cpu().permute(0, 3, 1, 2), m_a, o_a, 0.0, m_w, bias,
                        padding=1)
        v = v.permute(0, 2, 3, 1).reshape(-1, n)
        alpha, beta = Q.qconv_prepare(w, (m_a.reshape(1).cuda(), o_a.reshape(1).cuda(), 0, 15, 0, 0.0),
                                      (m_w.cuda(), -7, 7, 3, 0.0), bias.cuda(), I8)
    else:
        ca, cw, a, w = _operands((1000, 128), n, (n, 128), I8, g)
        v = R.code_gemm(ca.cpu(), cw.cpu(), m_a, o_a, 0.0, m_w, bias)
        alpha, beta = Q.qgemm_prepare(w, (m_a.reshape(1).cuda(), o_a.reshape(1).cuda(), 0, 15, 0, 0.0),
                                      (m_w.cuda(), -7, 7, 3, 0.0), bias.cuda(), I8)
    bn = list(_bn(n, g))
    bn[2] = bias.cuda() + torch.randn(n, generator=g, device="cuda") * 0.05      # running mean cancels the bias
    bn[3] = torch.rand(n, generator=g, device="cuda") * 1e-3 + 1e-3               # invstd ~ 25
    scale, offset = torch.tensor([8.0 / hi], device="cuda"), torch.tensor([0.07], device="cuda")
    gq = 1 / math.sqrt(v.numel() * hi)
    want = _restated_tail(v, bn, relu, scale, offset, lo, hi, gq).to(torch.uint8)
    t = Q.bnq_tail(bn[2], bn[3], scale, offset, lo, hi, gq, bn[0], bn[1], 1e-5, relu, torch.float32, I8)
    got = (Q.qconv_codes(a, w, alpha, beta, t, 1, 1) if conv else Q.qgemm_codes(a, w, alpha, beta, t)).reshape(-1, n)
    # negative control: BatchNorm folded into the producer's alpha / beta, quantized directly
    gamma, bb, rmean, rvar = bn
    sc = gamma / torch.sqrt(rvar + 1e-5)
    t_id = Q.bnq_tail(torch.zeros_like(rmean), torch.ones_like(rvar), scale, offset, lo, hi, gq, None, None, 0.0, relu,
                      torch.float32, I8)                         # the identity BatchNorm: invstd = 1 exactly
    a2, b2 = alpha * sc, (beta - rmean) * sc + bb
    folded = (Q.qconv_codes(a, w, a2, b2, t_id, 1, 1) if conv else Q.qgemm_codes(a, w, a2, b2, t_id)).reshape(-1, n)
    torch.cuda.synchronize()
    _same(got.cpu(), want, "chained codes vs the independent restatement")
    differ = int((folded != got).sum())
    assert differ > 0, "a BatchNorm folded into alpha / beta gave the same codes: the test cannot see a folding"
    return {"folded_codes_differ": differ}


# ---------------------------------------------------------------------------------------------------------------
# models
# ---------------------------------------------------------------------------------------------------------------
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
    """Chained sites (qgemm.forward_codes with a tail), layer calls with an fp32 / bf16 output (qgemm.qgemm /
    qgemm.qconv) and fused BatchNorm producers that wrote codes (fuse._bn_act_codes)."""

    def __init__(self):
        from dlmc_quant_b200 import fuse
        from dlmc_quant_b200 import qgemm as Q
        self.Q, self.fuse = Q, fuse
        self.chained = self.plain = self.bnq_codes = 0
        self.orig = (Q.forward_codes, Q.qgemm, Q.qconv, fuse._bn_act_codes)

    def __enter__(self):
        fwd, qg, qc, bac = self.orig

        def forward_codes(mod, *a, **k):
            self.chained += k.get("tail") is not None
            return fwd(mod, *a, **k)

        def plain(fn):
            def f(*a, **k):
                self.plain += 1
                return fn(*a, **k)
            return f

        def bn_act_codes(*a, **k):
            r = bac(*a, **k)
            self.bnq_codes += r is not None
            return r
        self.Q.forward_codes, self.Q.qgemm, self.Q.qconv = forward_codes, plain(qg), plain(qc)
        self.fuse._bn_act_codes = bn_act_codes
        return self

    def __exit__(self, *exc):
        self.Q.forward_codes, self.Q.qgemm, self.Q.qconv, self.fuse._bn_act_codes = self.orig


def _on_off(m, x):
    """(logits chained, logits with fuse.chain_spec patched out, counters of each)."""
    from dlmc_quant_b200 import fuse
    with torch.no_grad():
        m(x)
        with _Count() as con:
            y_on = m(x)
        orig = fuse.chain_spec
        fuse.chain_spec = lambda *a, **k: None
        try:
            with _Count() as coff:
                y_off = m(x)
        finally:
            fuse.chain_spec = orig
    torch.cuda.synchronize()
    return y_on, y_off, con, coff


def model_case(kind, convolutions=True):
    from dlmc_quant_b200 import fuse
    from dlmc_quant_b200 import qgemm as Q
    torch.backends.cudnn.deterministic = True
    m, x = _resnet(kind, batch=32 if kind == "r50" else 8)
    fuse.fuse_bn_act_quant(m)
    Q.enable_code_gemm(m, convolutions=convolutions)
    y_on, y_off, con, coff = _on_off(m, x)
    _same(y_on.view(torch.int32), y_off.view(torch.int32), "logits with the chain on vs off")
    want = (32 if kind == "r50" else 8) if convolutions else 0
    assert con.chained == want and coff.chained == 0, (con.chained, coff.chained)
    if kind == "r50" and convolutions:
        assert (coff.plain, con.plain) == (53, 21), (coff.plain, con.plain)
        assert con.bnq_codes == 15, con.bnq_codes                  # the residual sites bn3 (+ identity) -> relu
    return {"chained": con.chained, "layer_calls_plain_on": con.plain, "layer_calls_plain_off": coff.plain,
            "bnq_codes_on": con.bnq_codes, "bnq_codes_off": coff.bnq_codes}


def _stack(kind, dtype, consumer_enabled=True, n_mid=64, per_channel_consumer=False):
    from dlmc_quant_b200 import quantize_model
    nn = torch.nn
    torch.manual_seed(7)
    cfg = copy.deepcopy(CFG)
    if kind == "conv":
        net = nn.Sequential(nn.Conv2d(64, 64, 3, padding=1), nn.BatchNorm2d(64), nn.ReLU(), nn.Conv2d(64, 128, 1),
                            nn.BatchNorm2d(128), nn.ReLU(), nn.Conv2d(128, 64, 3, padding=1))
        x = torch.randn(8, 64, 20, 20, device="cuda").contiguous(memory_format=torch.channels_last)
        net = net.cuda().to(memory_format=torch.channels_last)
    elif kind == "linear4d":
        # a Linear on a 4-D input writes a contiguous [B, C, H, n]; BatchNorm2d normalises C: not a fusable layout
        net = nn.Sequential(nn.Linear(64, 64), nn.BatchNorm2d(16), nn.ReLU(), nn.Linear(64, 32)).cuda()
        x = torch.randn(8, 16, 5, 64, device="cuda")
    else:
        net = nn.Sequential(nn.Linear(256, n_mid), nn.BatchNorm1d(n_mid), nn.ReLU(), nn.Linear(n_mid, 32)).cuda()
        x = torch.randn(384, 256, device="cuda")
    if per_channel_consumer:
        cfg["override_options"] = [{"layers": [f"^{len(net) - 1}$"],
                                    "options": {"input": {"type": "minmax_channel"}}}]
    quantize_model(net, cfg, None)
    if per_channel_consumer:
        assert net[-1].in_scale.numel() > 1, "the consumer's input quantizer is not per-channel"
    with torch.no_grad():
        for bn in (mm for mm in net if isinstance(mm, (nn.BatchNorm1d, nn.BatchNorm2d))):
            bn.running_mean.normal_(0, 0.3)
            bn.running_var.uniform_(0.5, 1.5)
    net.eval()
    with torch.no_grad():
        net(x)
    if not consumer_enabled:
        net[-1].qconfig['input']['enable'] = False
    return net, x.to(dtype)


def stack_case(kind, dtype, want, consumer_enabled=True, n_mid=64, convolutions=True, per_channel_consumer=False):
    from dlmc_quant_b200 import fuse
    from dlmc_quant_b200 import qgemm as Q
    net, x = _stack(kind, dtype, consumer_enabled, n_mid, per_channel_consumer)
    fuse.fuse_bn_act_quant(net)
    Q.enable_code_gemm(net, convolutions=convolutions)
    y_on, y_off, con, _ = _on_off(net, x)
    _same(y_on, y_off, "stack output with the chain on vs off")
    assert con.chained == want, (con.chained, want)
    return {"chained": con.chained}


def tail_refusals_case():
    """bnq_tail and the wrappers refuse BatchNorm / quantizer tensors the kernel would read out of bounds."""
    from dlmc_quant_b200 import qgemm as Q
    from dlmc_quant_b200._lib import DlmcqError
    g = torch.Generator(device="cuda").manual_seed(3)
    _, _, a, w = _operands((256, 64), 64, (64, 64), I8, g)
    alpha, beta = torch.ones(64, device="cuda"), torch.zeros(64, device="cuda")
    ones, s, o = torch.ones(64, device="cuda"), torch.ones(1, device="cuda"), torch.zeros(1, device="cuda")
    bad = [lambda: Q.bnq_tail(ones, torch.ones(48, device="cuda"), s, o, 0, 15, 0.1),
           lambda: Q.bnq_tail(ones, ones, s, o, 0, 15, 0.1, gamma=torch.ones(64)),
           lambda: Q.bnq_tail(ones, ones.double(), s, o, 0, 15, 0.1),
           lambda: Q.bnq_tail(ones, ones, torch.ones(2, device="cuda"), o, 0, 15, 0.1),
           lambda: Q.qgemm_codes(a, w, alpha, beta, Q.bnq_tail(ones[:32], ones[:32], s, o, 0, 15, 0.1)),
           lambda: Q.qconv_codes(a.view(4, 8, 8, 64), w.view(64, 1, 1, 64), alpha, torch.zeros(4, 64, device="cuda"),
                                 Q.bnq_tail(ones[:48], ones[:48], s, o, 0, 15, 0.1))]
    for i, f in enumerate(bad):
        try:
            f()
        except DlmcqError:
            continue
        raise AssertionError(f"call {i} was not refused")
    torch.cuda.synchronize()
    return {}


def fallback_train_autograd_case():
    from dlmc_quant_b200 import fuse
    from dlmc_quant_b200 import qgemm as Q
    torch.backends.cudnn.deterministic = True
    m, x = _resnet("r18", batch=4)
    ref = copy.deepcopy(m)
    fuse.fuse_bn_act_quant(m)
    Q.enable_code_gemm(m, convolutions=True)
    fuse.fuse_bn_act_quant(ref)
    with _Count() as c:
        y = m(x)                                                   # eval, autograd on
        m.train()
        with torch.no_grad():
            y_train = m(x)
    with torch.no_grad():
        want = ref(x)
    ref.train()
    torch.cuda.synchronize()
    assert c.chained == 0 and torch.isfinite(y_train).all(), c.chained
    _same(y.detach(), want, "eval under autograd vs fuse alone")
    return {}


def producer_reference_case():
    """The producer on its original path (its code state made unusable): nothing chains, output unchanged."""
    from dlmc_quant_b200 import fuse
    from dlmc_quant_b200 import qgemm as Q
    net, x = _stack("linear", torch.float32)
    fuse.fuse_bn_act_quant(net)
    Q.enable_code_gemm(net)
    with torch.no_grad():
        net[0].wt_offset.add_(0.01)                                # per-channel weight offsets: unusable on codes
        y_on, y_off, con, _ = _on_off(net, x)
    assert con.chained == 0 and net[0].__dict__["_code_gemm"].usable is False
    _same(y_on, y_off, "producer on its original path")
    return {}


def toggles_case():
    from dlmc_quant_b200 import fuse
    from dlmc_quant_b200 import qgemm as Q
    torch.backends.cudnn.deterministic = True
    m, x = _resnet("r50", batch=8)
    m2, fo, co = copy.deepcopy(m), copy.deepcopy(m), copy.deepcopy(m)
    h_fo = fuse.fuse_bn_act_quant(fo)
    Q.enable_code_gemm(co, convolutions=True)
    with torch.no_grad():
        fuse_only, code_only = fo(x), co(x)
    h1 = fuse.fuse_bn_act_quant(m)
    Q.enable_code_gemm(m, convolutions=True)
    Q.enable_code_gemm(m2, convolutions=True)
    h2 = fuse.fuse_bn_act_quant(m2)
    with torch.no_grad():
        with _Count() as c:
            y1, y2 = m(x), m2(x)
        assert c.chained == 64, c.chained
        _same(y1, y2, "fuse then enable vs enable then fuse")
        Q.disable_code_gemm(m)
        _same(m(x), fuse_only, "after disable_code_gemm vs fuse alone")
        h2.unfuse()
        _same(m2(x), code_only, "after unfuse() vs the code GEMM alone")
    del h1, h_fo
    return {}


def graph_case():
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
    f32, bf16 = torch.float32, torch.bfloat16
    for i, (m, k, n) in enumerate(R50_CONV1):
        for dt, dn in ((f32, "f32"), (bf16, "bf16")):
            combo = COMBOS[(2 * i + (dt is bf16)) % len(COMBOS)]
            cases.append((f"raw_r50_conv1_{dn}_{m}x{k}x{n}", raw_gemm_case, dict(m=m, k=k, n=n, dtype=dt, combo=combo,
                                                                                seed=i)))
    for i, (h, cin, s) in enumerate(R50_CONV2):
        for dt, dn in ((f32, "f32"), (bf16, "bf16")):
            combo = COMBOS[(2 * i + 1 + (dt is bf16)) % len(COMBOS)]
            cases.append((f"raw_r50_conv2_{dn}_{h}x{cin}_s{s}", raw_conv_case,
                          dict(batch=B, h=h, cin=cin, n=cin, stride=s, dtype=dt, combo=combo, seed=i)))
    for ci, combo in enumerate(COMBOS):
        for dt, dn in ((f32, "f32"), (bf16, "bf16")):
            tag = f"{dn}_c{ci}"
            cases.append((f"raw_gemm_ragged_{tag}", raw_gemm_case, dict(m=1000, k=96, n=80, dtype=dt, combo=combo)))
            cases.append((f"raw_gemm_n144_{tag}", raw_gemm_case, dict(m=333, k=64, n=144, dtype=dt, combo=combo)))
            cases.append((f"raw_conv_n80_{tag}", raw_conv_case, dict(batch=3, h=11, cin=64, n=80, stride=2,
                                                                     dtype=dt, combo=combo)))
            cases.append((f"raw_conv_c192_{tag}", raw_conv_case, dict(batch=2, h=9, cin=192, n=144, stride=1,
                                                                      dtype=dt, combo=combo, ksize=5, pad=2)))
            for special in ("bn", "tiny_scale"):
                cases.append((f"raw_generic_{special}_gemm_{tag}", raw_gemm_case,
                              dict(m=515, k=64, n=96, dtype=dt, combo=combo, special=special)))
                cases.append((f"raw_generic_{special}_conv_{tag}", raw_conv_case,
                              dict(batch=2, h=10, cin=64, n=64, stride=1, dtype=dt, combo=combo, special=special)))
    for enc, k in ((I8, 8192), (E4M3, 65520)):
        for dt, dn in ((f32, "f32"), (bf16, "bf16")):
            combo = (enc, I8, 0, 255, True) if enc == I8 else (enc, E4M3, -16, 15, False)
            cases.append((f"raw_generic_acc_bound_{'i8' if enc == I8 else 'e4m3'}_{dn}", raw_gemm_case,
                          dict(m=200, k=k, n=32, dtype=dt, combo=combo, pattern="saturated")))
    cases.append(("restate_gemm", restate_case, dict(conv=False)))
    cases.append(("restate_conv", restate_case, dict(conv=True)))
    cases.append(("model_r50", model_case, dict(kind="r50")))
    cases.append(("model_r50_pointwise_only", model_case, dict(kind="r50", convolutions=False)))
    cases.append(("model_r18", model_case, dict(kind="r18")))
    for dt, dn in ((f32, "f32"), (bf16, "bf16")):
        cases.append((f"stack_conv_{dn}", stack_case, dict(kind="conv", dtype=dt, want=2)))
        cases.append((f"stack_linear_{dn}", stack_case, dict(kind="linear", dtype=dt, want=1)))
    cases.append(("fallback_consumer_unswitched", stack_case, dict(kind="conv", dtype=f32, want=0,
                                                                   convolutions=False)))
    cases.append(("fallback_consumer_disabled", stack_case, dict(kind="linear", dtype=f32, want=0,
                                                                 consumer_enabled=False)))
    cases.append(("fallback_n_not_16", stack_case, dict(kind="linear", dtype=f32, want=0, n_mid=72)))
    cases.append(("fallback_consumer_per_channel", stack_case, dict(kind="linear", dtype=f32, want=0,
                                                                    per_channel_consumer=True)))
    cases.append(("fallback_linear_4d_batchnorm2d", stack_case, dict(kind="linear4d", dtype=f32, want=0)))
    cases.append(("tail_refusals", tail_refusals_case, {}))
    cases.append(("fallback_producer_reference", producer_reference_case, {}))
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
