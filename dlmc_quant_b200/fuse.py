"""Activation fake-quant fused into its producer (SURVEY.md 8f row f2): BatchNorm (+ residual add) (+ ReLU) -> the
NEXT quantised layer's input fake-quant, as ONE forward and ONE backward op on channels-last tensors
(csrc/bnq_kernels.cu, C ABI `dlmcq_bnq_forward` / `dlmcq_bnq_backward`).

In the reference the chain is spread over the model definition and the quantised layer:

    out = self.bn(conv_out); out += identity; out = self.relu(out)         # model code (torchvision / model/classification)
    ... QConv2d.forward(out): input = fake_quant(out, in_scale, in_offset)   # modules/base.py:96-102, modules/conv.py:13-19

`fuse_bn_act_quant(model)` - opt-in, after `quantize_model` - rewires residual blocks and nn.Sequential runs so that this
chain runs as the fused op; parameters, buffers and state_dict keys are untouched (BatchNorm modules keep their
class and state, the quantised layers keep in_scale / in_offset), `unfuse()` on the returned handle restores the
original forwards.  Every fused site falls back to the unfused composition whenever the fused kernels do not apply
(tensor not channels-last, channel count not a multiple of the vector width, consumer's quantizer not initialised yet /
disabled / per-channel, cumulative-average BatchNorm), so results never depend on whether fusion happened - only speed.

Semantics (tests/test_gpu_bnq.py): given the BatchNorm output `a`, the fused a_q is bit-identical to this repo's
`fq_forward(a)` (itself bit-identical to the reference chain); BatchNorm's own arithmetic agrees with
`torch.nn.functional.batch_norm` within floating-point reduction tolerance, as any two batch-norm implementations do."""
import ctypes as C
import math
import types

import torch
from torch import nn

from . import _lib
from . import functional as F
from . import qgemm
from ._lib import BNQ_RELU, BNQ_RESIDUAL, BNQ_TRAINING, FORM_AFFINE, BnqDesc, QParams
from .scalar.modules.base import QBase

__all__ = ["bn_act_quant", "BnActQuantFunction", "fuse_bn_act_quant", "FuseHandle", "fusable"]

_ws_cache = {}


def _bnq_ws(device, desc):
    key = (desc.rows, desc.channels, desc.dtype)
    n = _ws_cache.get(key)
    if n is None:
        n = _ws_cache[key] = _lib.lib().dlmcq_bnq_workspace_bytes(C.byref(desc))
    return F._scratch(device, n), n      # no zero contract needed: the bnq kernels use no ticket counters


def _rows_channels(x):
    """(rows, C) when x is a dense channels-last matrix in memory, else None."""
    if x.dim() == 4:
        if x.is_contiguous(memory_format=torch.channels_last):
            return x.shape[0] * x.shape[2] * x.shape[3], x.shape[1]
        return None
    if x.dim() == 2 and x.is_contiguous():
        return x.shape[0], x.shape[1]
    return None


def _rows_channels_ok(rc, dtype):
    return rc is not None and rc[0] != 0 and rc[1] % (4 if dtype is torch.float32 else 8) == 0


def _bn_ok(bn):
    if bn.momentum is None or (not bn.training and bn.running_mean is None):
        return False                                   # cumulative moving average / nothing to normalise with
    if (bn.weight is not None and bn.weight.dtype is not torch.float32) or \
            (bn.running_mean is not None and bn.running_mean.dtype is not torch.float32):
        return False
    return True


def fusable(x, bn, identity=None):
    """Can the fused kernels take this tensor / BatchNorm?  (Cheap host checks only.)"""
    if not (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype in (torch.float32, torch.bfloat16)):
        return False
    if not _rows_channels_ok(_rows_channels(x), x.dtype) or not _bn_ok(bn):
        return False
    if identity is not None and (identity.shape != x.shape or identity.dtype != x.dtype or
                                 identity.stride() != x.stride() or not identity.is_cuda):
        return False
    return True


class BnActQuantFunction(torch.autograd.Function):
    """(a | None, a_q | None) = fused BatchNorm (+identity) (+ReLU) [-> fake-quant with `scale`, `offset`].

    bn_state = (running_mean | None, running_var | None, use_batch_stats, momentum, eps); q = (offset, lo, hi, g) or
    None (no quantizer: plain output only)."""

    @staticmethod
    def forward(ctx, x, gamma, beta, scale, identity, bn_state, q, relu, want_plain):
        rmean, rvar, batch_stats, momentum, eps = bn_state
        rows, ch = _rows_channels(x)
        flags = (BNQ_TRAINING if batch_stats else 0) | (BNQ_RELU if relu else 0) | (BNQ_RESIDUAL if identity is not None else 0)
        desc = BnqDesc(rows, ch, F._dtype_code(x), flags, float(eps), float(momentum))
        dev = x.device
        stats = torch.empty(2, ch, dtype=torch.float32, device=dev)          # save_mean, save_invstd
        a = torch.empty_like(x) if want_plain else None
        aq = torch.empty_like(x) if q is not None else None
        qp = None
        if q is not None:
            offset, lo, hi, g = q
            qp = QParams(FORM_AFFINE, int(lo), int(hi), float(g), scale.data_ptr(), offset.data_ptr())
        with F._on(dev):
            ws, n = _bnq_ws(dev, desc)
            _lib.check(_lib.lib().dlmcq_bnq_forward(
                F._ptr(x), F._ptr(identity), F._ptr(gamma), F._ptr(beta), F._ptr(rmean),
                F._ptr(rvar), stats.data_ptr(), stats.data_ptr() + 4 * ch, F._ptr(a), F._ptr(aq), C.byref(desc),
                C.byref(qp) if qp is not None else None, F._ptr(ws), n, F._stream_ptr()))
        ctx.desc, ctx.q, ctx.has_id = desc, q, identity is not None
        # x is always needed (xhat); the plain output only when z contains the identity (cannot be recomputed from x)
        ctx.save_for_backward(x, gamma, beta, scale, stats, a if identity is not None else None,
                              q[0] if q is not None else None)
        if a is not None and aq is not None:
            return a, aq
        return (a, None) if a is not None else (None, aq)

    @staticmethod
    def backward(ctx, d_a, d_q):
        x, gamma, beta, scale, stats, a_saved, offset = ctx.saved_tensors
        desc, q = ctx.desc, ctx.q
        ch = desc.channels
        dev = x.device

        def like_x(t):
            if t is None:
                return None
            if t.dtype != x.dtype or t.stride() != x.stride():
                t = torch.empty_like(x).copy_(t)
            return t
        d_a, d_q = like_x(d_a), like_x(d_q)
        if d_a is None and d_q is None:
            return (None,) * 9
        need_dx = ctx.needs_input_grad[0]
        dx = torch.empty_like(x) if need_dx else None
        dz = torch.empty_like(x) if ctx.has_id else None
        dgb = torch.empty(2, ch, dtype=torch.float32, device=dev)
        ds = torch.empty(1, dtype=torch.float32, device=dev) if (q is not None and d_q is not None) else None
        qp = None
        if ds is not None:
            _, lo, hi, g = q
            qp = QParams(FORM_AFFINE, int(lo), int(hi), float(g), scale.data_ptr(), offset.data_ptr())
        with F._on(dev):
            ws, n = _bnq_ws(dev, desc)
            _lib.check(_lib.lib().dlmcq_bnq_backward(
                F._ptr(x), F._ptr(a_saved), F._ptr(d_a), F._ptr(d_q if ds is not None else None), F._ptr(gamma), F._ptr(beta),
                stats.data_ptr(), stats.data_ptr() + 4 * ch, F._ptr(dx), F._ptr(dz), dgb.data_ptr(),
                dgb.data_ptr() + 4 * ch, F._ptr(ds), C.byref(desc), C.byref(qp) if qp is not None else None, F._ptr(ws),
                n, F._stream_ptr()))
        dgamma = dgb[0].to(gamma.dtype) if gamma is not None and ctx.needs_input_grad[1] else None
        dbeta = dgb[1].to(beta.dtype) if beta is not None and ctx.needs_input_grad[2] else None
        dscale = ds.reshape(scale.shape).to(scale.dtype) if ds is not None and ctx.needs_input_grad[3] else None
        return dx, dgamma, dbeta, dscale, dz, None, None, None, None


def _consumer_q(consumer, x):
    """(scale, (offset, lo, hi, g)) when `consumer`'s input quantizer can be fused into the producer of x, else None."""
    if not isinstance(consumer, QBase) or type(consumer).forward is not QBase.forward:
        return None
    if not consumer.qconfig['input']['enable'] or not (getattr(consumer, '_host_init', None) or {}).get('in'):
        return None                 # disabled, or the lazy observer init has not run yet (first forward): unfused
    s, off = consumer.in_scale, consumer.in_offset
    if s.numel() != 1 or off is None or off.numel() != 1 or s.device != x.device or s.dtype is not torch.float32:
        return None
    if off.dtype is not torch.float32 or off.device != x.device:
        return None
    g = 1 / math.sqrt(x.numel() * consumer.in_max_val)                                  # modules/base.py:96
    return s, (off, consumer.in_min_val, consumer.in_max_val, g)


def _unfused(x, bn, identity, relu):
    out = type(bn).forward(bn, x)       # the class's own forward: `bn.forward` may be one of the fused wrappers below
    if identity is not None:
        out = out + identity
    return torch.relu(out) if relu else out


def bn_act_quant(x, bn, consumer=None, identity=None, relu=True, want_plain=False):
    """-> (a | None, a_q | None).  a = relu(bn(x) + identity), a_q = consumer's input fake-quant of a (only when
    `consumer` is a ready QBase layer with a per-tensor input quantizer).  Fused when possible, else composed from
    the library ops; in the unfused case a is returned and a_q is None (the consumer quantises it itself)."""
    if not fusable(x, bn, identity):
        return _unfused(x, bn, identity, relu), None
    cq = _consumer_q(consumer, x) if consumer is not None else None
    batch_stats = bn.training or bn.running_mean is None
    if bn.training and bn.track_running_stats and bn.num_batches_tracked is not None:
        bn.num_batches_tracked.add_(1)                                      # nn.BatchNorm2d.forward bookkeeping
    state = (bn.running_mean, bn.running_var, batch_stats, bn.momentum, bn.eps)
    if cq is None:
        a, _ = BnActQuantFunction.apply(x, bn.weight, bn.bias, None, identity, state, None, relu, True)
        return a, None
    scale, q = cq
    return BnActQuantFunction.apply(x, bn.weight, bn.bias, scale, identity, state, q, relu,
                                    want_plain or identity is not None)


def _bn_act_codes(x, bn, consumer, identity, relu, want_plain):
    """Inference hand-off to the code GEMM: (a | None, codes) with codes = the consumer's input codes of
    a = relu(bn(x) + identity), one byte each in the consumer's operand encoding (dlmcq_bnq_forward_codes), when the
    fused kernels take x and `consumer` runs on codes in this call (qgemm.code_input_spec); else None."""
    if consumer is None or not fusable(x, bn, identity) or bn.training or bn.running_mean is None:
        return None
    cq = _consumer_q(consumer, x)
    if cq is None:
        return None
    spec = qgemm.code_input_spec(consumer, x.numel(), x.dtype, x.dim())
    if spec is None:
        return None
    encoding, g = spec
    scale, (offset, lo, hi, _) = cq
    rows, ch = _rows_channels(x)
    flags = (BNQ_RELU if relu else 0) | (BNQ_RESIDUAL if identity is not None else 0)
    desc = BnqDesc(rows, ch, F._dtype_code(x), flags, float(bn.eps), float(bn.momentum))
    stats = torch.empty(2, ch, dtype=torch.float32, device=x.device)          # save_mean, save_invstd
    a = torch.empty_like(x) if want_plain else None
    codes = torch.empty_like(x, dtype=torch.uint8)     # x's memory format: [rows, C] bytes
    qp = QParams(FORM_AFFINE, int(lo), int(hi), float(g), scale.data_ptr(), offset.data_ptr())
    with F._on(x.device):
        ws, n = _bnq_ws(x.device, desc)
        _lib.check(_lib.lib().dlmcq_bnq_forward_codes(
            F._ptr(x), F._ptr(identity), F._ptr(bn.weight), F._ptr(bn.bias), F._ptr(bn.running_mean),
            F._ptr(bn.running_var), stats.data_ptr(), stats.data_ptr() + 4 * ch, F._ptr(a), F._ptr(codes),
            C.byref(desc), C.byref(qp), int(encoding), F._ptr(ws), n, F._stream_ptr()))
    return a, codes


class _Output:
    """numel() and device of a layer output that is never materialised (the chained site's BatchNorm input)."""

    def __init__(self, shape, device):
        self.shape, self.device = shape, device

    def numel(self):
        return math.prod(self.shape)


def chain_spec(producer, in_shape, dtype, device, bn, consumer):
    """(encoding, g) when the site producer -> bn -> (ReLU) -> consumer runs as ONE kernel in this call - the code GEMM
    epilogue writes the consumer's input codes (qgemm.forward_codes with a tail) - else None.  It does exactly when the
    two-kernel chain it replaces would run: the producer runs on codes (qgemm._code_state), its output is `fusable` for
    the eval BatchNorm, and the consumer takes codes from a fused producer (_consumer_q, qgemm.code_input_spec); the
    codes' row width (the consumer's K or Cin) must also be a multiple of 16.  The result is byte-identical to that
    chain, so there is no switch: the site qualifies or it does not."""
    if consumer is None or bn.training or bn.running_mean is None or not _bn_ok(bn):
        return None
    if bn.running_var.dtype is not torch.float32 or (bn.bias is not None and bn.bias.dtype is not torch.float32):
        return None
    if qgemm._code_state(producer, dtype, len(in_shape)) is None:
        return None
    out = qgemm.output_shape(producer, in_shape)
    # the layouts `fusable` accepts for the output the code path writes: a Conv2d's [B, n, Ho, Wo] is channels-last
    # ([B*Ho*Wo, n] rows), a Linear's output is a contiguous [..., n] and is a [rows, C] matrix only when it has two
    # dimensions (a Linear on a 4-D input gives [B, C, H, n], which BatchNorm2d normalises along C: not fusable)
    if len(out) == 4 and isinstance(producer, nn.Conv2d):
        rc = (out[0] * out[2] * out[3], out[1])
    elif len(out) == 2 and not isinstance(producer, nn.Conv2d):
        rc = tuple(out)
    else:
        return None
    if not _rows_channels_ok(rc, dtype) or rc[1] % 16 != 0 or bn.num_features != rc[1]:
        return None
    shape = _Output(out, device)
    if _consumer_q(consumer, shape) is None:
        return None
    return qgemm.code_input_spec(consumer, shape.numel(), dtype, len(out))


def _chain(producer, x, bn, relu, consumer, codes=None, dtype=None):
    """The consumer's input codes when producer -> bn -> (ReLU) -> consumer runs chained in this call (chain_spec),
    else None (nothing has run).  The producer's input is x, or - behind another chained site - its codes `codes`
    (x then unused) with the dtype `dtype` of the layer outputs."""
    src = x if codes is None else codes
    dtype = x.dtype if codes is None else dtype
    if consumer is None or not src.is_cuda:
        return None
    spec = chain_spec(producer, tuple(src.shape), dtype, src.device, bn, consumer)
    if spec is None:
        return None
    if codes is None:
        codes = qgemm.input_codes(producer, x)
        if codes is None:
            return None                                  # a fused producer handed the producer its fake-quantised input
    return qgemm.forward_codes(producer, codes, dtype, tail=(bn, relu, consumer) + tuple(spec))


def _feed(consumer, a, aq):
    """Run the consumer layer on the fused op's result."""
    if aq is not None:
        return consumer.forward_prequantized(aq)
    return consumer(a)


def bn_act_into(x, bn, consumer, relu=True):
    """consumer(fake_quant(relu(bn(x)))) with the first three stages fused; a consumer switched to the code GEMM is
    handed its input codes instead of the fake-quantised tensor."""
    r = _bn_act_codes(x, bn, consumer, None, relu, want_plain=False)
    if r is not None:
        return qgemm.forward_codes(consumer, r[1], x.dtype)
    a, aq = bn_act_quant(x, bn, consumer, None, relu, want_plain=False)
    return _feed(consumer, a, aq)


def bn_add_act(x, bn, identity, next_consumer=None, relu=True):
    """relu(bn(x) + identity) as a plain tensor; when `next_consumer` is a ready quantised layer its input fake-quant
    is produced by the same kernel and travels with the tensor (`_dlmcq_q`), where QBase.forward picks it up - or, when
    the layer runs on the code GEMM, its input codes (`_dlmcq_codes`), which the code path picks up."""
    r = _bn_act_codes(x, bn, next_consumer, identity, relu, want_plain=True)
    if r is not None:
        a, codes = r
        a._dlmcq_codes = (next_consumer, codes)
        return a
    a, aq = bn_act_quant(x, bn, next_consumer, identity, relu, want_plain=True)
    if aq is not None:
        a._dlmcq_q = (next_consumer, aq)
    return a


# ------------------------------------------------------------------------------------------------------
# model rewiring
# ------------------------------------------------------------------------------------------------------
def _is_bn(m):
    return isinstance(m, (nn.BatchNorm2d, nn.BatchNorm1d)) and type(m).forward in (nn.BatchNorm2d.forward, nn.BatchNorm1d.forward,
                                                                                  nn.modules.batchnorm._BatchNorm.forward)


def _fused_sequential_run(mods, x):
    """Run a list of modules with [BatchNorm, ReLU?, QBase?] runs fused, and [QBase, BatchNorm, ReLU?, QBase] runs
    chained where they qualify (chain_spec)."""
    i, n = 0, len(mods)
    codes, dtype = None, x.dtype if isinstance(x, torch.Tensor) else None   # codes: mods[i]'s input from a chained site
    while i < n:
        m = mods[i]
        if isinstance(m, QBase) and i + 1 < n and _is_bn(mods[i + 1]):
            relu = i + 2 < n and isinstance(mods[i + 2], nn.ReLU)
            j = i + (3 if relu else 2)
            consumer = mods[j] if j < n and isinstance(mods[j], QBase) else None
            nxt = _chain(m, x, mods[i + 1], relu, consumer, codes, dtype)
            if nxt is not None:
                codes, i = nxt, j
                continue
        if codes is not None:
            x, codes = qgemm.forward_codes(m, codes, dtype), None
            i += 1
            continue
        if _is_bn(m):
            relu = i + 1 < n and isinstance(mods[i + 1], nn.ReLU)
            j = i + (2 if relu else 1)
            consumer = mods[j] if j < n and isinstance(mods[j], QBase) else None
            if consumer is not None:
                x = bn_act_into(x, m, consumer, relu)
                i = j + 1
            else:
                x, _ = bn_act_quant(x, m, None, None, relu, want_plain=True)
                i = j
            continue
        x = m(x)
        i += 1
    return x


def _sequential_forward(self, x):
    return _fused_sequential_run(list(self._modules.values()), x)


def _tv_bottleneck_forward(self, x):
    """torchvision.models.resnet.Bottleneck.forward with the BatchNorm / ReLU / next-layer quantizer chains fused, and
    conv1 -> bn1 -> relu -> conv2 (then conv2 -> bn2 -> relu -> conv3) chained where they qualify."""
    c2 = _chain(self.conv1, x, self.bn1, True, self.conv2)
    if c2 is None:
        out = self.conv1(x)
        out = bn_act_into(out, self.bn1, self.conv2)
        out = bn_act_into(out, self.bn2, self.conv3)
    else:
        c3 = _chain(self.conv2, None, self.bn2, True, self.conv3, c2, x.dtype)
        if c3 is None:
            out = bn_act_into(qgemm.forward_codes(self.conv2, c2, x.dtype), self.bn2, self.conv3)
        else:
            out = qgemm.forward_codes(self.conv3, c3, x.dtype)
    identity = x if self.downsample is None else self.downsample(x)
    return bn_add_act(out, self.bn3, identity, self._dlmcq_next)


def _tv_basic_forward(self, x):
    """torchvision.models.resnet.BasicBlock.forward, fused; conv1 -> bn1 -> relu -> conv2 chained where it qualifies."""
    c2 = _chain(self.conv1, x, self.bn1, True, self.conv2)
    if c2 is None:
        out = bn_act_into(self.conv1(x), self.bn1, self.conv2)
    else:
        out = qgemm.forward_codes(self.conv2, c2, x.dtype)
    identity = x if self.downsample is None else self.downsample(x)
    return bn_add_act(out, self.bn2, identity, self._dlmcq_next)


def _ref_block_forward(self, x):
    """model/classification/cifarresnet_large.py:45-46,76-77 `relu(residual_function(x) + shortcut(x))`, fused."""
    seq = list(self.residual_function._modules.values())
    h = _fused_sequential_run(seq[:-1], x)
    short = list(self.shortcut._modules.values())
    identity = _fused_sequential_run(short, x) if short else x
    return bn_add_act(h, seq[-1], identity, self._dlmcq_next)


def _block_kind(m):
    has = lambda *names: all(hasattr(m, n) for n in names)
    if has("conv1", "bn1", "conv2", "bn2", "conv3", "bn3", "downsample") and _is_bn(m.bn3):
        return "tv_bottleneck"
    if has("conv1", "bn1", "conv2", "bn2", "downsample") and not hasattr(m, "conv3") and _is_bn(m.bn2):
        return "tv_basic"
    if has("residual_function", "shortcut") and isinstance(m.residual_function, nn.Sequential):
        seq = list(m.residual_function._modules.values())
        if seq and _is_bn(seq[-1]):
            return "ref_block"
    return None


def _first_consumer(block, kind):
    if kind in ("tv_bottleneck", "tv_basic"):
        return block.conv1
    return next(iter(block.residual_function._modules.values()))


def _bn_forward(self, x):
    """A stand-alone BatchNorm on the fused kernels (no ReLU, no quantizer)."""
    return bn_act_quant(x, self, None, None, False, True)[0]


def _bn_relu_forward(self, x):
    """BatchNorm + the ReLU that follows it in the model's forward (a stem)."""
    return bn_act_quant(x, self, None, None, True, True)[0]


_FORWARDS = {"tv_bottleneck": _tv_bottleneck_forward, "tv_basic": _tv_basic_forward, "ref_block": _ref_block_forward}


class FuseHandle:
    def __init__(self):
        self.patched = []          # (module, had_instance_forward, previous)
        self.replaced = []         # (owner, attribute name, original module)
        self.blocks = 0
        self.sequentials = 0
        self.batchnorms = 0

    def _patch(self, module, fn):
        had = 'forward' in module.__dict__
        self.patched.append((module, had, module.__dict__.get('forward')))
        module.forward = types.MethodType(fn, module)

    def _replace(self, owner, name, new):
        self.replaced.append((owner, name, getattr(owner, name)))
        setattr(owner, name, new)

    def unfuse(self):
        for module, had, prev in self.patched:
            if had:
                module.forward = prev
            else:
                module.__dict__.pop('forward', None)
            module.__dict__.pop('_dlmcq_next', None)
        for owner, name, old in self.replaced:
            setattr(owner, name, old)
        self.patched, self.replaced = [], []


def fuse_bn_act_quant(model):
    """Rewire `model` (after quantize_model) so that BatchNorm (+add) (+ReLU) -> next layer's input fake-quant run as
    the fused kernels.  Handles torchvision-style residual blocks (conv1/bn1/.../downsample), the reference's own
    residual blocks (`residual_function` + `shortcut`, model/classification/cifarresnet*.py) and BatchNorm / ReLU /
    quantised-layer runs inside any nn.Sequential (RepVGG / MobileNet style stacks, downsample branches, stems).
    Returns a FuseHandle (`unfuse()` restores the model)."""
    h = FuseHandle()
    # residual blocks, chained in execution order inside their parent Sequential so that a block's closing
    # add + ReLU also produces the next block's quantised input
    for parent in model.modules():
        if not isinstance(parent, nn.Sequential):
            continue
        kids = list(parent._modules.values())
        kinds = [_block_kind(k) for k in kids]
        for i, (blk, kind) in enumerate(zip(kids, kinds)):
            if kind is None:
                continue
            nxt = None
            if i + 1 < len(kids) and kinds[i + 1] is not None:
                nxt = _first_consumer(kids[i + 1], kinds[i + 1])
            blk.__dict__['_dlmcq_next'] = nxt if isinstance(nxt, QBase) else None
            h._patch(blk, _FORWARDS[kind])
            h.blocks += 1
    # consecutive stages (layer1 -> layer2 ...): the last block of one Sequential feeds the first block of the next
    # sibling Sequential when the parent simply calls them in order (torchvision ResNet._forward_impl); only linked
    # when both are attributes named layerK / layerK+1, which is that convention
    for parent in model.modules():
        stages = [(n, m) for n, m in parent._modules.items() if isinstance(m, nn.Sequential) and n.startswith("layer")]
        for (n0, s0), (n1, s1) in zip(stages, stages[1:]):
            try:
                consecutive = int(n1[5:]) == int(n0[5:]) + 1
            except ValueError:
                consecutive = False
            k0 = list(s0._modules.values())
            k1 = list(s1._modules.values())
            if not (consecutive and k0 and k1):
                continue
            kind1 = _block_kind(k1[0])
            if _block_kind(k0[-1]) is not None and kind1 is not None:
                nxt = _first_consumer(k1[0], kind1)
                k0[-1].__dict__['_dlmcq_next'] = nxt if isinstance(nxt, QBase) else None
    # plain Sequential runs (stems, downsample branches, VGG-style stacks)
    patched = {id(m) for m, _, _ in h.patched}
    for m in model.modules():
        if isinstance(m, nn.Sequential) and id(m) not in patched and type(m).forward is nn.Sequential.forward:
            if any(_is_bn(k) for k in m._modules.values()):
                h._patch(m, _sequential_forward)
                h.sequentials += 1
    # torchvision-style stem: `x = self.relu(self.bn1(self.conv1(x)))` written out in the model's own forward - the
    # BatchNorm takes the ReLU in, and the (now redundant) ReLU module, which nothing else in such a model uses
    # (the blocks own theirs), becomes an Identity
    for m in model.modules():
        if all(hasattr(m, n) for n in ("conv1", "bn1", "relu", "maxpool", "layer1")) and _is_bn(m.bn1) and \
                isinstance(m.relu, nn.ReLU) and _block_kind(m) is None:
            h._patch(m.bn1, _bn_relu_forward)
            h._replace(m, "relu", nn.Identity())
            h.batchnorms += 1
    # every other BatchNorm that no rewired parent drives: the normalisation alone on the fused kernels
    owned = set()
    for module, _, _ in h.patched:
        if _is_bn(module):
            owned.add(id(module))
        for k in module._modules.values():
            if _is_bn(k):
                owned.add(id(k))
            elif isinstance(k, nn.Sequential) and _block_kind(module) == "ref_block":
                owned.update(id(b) for b in k._modules.values() if _is_bn(b))
    for m in model.modules():
        if _is_bn(m) and id(m) not in owned and 'forward' not in m.__dict__:
            h._patch(m, _bn_forward)
            h.batchnorms += 1
    return h
