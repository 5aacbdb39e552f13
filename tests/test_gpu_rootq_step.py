"""The RootQ quantizer step of BASELINE config C1 (ResNet-18 CIFAR, W4A4) against the eager fp32 chain and a float64
reference, over several steps and in eval.

`profiles/rootq_c1.py` runs that step as 8 grouped launches (`GroupedRootQ`: one prepare for the 42 quantizers, the
grouped weight and activation kernels each way).  Here the same layers (imported, not copied) run that step from a
CUDA graph, and the same data goes through the per-layer entries the RootQ modules call.  Between replays the
qparams and dy change in place, as a trainer changes them, and the running buffers carry over:
  step 0  the first-call initialisers;
  step 1  in_scale, in_run_scale x 0.25, dy = |dy|, weight bounds and their running buffers x 0.5: clipping
          dominates, so the scale gradients do not cancel and the relative part of their bar binds;
  step 2  asymmetric bounds (upper x 1.1, lower x 0.7) and alpha cycling over the clamp edges, so AMASK = 0 occurs;
  eval    a graph of a second GroupedRootQ with training=False.
Bars (the first arm against the references; every other arm bit-identical to the first where its output is exact):
  y, the running buffers and the 8-float states   bit for bit against R.rootq_act / R.rootq_wt on the GPU, step by
                                                  step (bf16: the fp32 result rounded once)
  activation dx      dy where autograd's gradient of the chain is non-zero, else 0
  dw                 |dw - dw64| <= 1e-5 |dw64| (bf16: (2^-8 + 1e-5) |dw64|), dw64 from tests/rootq_terms.py
  d in_scale, dU, dL, d alpha   1e-5 |exact| + 4e-7 sum|terms| against the float64 sum (d alpha exactly 0 where
                                the alpha clamp masks it)
R's delta = (ru - rl) / (hi - lo) divides by a Python int, which eager CUDA evaluates as a multiplication by the fp32
reciprocal; the kernels use the IEEE quotient, as the CPU does (DESIGN §2).  The reference is therefore given lo and
hi as device tensors, which makes every division of the chain a tensor / tensor division."""
import gc
import math
import time

import pytest
import torch

import bench
from oracle import restate as R
from profiles.rootq_c1 import cifar_resnet18_layers
from tests.golden_io import bits_equal, first_mismatch
from tests.rootq_terms import act_terms, wt_terms

pytestmark = pytest.mark.gpu

LO, HI, MOM = 0, 15, 0.1
Q = HI - LO
NAN = float("nan")
ALPHA_CYCLE = (1e-4, 0.5, 0.999, 1.0, 1.3, -0.2)


def Fn():
    from dlmc_quant_b200 import functional
    return functional


def same_bits(a, b, what):
    assert bits_equal(a, b), f"{what}: {first_mismatch(a, b)}"


class Bars:
    """The bars of the module docstring; remembers the worst error/tolerance ratio per bar."""

    def __init__(self):
        self.worst = {}

    def _note(self, bar, ratio):
        self.worst[bar] = max(self.worst.get(bar, 0.0), ratio)

    def red(self, bar, got, exact, abs_sum, what):
        got, exact, abs_sum = float(got), float(exact), float(abs_sum)
        if math.isnan(exact) or math.isnan(got):
            assert math.isnan(exact) and math.isnan(got), f"{what}: {got!r} vs float64 {exact!r}"
            return
        tol = 1e-5 * abs(exact) + 4e-7 * abs_sum
        ratio = abs(got - exact) / tol if tol > 0 else (0.0 if got == exact else math.inf)
        self._note(bar, ratio)
        assert ratio <= 1, f"{what}: {got!r} vs float64 {exact!r}, error/tolerance {ratio:.3g}"

    def dw(self, dw, dw64, rtol, what):
        err, tol = (dw.double() - dw64).abs(), rtol * dw64.abs()
        ok = err <= tol
        self._note("dw", float((err / tol)[tol > 0].max()) if bool((tol > 0).any()) else 0.0)
        assert bool(ok.all()), f"{what}: {int((~ok).sum())} elements beyond {rtol:.3g} relative"

    def report(self, what, t0):
        ratios = ", ".join(f"{k} {v:.3g}" for k, v in self.worst.items())
        print(f"\n{what}: worst error/tolerance: {ratios}; {time.perf_counter() - t0:.1f} s, peak device memory "
              f"{torch.cuda.max_memory_allocated() / 1e9:.2f} GB")


# --------------------------------------------------------------------------------------
# the network: layers, qparams, three sets of running buffers (g: grouped graph, p: per-layer entries, r: reference)
ARMS = ("g", "p", "r")


def c1_layers():
    """C1's 21 layers; a downsample quantizer (1x1 weight) reads its block's conv1 input, two layers earlier."""
    shapes = cifar_resnet18_layers()
    return shapes, [i - 2 if len(w) == 4 and w[2] == 1 else i for i, (_, w) in enumerate(shapes)]


def resnet50_layers():
    """bench.py's 54 ResNet-50 layers; a downsample quantizer reads its block's conv1 input."""
    layers = bench.resnet50_layers()
    names = [n for n, _, _ in layers]
    src = [names.index(n.replace("downsample.0", "conv1")) for n in names]
    return [(a, w) for _, a, w in layers], src


def make_net(shapes, src, batch, dtype, seed):
    """Inputs and initialisers as profiles/rootq_c1.py makes them: x ~ N(0,1) (post-ReLU x 2 after the stem),
    w ~ 0.03 N(0,1), dy ~ N(0,1), in_scale = (max - min) / Q, bounds = +-2 mean|w| sqrt(Q), alpha 0.25, running
    buffers = the parameters."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    net = []
    for i, (a, w) in enumerate(shapes):
        if src[i] == i:
            x = torch.randn((batch,) + tuple(a), generator=gen, device="cuda")
            x = (torch.relu(x) * 2 if i else x).to(dtype)
        else:
            x = net[src[i]]["x"]
        wt = (torch.randn(w, generator=gen, device="cuda") * 0.03).to(dtype)
        L = dict(x=x, w=wt, dyx=torch.randn(x.shape, generator=gen, device="cuda").to(dtype),
                 dyw=torch.randn(wt.shape, generator=gen, device="cuda").to(dtype), alpha=torch.tensor(0.25, device="cuda"),
                 g_i=1 / math.sqrt(x.numel() * HI), g_w=1 / math.sqrt(wt.numel() * HI))
        L["in_scale"] = R.rootq_act_init(x.float(), LO, HI).float().reshape(())
        up, dn = R.rootq_wt_init(wt.float(), HI)
        L["up"], L["dn"] = up.float().reshape(()), dn.float().reshape(())
        net.append(L)
    reset_buffers(net)
    return net


def reset_buffers(net):
    for L in net:
        for arm in ARMS:
            L[arm + "run"], L[arm + "rup"], L[arm + "rdn"] = L["in_scale"].clone(), L["up"].clone(), L["dn"].clone()


def grouped_outputs(net):
    for L in net:
        L["y"], L["dx"], L["ds"] = torch.empty_like(L["x"]), torch.empty_like(L["x"]), torch.empty(1, device="cuda")
        L["wq"], L["dw"], L["gw"] = torch.empty_like(L["w"]), torch.empty_like(L["w"]), torch.empty(3, device="cuda")


def grouped_step(G, net, training):
    """step_all_grouped of profiles/rootq_c1.py (eval: prepare and the forward launches only)."""
    dtype = net[0]["x"].dtype
    qs = []
    for L in net:
        qs.append(dict(kind="act", in_scale=L["in_scale"], run_scale=L["grun"], momentum=MOM, g=L["g_i"], lo=LO, hi=HI,
                       training=training))
        qs.append(dict(kind="wt", upper=L["up"], lower=L["dn"], alpha=L["alpha"], run_upper=L["grup"],
                       run_lower=L["grdn"], momentum=MOM, g=L["g_w"], lo=LO, hi=HI, training=training))
    states = G.prepare(qs)
    G.wt_forward([dict(w=L["w"], out=L["wq"], state=states[2 * i + 1]) for i, L in enumerate(net)], dtype)
    G.act_forward([dict(w=L["x"], out=L["y"], state=states[2 * i]) for i, L in enumerate(net)], dtype)
    if training:
        G.act_backward([dict(w=L["x"], dy=L["dyx"], out=L["dx"], state=states[2 * i], grads=L["ds"])
                        for i, L in enumerate(net)], dtype)
        G.wt_backward([dict(w=L["w"], dy=L["dyw"], out=L["dw"], state=states[2 * i + 1], grads=L["gw"])
                       for i, L in enumerate(net)], dtype)
    return states


def capture(net, training):
    """One GroupedRootQ per graph (a new table set would free the one an earlier graph reads).  The eager warm-up
    builds the descriptor tables outside the capture; the running buffers it advanced are put back."""
    G = Fn().GroupedRootQ("cuda")
    saved = [(L["grun"].clone(), L["grup"].clone(), L["grdn"].clone()) for L in net]
    grouped_step(G, net, training)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        grouped_step(G, net, training)
    for L, (a, b, c) in zip(net, saved):
        L["grun"].copy_(a)
        L["grup"].copy_(b)
        L["grdn"].copy_(c)
    return G, graph


def grouped_arm(net, G, graph, training):
    """Replay on poisoned outputs and states -> per-layer dicts of the grouped arm's results."""
    for L in net:
        for k in ("y", "dx", "ds", "wq", "dw", "gw"):
            L[k].fill_(NAN)
    if G.states is not None:
        G.states.fill_(NAN)
    if graph is None:
        grouped_step(G, net, training)
    else:
        graph.replay()
    torch.cuda.synchronize()
    return [dict(y=L["y"], dx=L["dx"], ds=L["ds"], wq=L["wq"], dw=L["dw"], gw=L["gw"], sa=G.states[2 * i],
                 sw=G.states[2 * i + 1], run=L["grun"], rup=L["grup"], rdn=L["grdn"]) for i, L in enumerate(net)]


def per_layer_arm(net, training):
    """The per-layer entries (rootq_*_prepare / _forward / _backward), as RootQConv2d calls them."""
    F, out = Fn(), []
    for L in net:
        sa = F.rootq_act_prepare(L["in_scale"], L["prun"], MOM, L["g_i"], LO, HI, training)
        sw = F.rootq_wt_prepare(L["up"], L["dn"], L["alpha"], L["prup"], L["prdn"], MOM, L["g_w"], LO, HI, training)
        o = dict(sa=sa, sw=sw, y=F.rootq_act_forward(L["x"], sa), wq=F.rootq_wt_forward(L["w"], sw), run=L["prun"],
                 rup=L["prup"], rdn=L["prdn"])
        if training:
            o["dx"], o["ds"] = F.rootq_act_backward(L["x"], L["dyx"], sa)
            o["dw"], o["gw"] = F.rootq_wt_backward(L["w"], L["dyw"], sw)
        out.append(o)
    torch.cuda.synchronize()
    return out


def check_step(net, arms, training, bars, what, degenerate=False):
    """All bars for one step of every arm (name, per-layer results); advances the reference's running buffers.
    degenerate: dw is checked for NaN placement and sign only."""
    lo_t, hi_t = torch.tensor(LO, device="cuda"), torch.tensor(HI, device="cuda")
    dtype = net[0]["x"].dtype
    rtol = 1e-5 if dtype == torch.float32 else 2.0 ** -8 + 1e-5
    for i, L in enumerate(net):
        name = f"{what}, layer {i}"
        first = arms[0][1][i]
        # ---- activation quantizer
        xs = L["x"].float().detach().requires_grad_(training)
        y_ref, new_run = R.rootq_act(xs, L["in_scale"], L["rrun"], MOM, lo_t, hi_t, training)
        rs = new_run.reshape(()) if training else L["rrun"]
        want_sa = torch.stack([rs, rs * Q, *torch.tensor([L["g_i"], MOM, Q], device="cuda")]).float()
        if training:
            (gx,) = torch.autograd.grad(y_ref, xs, torch.ones_like(y_ref))
            dx_ref = torch.where(gx != 0, L["dyx"], 0.0)
            del gx
            a = act_terms(L["x"].float(), L["dyx"].float(), rs, Q)
            mg = MOM * L["g_i"]
            ds64, ds_abs = mg * float(a.terms.sum()), mg * float(a.terms.abs().sum())
            del a
        y_ref = y_ref.detach().to(dtype)
        L["rrun"] = rs.detach().clone()
        # ---- weight quantizer
        with torch.no_grad():
            wq_ref, U, Lb = R.rootq_wt(L["w"].float(), L["up"], L["dn"], L["alpha"], L["rrup"], L["rrdn"], MOM, lo_t, hi_t,
                                       training)
        U, Lb = U.reshape(()), Lb.reshape(())
        t = wt_terms(L["w"].float(), L["dyw"].float(), U, Lb, L["alpha"], Q)
        want_sw = torch.tensor([float(U), float(Lb), float(t.delta), float(t.alpha), L["g_w"], MOM, t.amask, Q],
                               device="cuda")
        L["rrup"], L["rrdn"] = U.clone(), Lb.clone()
        for arm, res in arms:
            r, n = res[i], f"{name} ({arm})"
            same_bits(r["y"], y_ref, n + " activation y")
            same_bits(r["wq"], wq_ref.to(dtype), n + " weight y")
            same_bits(r["sa"][:5], want_sa, n + " activation state")
            same_bits(r["sw"], want_sw, n + " weight state")
            same_bits(r["run"], L["rrun"], n + " in_run_scale")
            same_bits(r["rup"], L["rrup"], n + " wt_run_upper")
            same_bits(r["rdn"], L["rrdn"], n + " wt_run_lower")
            if not training:
                continue
            same_bits(r["dx"], dx_ref, n + " activation dx")
            bars.red("d in_scale", r["ds"][0], ds64, ds_abs, n + " d in_scale")
            if degenerate:
                nan64 = t.dw.isnan()
                assert torch.equal(r["dw"].isnan(), nan64), f"{n} dw: NaN placement"
                assert torch.equal(r["dw"].float()[~nan64].sign(), t.dw[~nan64].sign().float()), f"{n} dw: sign"
            else:
                bars.dw(r["dw"], t.dw, rtol, n + " dw")
            if r is not first:
                same_bits(r["dw"], first["dw"], n + " dw against " + arms[0][0])
            mg = MOM * L["g_w"]
            s, sa = t.terms.sum(1).tolist(), t.terms.abs().sum(1).tolist()
            bars.red("dU", r["gw"][0], mg * s[0], mg * sa[0], n + " d wt_upper")
            bars.red("dL", r["gw"][1], mg * s[1], mg * sa[1], n + " d wt_lower")
            if t.amask:
                bars.red("dalpha", r["gw"][2], s[2], sa[2], n + " d wt_alpha")
            else:
                assert float(r["gw"][2]) == 0.0, f"{n}: d wt_alpha must be 0 where the alpha clamp masks it"
        del t, y_ref, wq_ref
        if training:
            del dx_ref


def release():
    gc.collect()
    torch.cuda.empty_cache()


def change_step1(net):
    for L in net:
        L["in_scale"].mul_(0.25)
        L["dyx"].abs_()
        for arm in ARMS:
            L[arm + "run"].mul_(0.25)
        for k in ("up", "dn", *(arm + b for arm in ARMS for b in ("rup", "rdn"))):
            L[k].mul_(0.5)


def change_step2(net):
    for i, L in enumerate(net):
        for k in ("up", *(arm + "rup" for arm in ARMS)):
            L[k].mul_(1.1)
        for k in ("dn", *(arm + "rdn" for arm in ARMS)):
            L[k].mul_(0.7)
        L["alpha"].fill_(ALPHA_CYCLE[i % len(ALPHA_CYCLE)])


def run_schedule(shapes, src, batch, dtype, changes, what):
    """Training replays, each after its change of the qparams and dy, then one eval replay; both arms each step."""
    torch.cuda.reset_peak_memory_stats()
    t0, bars = time.perf_counter(), Bars()
    net = make_net(shapes, src, batch, dtype, 2333)
    grouped_outputs(net)
    Gt, gt = capture(net, True)
    Ge, ge = capture(net, False)
    try:
        for k, change in enumerate(changes):
            change(net)
            arms = [("grouped", grouped_arm(net, Gt, gt, True)), ("per layer", per_layer_arm(net, True))]
            check_step(net, arms, True, bars, f"{what}, step {k}")
            if change is change_step2:
                assert bool((Gt.states[1::2, 6] == 0).any()), "step 2 must mask some alpha gradient"
            del arms
        arms = [("grouped", grouped_arm(net, Ge, ge, False)), ("per layer", per_layer_arm(net, False))]
        check_step(net, arms, False, bars, f"{what}, eval")
        bars.report(what, t0)
    finally:
        del net, Gt, gt, Ge, ge
        release()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("batch", [1, 128])
def test_c1_step_vs_float64_reference(batch, dtype):
    """A: C1's 42 quantizers as profiles/rootq_c1.py runs them, three training steps and eval."""
    shapes, src = c1_layers()
    run_schedule(shapes, src, batch, dtype, [lambda net: None, change_step1, change_step2],
                 f"C1 batch {batch} {dtype}")


def test_resnet50_108_quantizers_vs_float64_reference():
    """B: 108 quantizers (ResNet-50's 54 layers), so the prepare launch runs on two 64-thread CTAs; batch 8 keeps
    the activations near C1's 85 M elements."""
    shapes, src = resnet50_layers()
    assert 2 * len(shapes) > 64
    run_schedule(shapes, src, 8, torch.float32, [lambda net: None], "ResNet-50 batch 8")


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("n", [(1 << 25) - 3, (1 << 25) + 5])
def test_per_tensor_backward_around_the_grid_cap(n, dtype):
    """C: the per-tensor backward runs on 888 CTAs below 2^25 elements and on 2048 from there; both sizes have a
    ragged tail.  Activation and weight quantizers through the per-layer entries, one training step."""
    torch.cuda.reset_peak_memory_stats()
    t0, bars = time.perf_counter(), Bars()
    net = make_net([((n,), (n,))], [0], 1, dtype, 77)
    L = net[0]
    L["in_scale"].mul_(0.5)                               # some of the activations clip at the top
    L["up"].mul_(0.6)
    L["dn"].mul_(0.6)
    L["alpha"].fill_(0.3)
    reset_buffers(net)
    try:
        check_step(net, [("per layer", per_layer_arm(net, True))], True, bars, f"n = {n} {dtype}")
        bars.report(f"per-tensor n = {n} {dtype}", t0)
    finally:
        del net, L
        release()


def degenerate_net(dtype):
    """D: a dead (all-zero) activation, all-zero weights, crossed bounds, delta and rs below 2^-40, and NaN, +-inf,
    -0 inside a 128-bit vector and in the ragged tail."""
    gen = torch.Generator(device="cuda").manual_seed(99)
    shapes = [((4, 8, 6, 6), (16, 8, 3, 3))] * 4 + [((4099,), (4099,))]
    net = make_net(shapes, list(range(len(shapes))), 1, dtype, 98)
    net[0]["x"].zero_()                                   # constant activation: in_scale = run = 0
    net[1]["w"].zero_()                                   # U = L = 0, delta = 0
    net[2]["up"].fill_(-0.05)                             # U < L
    net[2]["dn"].fill_(0.05)
    tiny = 2.0 ** -44
    net[3]["x"].copy_((torch.relu(torch.randn(net[3]["x"].shape, generator=gen, device="cuda")) * tiny).to(dtype))
    net[3]["w"].copy_((torch.randn(net[3]["w"].shape, generator=gen, device="cuda") * tiny).to(dtype))
    specials = torch.tensor([NAN, math.inf, -math.inf, -0.0], device="cuda").to(dtype)
    for k in ("x", "w"):
        v = net[4][k].reshape(-1)
        v[4:8] = specials
        v[-4:] = specials
    for L in net:
        L["in_scale"] = R.rootq_act_init(L["x"].float(), LO, HI).float().reshape(())
        up, dn = R.rootq_wt_init(L["w"].float(), HI)
        L["up"], L["dn"] = up.float().reshape(()), dn.float().reshape(())
    net[2]["up"].fill_(-0.05)
    net[2]["dn"].fill_(0.05)
    net[4]["in_scale"].fill_(0.2)
    net[4]["up"].fill_(0.1)
    net[4]["dn"].fill_(-0.1)
    reset_buffers(net)
    assert float(net[0]["in_scale"]) == 0.0 and float(net[1]["up"]) == 0.0 == float(net[1]["dn"])
    assert 0 < float(net[3]["in_scale"]) < 2.0 ** -40 and 0 < float(net[3]["up"] - net[3]["dn"]) / Q < 2.0 ** -40
    return net


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_degenerate_states(dtype):
    """D: both arms, eager, one training step and eval; dw is checked for NaN placement and sign."""
    t0, bars = time.perf_counter(), Bars()
    net = degenerate_net(dtype)
    grouped_outputs(net)
    G = Fn().GroupedRootQ("cuda")
    arms = [("grouped", grouped_arm(net, G, None, True)), ("per layer", per_layer_arm(net, True))]
    check_step(net, arms, True, bars, f"degenerate {dtype}", degenerate=True)
    G = Fn().GroupedRootQ("cuda")
    arms = [("grouped", grouped_arm(net, G, None, False)), ("per layer", per_layer_arm(net, False))]
    check_step(net, arms, False, bars, f"degenerate {dtype}, eval", degenerate=True)
    bars.report(f"degenerate {dtype}", t0)
