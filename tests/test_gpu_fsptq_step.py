"""The post-training path of BASELINE configs C3 (RepVGG-A0, W8A8) and C4 (MobileOne-S0, W4A8), and the AdaRound
kernels of the FSPTQ block reconstruction, against float64 and exact references at the configs' real sizes.

Layer lists come from profiles/calibration_c3_c4.py and bench.py; data is made as run_config makes it (x ~ N(0,1),
relu * 2 after the stem, w ~ 0.03 N(0,1)), on the device.  bf16 tensors follow the repository's convention: the
oracle runs on the up-converted values and the kernel's result is that fp32 value rounded once.

Bars (each prints its worst error/tolerance ratio):
  init_alpha    |a - a_ref| <= 2e-6 |a_ref| + 1e-6 against R.adaround_init_alpha on the GPU, NaN positions identical
  hard forward  bit-exact against R.fq_adaround(training=False) on the GPU
  soft forward  |y - y64| <= 2^-22 |y64| + 2^-21 s   (h carries a few ulp of absolute error; floor + h rounds once)
  d scale       1e-5 |exact| + 4e-7 sum|terms| against the float64 sum of tests/adaround_terms.py's terms per channel
  d alpha       zero pattern = the float64 masks except within 2^-22 of a mask edge (counted and reported);
                elsewhere |da - da64| <= 8 2^-24 |da64| k, with k = max(1, sigma / (1 - sigma)): the reference's
                own formula forms 1 - sigma, which multiplies sigma's rounding error by k (up to 11 at alpha = ln 11);
                the ratio against the bar without k is reported as "dalpha (k = 1)"
  bf16          y and d alpha (2^-8 + 1e-5) relative, d scale as fp32
The min/max observers and the qparams the modules derive are compared with R evaluated on CPU tensors: the library
divides by 2^n - 1 as IEEE does (DESIGN.md §2), whereas eager CUDA multiplies by the reciprocal of a Python-int
divisor.  The min and max of a tensor do not depend on the order of reduction, so R is given [min(x), max(x)]."""
import gc
import math
import time

import pytest
import torch

import bench
from oracle import restate as R
from profiles.calibration_c3_c4 import mobileone_s0_layers, repvgg_a0_layers
from tests.adaround_terms import ada_terms, l2loss_channel_rows
from tests.golden_io import bits_equal, first_mismatch
from tests.test_gpu_modules import capture
from tests.test_gpu_rootq_obs import _sweep_rows_equivalent

pytestmark = pytest.mark.gpu

NAN, INF = float("nan"), float("inf")
LN11 = float(torch.tensor(math.log(11.0)))          # the fp32 value
BF16_RTOL = 2.0 ** -8 + 1e-5


def Fn():
    from dlmc_quant_b200 import functional
    return functional


def same_bits(a, b, what):
    assert bits_equal(a.cpu(), b.cpu()), f"{what}: {first_mismatch(a.cpu(), b.cpu())}"


def release():
    gc.collect()
    torch.cuda.empty_cache()


class Bars:
    """Worst error/tolerance ratio per bar, and counts to report."""

    def __init__(self):
        self.worst, self.counts = {}, {}

    def note(self, bar, ratio):
        self.worst[bar] = max(self.worst.get(bar, 0.0), float(ratio))

    def count(self, what, n):
        self.counts[what] = self.counts.get(what, 0) + int(n)

    def elementwise(self, bar, err, tol, what):
        ok = err <= tol
        pos = tol > 0
        if bool(pos.any()):
            self.note(bar, (err[pos] / tol[pos]).max())
        bad = ~ok
        assert not bool(bad.any()), f"{what}: {int(bad.sum())} elements beyond the {bar} bar, e.g. error " \
                                    f"{float(err[bad][0]):.3g} tolerance {float(tol[bad][0]):.3g}"

    def red(self, bar, got, exact, abs_sum, what):
        """Reduced values: |got - exact| <= 1e-5 |exact| + 4e-7 abs_sum elementwise over vectors."""
        got, exact, abs_sum = got.double().reshape(-1), exact.double().reshape(-1), abs_sum.double().reshape(-1)
        nan = exact.isnan()
        assert torch.equal(got.isnan(), nan), f"{what}: NaN positions"
        self.elementwise(bar, (got - exact).abs()[~nan], (1e-5 * exact.abs() + 4e-7 * abs_sum)[~nan], what)

    def report(self, what, t0):
        ratios = ", ".join(f"{k} {v:.3g}" for k, v in self.worst.items())
        counts = "".join(f"; {k}: {v}" for k, v in self.counts.items())
        print(f"\n{what}: worst error/tolerance: {ratios}{counts}; {time.perf_counter() - t0:.1f} s, peak device "
              f"memory {torch.cuda.max_memory_allocated() / 1e9:.2f} GB")


# --------------------------------------------------------------------------------------
# AdaRound: one weight tensor through the three entries, every bar
def perturb_alpha(alpha, gen):
    """Some elements saturate on each side, some sit on 0, -0, +-ln 11 and the fp32 neighbours of +-ln 11."""
    flat = alpha.view(-1)
    n = flat.numel()
    ln11 = torch.tensor(LN11)
    up, dn = torch.nextafter(ln11, torch.tensor(INF)), torch.nextafter(ln11, torch.tensor(0.0))
    specials = [0.0, -0.0, LN11, -LN11, float(up), -float(up), float(dn), -float(dn)]
    idx = torch.randperm(n, generator=gen, device=alpha.device)
    k = max(1, n // 64)
    for j, v in enumerate(specials):
        flat[idx[j * k:(j + 1) * k]] = v
    b = len(specials) * k
    flat[idx[b:b + 2 * k]] = (torch.rand(2 * k, generator=gen, device=alpha.device) * 10 + 2.5).to(alpha.dtype)
    flat[idx[b + 2 * k:b + 4 * k]] = -(torch.rand(2 * k, generator=gen, device=alpha.device) * 10 + 2.5).to(alpha.dtype)


def check_init_alpha(bars, alpha, w, s, what):
    ref = R.adaround_init_alpha(w.float(), s)
    nan = ref.isnan()
    assert torch.equal(alpha.isnan(), nan), f"{what}: init_alpha NaN positions"
    rtol = 2e-6 if alpha.dtype == torch.float32 else 2.0 ** -8 + 2e-6
    a, r = alpha.double()[~nan], ref.double()[~nan]
    bars.elementwise("init_alpha", (a - r).abs(), rtol * r.abs() + 1e-6, what + " init_alpha")


def check_soft(bars, y, t, s, what):
    rtol = 2.0 ** -22 if y.dtype == torch.float32 else BF16_RTOL
    tol = rtol * t.y.abs() + 2.0 ** -21 * s.double().expand_as(t.y)
    bars.elementwise("soft forward", (y.double() - t.y).abs(), tol, what + " soft forward")


def check_dalpha(bars, da, t, what):
    """Zero pattern against the float64 masks (and dy = 0, which randn does produce) away from the mask edges;
    relative bar elsewhere."""
    near = t.near_pre | t.near_q
    nz = da.float() != 0
    differ = nz != (t.da != 0)
    if bool((differ & ~near).any()):
        j = (differ & ~near).reshape(-1).nonzero()[0, 0]
        e = {k: float(getattr(t, k).reshape(-1)[j]) for k in ("fl", "sg", "pre", "q", "da")}
        raise AssertionError(f"{what} dalpha: zero pattern differs from the float64 masks at "
                             f"{int((differ & ~near).sum())} elements away from a mask edge, e.g. element {int(j)}: "
                             f"kernel {float(da.reshape(-1)[j])!r}, float64 {e}")
    bars.count("boundary-excluded elements", near.sum())
    bars.count("of which the kernel decided differently", (differ & near).sum())
    sel = t.mask & ~near
    d64 = t.da[sel]
    err = (da.double()[sel] - d64).abs()
    if da.dtype == torch.float32:
        sg = t.sg[sel]
        k = torch.clamp(sg / (1.0 - sg), min=1.0)
        base = 8 * 2.0 ** -24 * d64.abs()
        pos = base > 0
        if bool(pos.any()):
            bars.note("dalpha (k = 1)", (err[pos] / base[pos]).max())
        bars.elementwise("dalpha", err, base * k, what + " dalpha")
    else:
        bars.elementwise("dalpha", err, BF16_RTOL * d64.abs(), what + " dalpha")


def check_adaround(bars, w, s, alpha, dy, lo, hi, what, ch_axis=0):
    """Every AdaRound bar for one tensor; s is the [C] scale of channel axis ch_axis."""
    F = Fn()
    shape = [1] * w.dim()
    shape[ch_axis] = -1
    sb = s.reshape(shape)
    dt = w.dtype
    hard = F.adaround_forward(w, alpha, s, lo, hi, soft=False, ch_axis=ch_axis)
    same_bits(hard, R.fq_adaround(w.float(), sb, alpha.float(), lo, hi, False).to(dt), what + " hard forward")
    del hard
    t = ada_terms(w.float(), alpha.float(), sb, dy.float(), lo, hi)
    y = F.adaround_forward(w, alpha, s, lo, hi, soft=True, ch_axis=ch_axis)
    assert y.dtype == dt
    check_soft(bars, y, t, sb, what)
    del y
    da, ds = F.adaround_backward(w, alpha, dy, s, lo, hi, ch_axis=ch_axis)
    assert da.dtype == dt and ds.dtype == torch.float32
    red = [d for d in range(w.dim()) if d != ch_axis]
    bars.red("d scale", ds, t.ds.sum(dim=red), t.ds.abs().sum(dim=red), what + " d scale")
    check_dalpha(bars, da, t, what)
    bars.count("elements", w.numel())
    return da, ds


def weight_case(shape, bits, dtype, gen):
    """w ~ 0.03 N(0,1); s = min/max per channel + 1e-6 (FSPTQBase.forward); alpha = init_alpha, perturbed."""
    from dlmc_quant_b200.scalar import ops
    lo, hi = R.qrange(True, bits)
    w = (torch.randn(shape, generator=gen, device="cuda") * 0.03).to(dtype)
    s = ops.quantize_minmax_channel(w, bits, True, ch_axis=0)[0].reshape(-1) + 1e-6
    alpha = Fn().adaround_init_alpha(w, s)
    dy = torch.randn(shape, generator=gen, device="cuda").to(dtype)
    return w, s, alpha, dy, lo, hi


def network_weights(net):
    if net == "C3":
        return [w for _, w in repvgg_a0_layers()], 8
    if net == "C4":
        return [w for _, w in mobileone_s0_layers()], 4
    return [w for _, _, w in bench.resnet50_layers()], 4


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("net", ["C3", "C4", "ResNet-50"])
def test_adaround_every_weight_tensor(net, dtype):
    """a: every weight tensor of the network, init_alpha, hard and soft forward, backward."""
    torch.cuda.reset_peak_memory_stats()
    t0, bars = time.perf_counter(), Bars()
    gen = torch.Generator(device="cuda").manual_seed(2333)
    shapes, bits = network_weights(net)
    for i, shape in enumerate(shapes):
        w, s, alpha, dy, lo, hi = weight_case(shape, bits, dtype, gen)
        check_init_alpha(bars, alpha, w, s.reshape([-1] + [1] * (w.dim() - 1)), f"{net} layer {i}")
        perturb_alpha(alpha, gen)
        check_adaround(bars, w, s, alpha, dy, lo, hi, f"{net} {dtype} layer {i} {tuple(shape)}")
        del w, s, alpha, dy
    bars.report(f"AdaRound {net} W{bits} {dtype}", t0)
    release()


# --------------------------------------------------------------------------------------
# b: backward geometry - segment-count boundaries, multi-segment rows, outer > 1, determinism
GEOMETRY = [
    ((8, 2048), 0), ((8, 2049), 0), ((16, 2304), 0), ((16, 4608), 0), ((4, 5000), 0), ((2, 60000), 0),
    ((1, 777), 0), ((1, 60000), 0), ((1000, 9), 0), ((1280, 27), 0),
    ((3, 16, 300), 1), ((3, 16, 2500), 1), ((5, 7, 9), 1),
]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("shape,ch_axis", GEOMETRY)
def test_adaround_backward_geometry(shape, ch_axis, dtype):
    t0, bars = time.perf_counter(), Bars()
    gen = torch.Generator(device="cuda").manual_seed(sum(shape) + ch_axis)
    lo, hi = R.qrange(True, 4)
    w = (torch.randn(shape, generator=gen, device="cuda") * 0.03).to(dtype)
    red = [d for d in range(w.dim()) if d != ch_axis]
    s = w.float().abs().amax(dim=red) / hi + 1e-6
    shp = [1] * w.dim()
    shp[ch_axis] = -1
    alpha = Fn().adaround_init_alpha(w, s, ch_axis=ch_axis)
    check_init_alpha(bars, alpha, w, s.reshape(shp), f"{shape}")
    perturb_alpha(alpha, gen)
    dy = torch.randn(shape, generator=gen, device="cuda").to(dtype)
    da, ds = check_adaround(bars, w, s, alpha, dy, lo, hi, f"{shape} ch_axis {ch_axis}", ch_axis=ch_axis)
    for _ in range(10):
        da2, ds2 = Fn().adaround_backward(w, alpha, dy, s, lo, hi, ch_axis=ch_axis)
        same_bits(da2, da, "repeated backward dalpha")
        same_bits(ds2, ds, "repeated backward d scale")
    bars.report(f"geometry {shape} ch_axis {ch_axis} {dtype}", t0)


# --------------------------------------------------------------------------------------
# c: special values
def special_case(bits):
    lo, hi = R.qrange(True, bits)
    scales = [0.01, 1e-30, 0.0]
    tiny = 2.0 ** -149
    alphas = [0.0, -0.0, tiny, -tiny, 20.0, -20.0, INF, -INF, NAN]
    rows = []
    for s in scales:
        st = torch.tensor(s)
        ws = [0.0, -0.0, INF, -INF, NAN, tiny, -tiny, 1e-40, -1e-40]
        for k in range(lo - 2, hi + 3):
            v = torch.tensor(float(k)) * st
            ws += [float(v), float(torch.nextafter(v, torch.tensor(INF))),
                   float(torch.nextafter(v, torch.tensor(-INF)))]
        rows.append([(a_, b_) for a_ in ws for b_ in alphas])
    k = max(len(r) for r in rows)
    w = torch.zeros(len(scales), k)
    a = torch.zeros(len(scales), k)
    for c, r in enumerate(rows):
        w[c, :len(r)] = torch.tensor([p[0] for p in r])
        a[c, :len(r)] = torch.tensor([p[1] for p in r])
    return w.cuda(), a.cuda(), torch.tensor(scales).cuda(), lo, hi


@pytest.mark.parametrize("bits", [4, 8])
def test_adaround_special_values(bits):
    F = Fn()
    w, alpha, s, lo, hi = special_case(bits)
    sb = s.reshape(-1, 1)
    same_bits(F.adaround_forward(w, alpha, s, lo, hi, soft=False), R.fq_adaround(w, sb, alpha, lo, hi, False),
              "hard forward")
    init = F.adaround_init_alpha(w, s)
    ref = R.adaround_init_alpha(w, sb)
    assert torch.equal(init.isnan(), ref.isnan()), "init_alpha NaN positions"
    fin = torch.isfinite(ref)
    assert torch.equal(torch.isfinite(init), fin) and torch.equal(init[~fin & ~ref.isnan()], ref[~fin & ~ref.isnan()])
    dy = torch.ones_like(w)
    y_ref, ds_ref, da_ref = R.fq_adaround_fwd_bwd(w, sb, alpha, lo, hi, dy)
    y = F.adaround_forward(w, alpha, s, lo, hi, soft=True)
    assert torch.equal(y.isnan(), y_ref.isnan()), "soft forward NaN pattern"
    assert torch.equal(y == 0, y_ref == 0), "soft forward zero pattern"
    assert torch.equal(y.isinf(), y_ref.isinf()), "soft forward inf pattern"
    da, ds = F.adaround_backward(w, alpha, dy, s, lo, hi)
    assert torch.equal(da.isnan(), da_ref.isnan()), "dalpha NaN pattern"
    assert torch.equal(da == 0, da_ref == 0), "dalpha zero pattern"
    assert torch.equal(ds.isnan(), ds_ref.reshape(-1).isnan()), "d scale NaN pattern"


def test_adaround_inclusive_clamp_edges():
    """floor(w / s) = hi - 1 or lo - 1 and h = 1 - 1.8e-6: floor + h rounds to hi or lo in fp32, where the reference's
    clamp passes the gradient (its backward is inclusive), although the float64 sum lies just inside or outside."""
    F = Fn()
    lo, hi = R.qrange(True, 8)
    s = torch.tensor([0.01, 0.003], device="cuda")
    alphas = [LN11 - 1e-5, LN11 - 2e-5, LN11 - 3e-5]
    v = torch.tensor([hi - 0.5] * 3 + [lo - 0.5] * 3, device="cuda")
    w = s.reshape(-1, 1) * v
    alpha = torch.tensor(alphas * 2, device="cuda").repeat(2, 1)
    sb = s.reshape(-1, 1)
    y = F.adaround_forward(w, alpha, s, lo, hi, soft=True)
    bound = torch.tensor([float(hi)] * 3 + [float(lo)] * 3, device="cuda")
    same_bits(y, bound * sb, "floor + h on the clamp bound")
    dy = torch.ones_like(w)
    _, _, da_ref = R.fq_adaround_fwd_bwd(w, sb, alpha, lo, hi, dy)
    da, _ = F.adaround_backward(w, alpha, dy, s, lo, hi)
    assert bool((da_ref != 0).all()), "the reference passes the gradient on the clamp bounds"
    assert bool((da != 0).all()), f"dalpha must pass on the clamp bounds: {da}"
    assert torch.allclose(da, da_ref, rtol=1e-5, atol=0)


# --------------------------------------------------------------------------------------
# d: the C3 / C4 calibration pass at batch 128, as profiles/calibration_c3_c4.py calls it
def minmax_tensor_ref(x, bits, signed):
    mm = torch.stack([x.min(), x.max()]).float().cpu()
    s, o = R.obs_minmax_tensor(mm, bits, signed)
    return s.float().reshape(()), torch.as_tensor(o).float().reshape(())


def sweep_sse64(x, stats, bits):
    """80 float64 sums of the fp32 candidate chain (ops.py:53-61), candidates formed as the reference forms them on
    CPU tensors (IEEE division)."""
    qmax = 2 ** bits - 1
    lo, hi = stats[0, 0].cpu(), stats[0, 1].cpu()
    out, cands = [], []
    for i in range(R.N_SWEEP):
        r = 1 - 0.01 * i
        c_hi, c_lo = r * hi, r * lo
        sc = (c_hi - c_lo) / qmax
        zp = torch.round(-c_lo / sc)
        cands.append((sc, zp))
        scd, zpd = sc.cuda(), zp.cuda()
        xq = ((torch.round(x / scd) + zpd).clamp(0, qmax) - zpd) * scd
        out.append(((xq - x) ** 2).double().sum())
        del xq
    return torch.stack(out).cpu(), cands


def calib_data(shape_a, shape_w, i, batch, gen):
    x = torch.randn((batch,) + tuple(shape_a), generator=gen, device="cuda")
    if i:
        x = torch.relu(x) * 2
    w = torch.randn(shape_w, generator=gen, device="cuda") * 0.03
    return x, w


def zp_terms(x, dy, scale, off, lo, hi):
    """The d scale terms of test_gpu_fq.test_backward_vs_oracle, FORM_ZP / FORM_SYM (off None)."""
    v = x / scale
    t = R.round_ste(v) + (off if off is not None else 0)
    inside = (t >= lo) & (t <= hi)
    deq = t.clamp(lo, hi) - (off if off is not None else 0)
    return dy.double() * (deq.double() - torch.where(inside, v, torch.zeros_like(v)).double())


def check_fq_pair(bars, x, w, s_in, o_in, s_w, abits, wlo, whi, gen, what):
    from dlmc_quant_b200._lib import FORM_SYM, FORM_ZP
    F = Fn()
    amax = 2 ** abits - 1
    qx = F.fq_forward(x, s_in, o_in, 0, amax, FORM_ZP)
    same_bits(qx, R.fq_zp(x, s_in, o_in, 0, amax), what + " ZP forward")
    del qx
    sw = s_w.reshape(-1) + 1e-6
    swb = sw.reshape([-1] + [1] * (w.dim() - 1))
    qw = F.fq_forward(w, sw, None, wlo, whi, FORM_SYM, ch_axis=0)
    same_bits(qw, R.fq_sym(w, swb, wlo, whi), what + " SYM forward")
    del qw
    for name, t, sc, off, lo, hi, ax in (("ZP", x, s_in, o_in, 0, amax, None), ("SYM", w, swb, None, wlo, whi, 0)):
        dy = torch.randn(t.shape, generator=gen, device="cuda")
        form = FORM_ZP if off is not None else FORM_SYM
        d, ds = F.fq_backward(t, dy, sc.reshape(-1) if ax == 0 else sc, off, lo, hi, form, ch_axis=ax)
        ts = t.detach().clone().requires_grad_(True)
        ss = sc.detach().clone().requires_grad_(True)
        y = R.fq_zp(ts, ss, off, lo, hi) if off is not None else R.fq_sym(ts, ss, lo, hi)
        (dref,) = torch.autograd.grad(y, (ts,), dy)
        del y, ts, ss
        assert torch.equal(d == 0, dref == 0), f"{what} {name} dx: clamp mask"
        err, tol = (d.double() - dref.double()).abs(), 1e-6 * dref.double().abs()
        bars.elementwise(f"{name} dx", err, tol, f"{what} {name} dx")
        del err, tol, dref, d
        terms = zp_terms(t, dy, sc, off, lo, hi)
        red = [k for k in range(t.dim()) if k != 0] if ax == 0 else list(range(t.dim()))
        bars.red(f"{name} d scale", ds, terms.sum(dim=red), terms.abs().sum(dim=red), f"{what} {name} d scale")
        del terms, dy


@pytest.mark.parametrize("cfg", ["C3", "C4"])
def test_calibration_pass_batch128(cfg):
    """d: min/max observers, the 80-candidate tensor sweep, the channel sweep over every row, ZP / SYM fake-quant."""
    from dlmc_quant_b200.scalar import ops
    torch.cuda.reset_peak_memory_stats()
    t0, bars = time.perf_counter(), Bars()
    layers, wbits, abits = (repvgg_a0_layers(), 8, 8) if cfg == "C3" else (mobileone_s0_layers(), 4, 8)
    wlo, whi = R.qrange(True, wbits)
    gen = torch.Generator(device="cuda").manual_seed(2333)
    F = Fn()
    for i, (a, wshape) in enumerate(layers):
        what = f"{cfg} layer {i}"
        x, w = calib_data(a, wshape, i, 128, gen)
        # min/max observers
        s_in, o_in = ops.quantize_minmax_tensor(x, abits, False)
        rs, ro = minmax_tensor_ref(x, abits, False)
        same_bits(s_in, rs, what + " minmax tensor scale")
        same_bits(o_in, ro, what + " minmax tensor offset")
        s_w, o_w = ops.quantize_minmax_channel(w, wbits, True, ch_axis=0)
        rsw, row = R.obs_minmax_channel(w.cpu(), wbits, True, ch_axis=0)
        same_bits(s_w, rsw, what + " minmax channel scale")
        same_bits(o_w, row, what + " minmax channel offset")
        check_fq_pair(bars, x, w, s_in, o_in, s_w, abits, wlo, whi, gen, what + " min/max")
        # tensor sweep: all 80 sums, the pick
        stats = F.obs_stats(x)
        sse = F.sweep_tensor_sse(x, stats, abits, True).cpu()
        sse64, cands = sweep_sse64(x, stats, abits)
        bars.elementwise("sweep sums", (sse.double() - sse64).abs(), 1e-5 * sse64.abs(), what + " sweep sums")
        ls, lo_, picked = F.sweep_tensor(x, abits, True)
        qs, qo = ops.quantize_l2loss_tensor(x, abits, False)
        same_bits(qs, ls.reshape(()), what + " ops scale")
        same_bits(qo, lo_.reshape(()), what + " ops offset")
        _, _, rp = R.obs_l2loss_tensor(x, abits, False, return_index=True)
        p = int(picked)
        bars.count("layers accepting a candidate", p >= 0)
        bars.count("layers keeping the min/max answer", p < 0)
        if p == rp:
            if p >= 0:
                same_bits(ls, cands[p][0].reshape(1), what + " sweep scale")
                same_bits(lo_, cands[p][1].reshape(1), what + " sweep offset")
            else:
                same_bits(ls, (stats[0, 1].cpu() / (2 ** abits - 1)).reshape(1), what + " fallback scale")
        else:
            assert p >= 0 and rp >= 0, f"{what}: picked {p}, reference {rp}"
            tie = abs(float(sse64[p]) - float(sse64[rp])) / float(sse64[rp])
            bars.count("near-tie picks", 1)
            assert tie <= 2e-5, f"{what}: picked {p}, reference {rp}, float64 losses differ by {tie:.3g}"
        # channel sweep over every row
        cs, co = ops.quantize_l2loss_channel(w, wbits, True, ch_axis=0)
        rows = w.reshape(w.shape[0], -1)
        rcs, rco = l2loss_channel_rows(rows, wbits, True)
        same = (cs.reshape(-1) == rcs) & (co.reshape(-1) == rco)
        bars.count("channel rows", rows.shape[0])
        bars.count("channel rows picked differently (near-ties)", (~same).sum())
        _sweep_rows_equivalent(rows.cpu(), cs.reshape(-1).cpu(), co.reshape(-1).cpu(), rcs.cpu(), rco.cpu(), wbits)
        check_fq_pair(bars, x, w, qs, qo, cs, abits, wlo, whi, gen, what + " MSE sweep")
        del x, w, stats, sse64
        release()
    bars.report(f"calibration {cfg} batch 128", t0)


# --------------------------------------------------------------------------------------
# e: the FSPTQ module step (first forward, backward, eval), RepVGG deploy / MobileOne layers
def module_specs(cfg):
    """(kind, in shape, weight shape, stride, padding, groups) of every layer."""
    layers = repvgg_a0_layers() if cfg == "C3" else mobileone_s0_layers()
    out = []
    for i, (a, w) in enumerate(layers):
        if len(w) == 2:
            out.append(("linear", a, w, 1, 0, 1))
            continue
        nxt = layers[i + 1][0]
        stride = 2 if len(nxt) == 3 and nxt[1] < a[1] else 1
        if cfg == "C3" and len(nxt) == 1:
            stride = 2                                         # the 1280-wide stage's only block
        groups = a[0] if w[1] == 1 and a[0] > 1 else 1
        out.append(("conv", a, w, stride, w[2] // 2, groups))
    return out


def make_module(kind, a, w, stride, pad, groups, wbits, ada):
    from dlmc_quant_b200.scalar.FSPTQuant import FSPTQConv2d, FSPTQLinear
    q = {"weight": {"enable": True, "type": "minmax_channel", "args": {"n_bits": wbits, "signed": True, "ch_axis": 0}},
         "input": {"enable": True, "type": "minmax_tensor", "args": {"n_bits": 8, "signed": False}}}
    if ada:
        q["weight"]["recon_type"] = "adaround"
    if kind == "linear":
        return FSPTQLinear(w[1], w[0], qconfig=q, device="cuda")
    return FSPTQConv2d(a[0], w[0], w[2], stride=stride, padding=pad, groups=groups, qconfig=q, device="cuda")


@pytest.mark.parametrize("ada", [True, False], ids=["adaround", "sym"])
@pytest.mark.parametrize("cfg", ["C3", "C4"])
def test_module_step(cfg, ada):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.cuda.reset_peak_memory_stats()
    t0, bars = time.perf_counter(), Bars()
    wbits = 8 if cfg == "C3" else 4
    wlo, whi = R.qrange(True, wbits)
    gen = torch.Generator(device="cuda").manual_seed(4666)
    for i, (kind, a, wshape, stride, pad, groups) in enumerate(module_specs(cfg)):
        what = f"{cfg} {'AdaRound' if ada else 'SYM'} layer {i} {kind} {tuple(wshape)}"
        x, w = calib_data(a, wshape, i, 32, gen)
        m = make_module(kind, a, wshape, stride, pad, groups, wbits, ada)
        assert tuple(m.weight.shape) == tuple(wshape)
        with torch.no_grad():
            m.weight.copy_(w)
        m.train()
        seen = capture(m)
        xr = x.clone().requires_grad_(True)
        y = m(xr)
        # first forward: qparams, alpha, qx, qw
        rs, ro = minmax_tensor_ref(x, 8, False)
        same_bits(m.in_scale.detach().reshape(()), rs, what + " in_scale")
        same_bits(m.in_offset.reshape(()), ro, what + " in_offset")
        rsw = R.obs_minmax_channel(w.cpu(), wbits, True, ch_axis=0)[0]
        ws = (rsw.reshape(m.wt_scale.shape) + 1e-6).cuda()
        same_bits(m.wt_scale.detach(), ws, what + " wt_scale")
        same_bits(seen["qx"].detach(), R.fq_zp(x, m.in_scale.detach(), m.in_offset, 0, 255), what + " qx")
        dy = torch.randn(y.shape, generator=gen, device="cuda")
        if ada:
            check_init_alpha(bars, m.alpha.detach(), w, ws, what)
            alpha = m.alpha.detach().clone()
        else:
            same_bits(seen["qw"].detach(), R.fq_sym(w, ws, wlo, whi), what + " qw")
        y.backward(dy)
        gqw, gqx = seen["qw"].grad, seen["qx"].grad
        # backward
        if ada:
            t = ada_terms(w, alpha, ws, gqw, wlo, whi)
            check_soft(bars, seen["qw"].detach(), t, ws, what)
            assert m.weight.grad is not None and not bool(m.weight.grad.any()), what + ": weight.grad must be zero"
            check_dalpha(bars, m.alpha.grad, t, what)
            red = list(range(1, w.dim()))
            bars.red("d wt_scale", m.wt_scale.grad.reshape(-1), t.ds.sum(dim=red), t.ds.abs().sum(dim=red),
                     what + " wt_scale.grad")
            del t
        else:
            terms = zp_terms(w, gqw, ws, None, wlo, whi)
            red = list(range(1, w.dim()))
            bars.red("d wt_scale", m.wt_scale.grad.reshape(-1), terms.sum(dim=red), terms.abs().sum(dim=red),
                     what + " wt_scale.grad")
        terms = zp_terms(x, gqx, m.in_scale.detach(), m.in_offset, 0, 255)
        bars.red("d in_scale", m.in_scale.grad.reshape(-1), terms.sum().reshape(1), terms.abs().sum().reshape(1),
                 what + " in_scale.grad")
        del terms, seen, y
        # eval: hard rounding (AdaRound) / the same symmetric fake-quant
        m.eval()
        seen = capture(m)
        with torch.no_grad():
            m(x)
        want = R.fq_adaround(w, ws, alpha, wlo, whi, False) if ada else R.fq_sym(w, ws, wlo, whi)
        same_bits(seen["qw"], want, what + " eval qw")
        del m, seen, x, w, xr
        release()
    bars.report(f"module step {cfg} {'AdaRound' if ada else 'SYM'} batch 32", t0)
