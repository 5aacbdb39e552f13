"""The benchmarked quantizer step and the grouped weight kernels against a float64 reference.

`bench.py` times one step of the 54 ResNet-50 W4A4 quantizer pairs: per-tensor activation fake-quant forward
(`dlmcq_fq_forward`), its backward with the scale-gradient reduction deferred (`dlmcq_fq_backward_partials` +
one `dlmcq_fq_finalize_many`), and all 54 per-channel weight tensors through one grouped launch each way
(`GroupedFakeQuant`).  Here that exact workload (`bench.Workload`, imported, not copied) is replayed from its CUDA
graphs at batch 1 and at the published batch 128 and every output is compared with the eager fp32 chain of the
reference, evaluated layer by layer on the GPU with plain torch ops:
  - y and dx bit for bit (dx = dy where autograd's gradient of the chain is non-zero, else 0);
  - every scale gradient against the float64 sum of its fp32 per-element terms, with red_close's bar
    (1e-5 relative + 2e-7 * sum|terms|).
The grouped kernels are also run on a table that mixes all four forms, per-channel and per-tensor entries, offsets,
ranges, row lengths around the 4096-element segment and unaligned starts, in fp32 and bf16, against the oracle."""
import gc
import math
import os

import numpy as np
import pytest
import torch

import bench
from oracle import restate as R
from tests.golden_io import bits_equal, first_mismatch
from tests.test_gpu_fq import A1, AFFINE, SYM, ZP, F, dev, exact, oracle_fwd, red_close

pytestmark = pytest.mark.gpu


def same_bits(a, b, what):
    """`exact` evaluated where the tensors live: the step's activations are up to 411 MB each."""
    assert bits_equal(a, b), f"{what}: {first_mismatch(a, b)}"


# --------------------------------------------------------------------------------------
# reference: the eager fp32 chain of one quantizer on a [rows, inner] view (one row per channel, or one row for a
# per-tensor quantizer); scale and a tensor offset are [rows, 1], an absent offset is the number 0
def scale_grad_terms(form, x, dy, scale, off, lo, hi, g):
    """float64 per-element terms whose row sums are the scale gradients, from the fp32 values the forward forms
    (tests/test_gpu_fq.py::test_backward_vs_oracle):
      AFFINE  g * dy * (code - inside * u),  u = (x - off) / s'   (s' = grad_scale(s, g), the forward's divisor)
      ZP/SYM  dy * ((clamp(t) - zp) - inside * v),  v = x / s, t = round(v) + zp
      A1      g * dy * (lo | hi | round(q) - q),  q = x / s        (FunLSQ.backward: no offset, no epsilon)"""
    if form == AFFINE:
        u = (x - off) / R.grad_scale(scale, g)
        inside = (u >= lo) & (u <= hi)
        term = R.round_ste(u.clamp(lo, hi)).double() - torch.where(inside, u, 0.0).double()
        mul = g
    elif form == A1:
        q = x / scale
        edge = torch.where(q < lo, float(lo), torch.where(q > hi, float(hi), 0.0))
        term = torch.where((q >= lo) & (q <= hi), q.round() - q, edge).double()
        mul = g
    else:
        v = x / scale
        t = R.round_ste(v) + off
        inside = (t >= lo) & (t <= hi)
        term = (t.clamp(lo, hi) - off).double() - torch.where(inside, v, 0.0).double()
        mul = 1.0
    term *= dy.double()
    term *= mul
    return term


def reference(form, x, dy, scale, off, lo, hi, g):
    """-> y, dx, and per row the float64 sum of the scale-gradient terms and the sum of their magnitudes.
    dx is dy where autograd's gradient of the fp32 chain is non-zero and 0 elsewhere (the chain itself computes
    (dy * s) / s, one ulp away from dy); A1 takes FunLSQ.backward's dx, row by row, as the reference does."""
    with torch.no_grad():
        y = oracle_fwd(form, x, scale, off, lo, hi, g)[1]
    if form == A1:
        dx = torch.stack([R.fun_lsq_backward(x[r], scale[r], lo, hi, g, dy[r])[0] for r in range(x.shape[0])])
    else:
        chain = {AFFINE: lambda v: R.fq_affine(v, scale, off, lo, hi, g),
                 ZP: lambda v: R.fq_zp(v, scale, off, lo, hi),
                 SYM: lambda v: R.fq_sym(v, scale, lo, hi)}[form]
        xs = x.detach().requires_grad_(True)
        (gx,) = torch.autograd.grad(chain(xs), xs, torch.ones((), dtype=x.dtype, device=x.device).expand(x.shape))
        dx = torch.where(gx != 0, dy, 0.0)
        del gx, xs
    with torch.no_grad():
        t = scale_grad_terms(form, x, dy, scale, off, lo, hi, g)
        return y, dx, t.sum(1), t.abs().sum(1)


def check_dscale(ds, exact_sum, abs_sum, what):
    """red_close(ds, exact_sum, abs_sum=abs_sum * 0.5), i.e. |err| <= 1e-5 |exact| + 2e-7 sum|t|, with the worst
    error-to-tolerance ratio in the message.  Returns that ratio."""
    mine, ref = ds.detach().double().cpu().reshape(-1), exact_sum.double().cpu().reshape(-1)
    tol = 1e-5 * ref.abs() + 4e-7 * 0.5 * abs_sum.double().cpu().reshape(-1)
    worst = float(torch.nan_to_num((mine - ref).abs() / tol, nan=math.inf).max())
    try:
        red_close(ds, exact_sum, abs_sum=abs_sum * 0.5)
    except AssertionError as e:
        raise AssertionError(f"{what}: worst error/tolerance {worst:.3g}; {e}") from None
    return worst


# --------------------------------------------------------------------------------------
# A. the benchmark step as timed
def step_outputs(wl):
    """(name, tensor) of everything one step writes."""
    for (name, _, _), a, w in zip(wl.layers, wl.acts, wl.wts):
        yield f"{name} activation y", a["y"]
        yield f"{name} activation dx", a["dx"]
        yield f"{name} weight y", w["y"]
        yield f"{name} weight dx", w["dx"]
    yield "dscale", wl.dscale


def replay(wl):
    """One step as bench.py's run_ours replays it, on outputs poisoned with NaN: capture() already ran the step
    eagerly, and a replay that skipped a write must not pass on the values that run left behind."""
    for _, t in step_outputs(wl):
        t.fill_(float("nan"))
    wl.g_fwd.replay()
    wl.g_bwd.replay()
    wl.g_wt.replay()
    torch.cuda.synchronize()


def check_quantizer(x, dy, y, dx, scale, off, lo, hi, g, what):
    """AFFINE fake-quant of one tensor (rows = scale entries): y and dx bit for bit, y on the code grid.
    -> per-row float64 scale-gradient sum and sum of |terms|."""
    rows = scale.numel()
    x2, dy2 = x.reshape(rows, -1), dy.reshape(rows, -1)
    s2 = scale.reshape(rows, 1)
    o2 = off.reshape(rows, 1) if off is not None else 0.0
    y_ref, dx_ref, ds_exact, ds_abs = reference(AFFINE, x2, dy2, s2, o2, lo, hi, g)
    same_bits(y.reshape(rows, -1), y_ref, what + " y")
    del y_ref
    # (y - off) / s' is an integer code in [lo, hi], up to the two fp32 roundings of y = code * s' + off
    # (below 2^-23 * (|code| + |off| / s') < 1e-4 code units for these qparams)
    o64 = o2.double() if off is not None else 0.0
    c = (y.reshape(rows, -1).double() - o64) / R.grad_scale(s2, g).double()
    r = c.round()
    assert float((c - r).abs().max()) <= 1e-3, f"{what}: y off the code grid"
    assert float(r.min()) >= lo and float(r.max()) <= hi, f"{what}: codes outside [{lo}, {hi}]"
    del c, r
    same_bits(dx.reshape(rows, -1), dx_ref, what + " dx")
    return ds_exact, ds_abs


def check_step(wl, what):
    """All bars for the step just replayed.  -> worst scale-gradient error/tolerance (activations, weights)."""
    exact_sums, abs_sums = [], []
    for (name, _, _), a in zip(wl.layers, wl.acts):
        qp = a["qp"]
        e, t = check_quantizer(a["x"], a["dy"], a["y"], a["dx"], a["scale"], a["off"], qp.lo, qp.hi, qp.g,
                               f"{what}: {name} activation")
        exact_sums.append(e)
        abs_sums.append(t)
    for (name, _, _), w in zip(wl.layers, wl.wts):
        e, t = check_quantizer(w["x"], w["dy"], w["y"], w["dx"], w["scale"], w["offset"], w["lo"], w["hi"], w["g"],
                               f"{what}: {name} weight")
        exact_sums.append(e)
        abs_sums.append(t)
    # wl.dscale: the 54 activation entries, then every weight channel in layer order
    exact_sum, abs_sum = torch.cat(exact_sums), torch.cat(abs_sums)
    assert exact_sum.numel() == wl.dscale.numel()
    n = len(wl.acts)
    return (check_dscale(wl.dscale[:n], exact_sum[:n], abs_sum[:n], f"{what}: activation dscale"),
            check_dscale(wl.dscale[n:], exact_sum[n:], abs_sum[n:], f"{what}: weight dscale"))


def release():
    """Hand a deleted workload's memory back (22 GB at batch 128) before the next test."""
    gc.collect()
    torch.cuda.empty_cache()


@pytest.mark.parametrize("batch", [1, 128])
def test_benchmark_step_vs_float64_reference(batch):
    """Batch 128 is the published configuration (about 22 GB of device tensors); batch 1 runs the same 54 shapes
    on grids with fewer CTAs than SMs.  After the min/max-scale step the graphs are replayed again, unchanged, and
    then with every scale multiplied by 0.25 and every activation dy replaced by |dy|, in place: a replay must read
    qparams and gradients that changed between replays (the trainer learns the scales every step), and with a few
    percent of each activation clipped at hi and dy > 0 the activation scale gradients no longer cancel, so the
    1e-5 relative part of their bar is what binds."""
    torch.cuda.reset_peak_memory_stats()
    wl = bench.Workload(batch, torch.device("cuda"), 2333)
    try:
        wl.capture()
        replay(wl)
        unclipped = check_step(wl, f"batch {batch}, min/max scales")
        ds = wl.dscale.clone()
        replay(wl)
        same_bits(wl.dscale, ds, f"batch {batch}: dscale of a second replay")

        for a in wl.acts:
            a["scale"].mul_(0.25)
            a["dy"].abs_()
        for w in wl.wts:
            w["scale"].mul_(0.25)
        replay(wl)
        clipped = check_step(wl, f"batch {batch}, scales x 0.25, dy = |dy|")
        # post-ReLU layers (all but the first): u >= 0, so with dy > 0 the zeros of dx are exactly the elements
        # clipped at hi
        clip_frac = min(float((a["dx"] == 0).float().mean()) for a in wl.acts[1:])
        assert clip_frac > 0.005, f"batch {batch}: the clipped variant clips only {clip_frac:.2%} of some layer"
        print(f"\nbatch {batch}: worst dscale error/tolerance (activations, weights): min/max scales "
              f"{unclipped[0]:.3g}, {unclipped[1]:.3g}; clipped {clipped[0]:.3g}, {clipped[1]:.3g}; "
              f"least clipped share {clip_frac:.2%}; peak device memory "
              f"{torch.cuda.max_memory_allocated() / 1e9:.1f} GB")
    finally:
        del wl
        release()


def test_replay_is_bitwise_repeatable():
    """Two replays of the step give the same y, dx and scale gradients bit for bit (the scale-gradient
    reductions sum fixed partials in a fixed order, DeferredScaleGrads / grouped_finalize_kernel)."""
    wl, first = bench.Workload(1, torch.device("cuda"), 2333), []
    try:
        wl.capture()
        replay(wl)
        first = [(name, t.clone()) for name, t in step_outputs(wl)]
        replay(wl)
        for (name, t0), (_, t1) in zip(first, step_outputs(wl)):
            same_bits(t1, t0, name + " of a second replay")
    finally:
        del wl, first
        release()


# --------------------------------------------------------------------------------------
# B. bench.py --dump-outputs
def test_dump_outputs(tmp_path):
    """54 x 4 + 1 files with the documented names, each the live tensor at the documented sample indices, and
    byte-identical for a second Workload built from the same seed."""
    def dumped(directory):
        wl = bench.Workload(1, torch.device("cuda"), 2333)
        wl.capture()
        replay(wl)
        bench.dump_outputs(wl, str(directory))
        return wl

    wl = dumped(tmp_path / "a")
    names = [f"{name}.{kind}" for name, _, _ in wl.layers for kind in ("act_y", "act_dx", "wt_y", "wt_dx")]
    files = sorted(n + ".npy" for n in names + ["dscale"])
    assert sorted(os.listdir(tmp_path / "a")) == files
    gen = torch.Generator().manual_seed(2333)
    for (name, _, _), a, w in zip(wl.layers, wl.acts, wl.wts):
        for kind, t in (("act_y", a["y"]), ("act_dx", a["dx"]), ("wt_y", w["y"]), ("wt_dx", w["dx"])):
            flat = t.reshape(-1)
            if flat.numel() > bench.DUMP_SAMPLE:
                idx = torch.randint(flat.numel(), (bench.DUMP_SAMPLE,), generator=gen).sort().values
                flat = flat[idx.to(flat.device)]
            exact(torch.from_numpy(np.load(tmp_path / "a" / f"{name}.{kind}.npy")), flat, f"{name}.{kind}")
    exact(torch.from_numpy(np.load(tmp_path / "a" / "dscale.npy")), wl.dscale, "dscale")
    del wl
    release()
    dumped(tmp_path / "b")
    release()
    for f in files:
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes(), f"{f} differs between runs"


# --------------------------------------------------------------------------------------
# C. grouped kernels against the oracle
ROW_LENGTHS = (1, 9, 147, 4095, 4096, 4097, 4608, 8193)     # around GROUP_SEG = 4096, with ResNet's 147 and 4608
RANGES = ((-7, 7), (0, 15), (-127, 127), (0, 255))


def mixed_table():
    """Every form x every row length (32 entries) -> list of dicts (form, lo, hi, x [ch, inner], dy, scale [ch],
    offset [ch] | None).  Each form gets all four ranges; every row length appears both per channel and, as
    1-3 rows of it, per tensor (channels=1, inner=numel); offsets alternate between None and per-channel float
    offsets (AFFINE, A1) or integer zero-points (ZP)."""
    gen = torch.Generator().manual_seed(4666)
    table = []
    for form in (A1, AFFINE, ZP, SYM):
        for j, length in enumerate(ROW_LENGTHS):
            lo, hi = RANGES[j % 4]
            rows = 1 + len(table) % 3
            ch, inner = (1, rows * length) if (j + form) % 3 == 1 else (rows, length)
            x = torch.randn(ch, inner, generator=gen) * 0.05
            dy = torch.randn(ch, inner, generator=gen)
            # 0.4 .. 1.2 x the scale that just covers each row: some rows clip, others do not
            scale = (torch.rand(ch, generator=gen) * 0.8 + 0.4) * x.abs().amax(1) / max(-lo, hi)
            offset = None
            if form != SYM and j % 2 == 1:
                offset = (torch.randint(0, 5, (ch,), generator=gen).float() if form == ZP
                          else torch.randn(ch, generator=gen) * 0.01)
            table.append(dict(form=form, lo=lo, hi=hi, x=x, dy=dy, scale=scale, offset=offset))
    return table


def resnet50_weight_table():
    """The benchmark's 54 weight tensors and qparams: per-channel min/max scales, signed 4-bit; zero offsets,
    as group_weight_quantizers passes them."""
    gen = torch.Generator(device="cuda").manual_seed(2333)
    table = []
    for _, _, shape in bench.resnet50_layers():
        c = shape[0]
        x = (torch.randn(shape, generator=gen, device="cuda") * 0.02).bfloat16().float().reshape(c, -1)
        dy = torch.randn(x.shape, generator=gen, device="cuda").bfloat16().float()
        scale = R.obs_minmax_channel(x, 4, True)[0].reshape(c)
        table.append(dict(form=AFFINE, lo=-7, hi=7, x=x, dy=dy, scale=scale, offset=torch.zeros_like(scale)))
    return table


def run_grouped(table, dtype, unaligned):
    """One GroupedFakeQuant forward and one backward over `table`.  x, dy, y, dx and the scale gradients are views
    into flat buffers, one element apart, outputs prefilled with NaN.  Starts are 16-byte aligned, except that with
    `unaligned` every other entry starts at an element offset that is not a multiple of 4 (fp32) or 8 (bf16), so
    one launch runs both the 128-bit and the scalar segment paths.
    -> forward entries, backward entries (`y` = dx), and the NaN that must be left outside them"""
    starts, dstarts, cur, dcur = [], [], 0, 0
    for k, t in enumerate(table):
        aligned = -(-cur // 8) * 8
        starts.append(aligned + (1 + k % 3 if unaligned and k % 2 else 0))
        cur = starts[-1] + t["x"].numel() + 1
        dstarts.append(dcur)
        dcur += t["x"].shape[0] + 1
    nan = float("nan")
    xf, dyf = torch.zeros(cur, dtype=dtype, device="cuda"), torch.zeros(cur, dtype=dtype, device="cuda")
    yf, dxf = torch.full_like(xf, nan), torch.full_like(xf, nan)
    dsf = torch.full((dcur,), nan, device="cuda")
    gaps, dgaps = torch.ones(cur, dtype=torch.bool, device="cuda"), torch.ones(dcur, dtype=torch.bool, device="cuda")
    fwd, bwd = [], []
    for t, s, d in zip(table, starts, dstarts):
        ch, inner = t["x"].shape
        n = ch * inner
        xf[s:s + n] = dev(t["x"]).reshape(-1).to(dtype)
        dyf[s:s + n] = dev(t["dy"]).reshape(-1).to(dtype)
        gaps[s:s + n] = False
        dgaps[d:d + ch] = False
        e = dict(x=xf[s:s + n], dy=dyf[s:s + n], y=yf[s:s + n], scale=dev(t["scale"]).contiguous(),
                 offset=dev(t["offset"]).contiguous() if t["offset"] is not None else None, dscale=dsf[d:d + ch],
                 channels=ch, inner=inner, form=t["form"], lo=t["lo"], hi=t["hi"], g=R.lsq_g(n, t["hi"]))
        fwd.append(e)
        bwd.append(dict(e, y=dxf[s:s + n]))
    F().GroupedFakeQuant("cuda").forward(fwd, dtype)
    F().GroupedFakeQuant("cuda").backward(bwd, dtype)
    torch.cuda.synchronize()
    return fwd, bwd, (yf[gaps], dxf[gaps], dsf[dgaps])


def check_grouped(table, dtype, unaligned, what):
    """y and dx bit for bit against the oracle (bf16: the fp32 result rounded once), scale gradients against
    float64 terms, nothing written outside the entries.  -> worst scale-gradient error/tolerance."""
    fwd, bwd, untouched = run_grouped(table, dtype, unaligned)
    exact_sums, abs_sums = [], []
    for k, (t, e, b) in enumerate(zip(table, fwd, bwd)):
        ch = e["channels"]
        x, dy = e["x"].float().reshape(ch, -1), e["dy"].float().reshape(ch, -1)
        off = e["offset"].reshape(ch, 1) if e["offset"] is not None else 0.0
        y_ref, dx_ref, ds_exact, ds_abs = reference(t["form"], x, dy, e["scale"].reshape(ch, 1), off, t["lo"],
                                                    t["hi"], e["g"])
        name = (f"{what} entry {k} (form {t['form']}, {ch} x {e['inner']}, [{t['lo']}, {t['hi']}], offset "
                f"{'none' if e['offset'] is None else 'per channel'}, start {e['x'].storage_offset()})")
        exact(e["y"], y_ref.to(dtype).reshape(-1), name + " y")
        exact(b["y"], dx_ref.to(dtype).reshape(-1), name + " dx")
        exact_sums.append(ds_exact)
        abs_sums.append(ds_abs)
    assert all(bool(u.isnan().all()) for u in untouched), f"{what}: written outside the entries"
    return check_dscale(torch.cat([b["dscale"] for b in bwd]), torch.cat(exact_sums), torch.cat(abs_sums),
                        f"{what}: dscale")


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_grouped_mixed_table_vs_oracle(dtype):
    worst = check_grouped(mixed_table(), dtype, True, f"mixed table {dtype}")
    print(f"\nmixed table {dtype}: worst dscale error/tolerance {worst:.3g}")


def test_grouped_resnet50_weights_bf16_vs_oracle():
    """The configuration group_weight_quantizers produces for a bf16 ResNet-50: the benchmark's 54 weight shapes
    and qparams in one launch per direction.  Every size is a multiple of 8 elements, so group.py's back-to-back
    output buffer starts every tensor 16-byte aligned, as here."""
    worst = check_grouped(resnet50_weight_table(), torch.bfloat16, False, "ResNet-50 weights bf16")
    print(f"\nResNet-50 weights bf16: worst dscale error/tolerance {worst:.3g}")
