"""GPU parity tests: RootQ kernels and PTQ observers, through the C ABI, against the golden
fixtures (reference outputs) and the oracle restatement."""
import math

import pytest
import torch

from oracle import restate as R
from tests.golden_io import bits_equal, first_mismatch, load
from tests.test_gpu_fq import F, dev, exact, red_close

pytestmark = pytest.mark.gpu

ROOTQ = load("rootq")


def _scalar(t):
    return t.reshape(()).float().cuda().clone()


@pytest.mark.parametrize("name", sorted(n for n in ROOTQ if n.startswith("conv_") and not n.endswith("_step1")))
def test_golden_rootq(name):
    c = ROOTQ[name]
    q = c.meta["qconfig"]
    m = q["momentum"]
    x, w = c.inp["x"], c.inp["weight"]
    ilo, ihi = R.qrange(False, q["input"]["args"]["n_bits"])
    wlo, whi = R.qrange(False, q["weight"]["args"]["n_bits"])
    g_i, g_w = 1 / math.sqrt(x.numel() * ihi), 1 / math.sqrt(w.numel() * whi)
    if name.endswith("_eval"):
        run = _scalar(c.out["buf_in_run_scale"])
        st = F().rootq_act_prepare(_scalar(c.out["param_in_scale"]), run, m, g_i, ilo, ihi, False)
        exact(F().rootq_act_forward(dev(x), st), c.out["qx"], "qx eval")
        ru, rl = _scalar(c.out["buf_wt_run_upper"]), _scalar(c.out["buf_wt_run_lower"])
        sw = F().rootq_wt_prepare(_scalar(c.out["param_wt_upper"]), _scalar(c.out["param_wt_lower"]),
                                  _scalar(c.out["param_wt_alpha"]), ru, rl, m, g_w, wlo, whi, False)
        exact(F().rootq_wt_forward(dev(w), sw), c.out["qw"], "qw eval")
        exact(run, c.out["buf_in_run_scale"], "eval must not touch run_scale")
        return
    run = _scalar(c.inp["pre_in_run_scale"])
    st = F().rootq_act_prepare(_scalar(c.inp["pre_in_scale"]), run, m, g_i, ilo, ihi, True)
    exact(run, c.out["buf_in_run_scale"], "EMA'd run_scale")
    exact(F().rootq_act_forward(dev(x), st), c.out["qx"], "qx")
    dx, ds = F().rootq_act_backward(dev(x), dev(c.out["d_qx"]), st)
    assert torch.equal(dx.cpu() == 0, c.out["dx"] == 0)
    assert torch.allclose(dx.cpu(), c.out["dx"], rtol=1e-6, atol=0)
    red_close(ds, c.out["grad_in_scale"], abs_sum=(c.out["d_qx"].abs().sum() * ihi * m * g_i).reshape(1), rtol=1e-5)

    ru, rl = _scalar(c.inp["pre_wt_run_upper"]), _scalar(c.inp["pre_wt_run_lower"])
    sw = F().rootq_wt_prepare(_scalar(c.inp["pre_wt_upper"]), _scalar(c.inp["pre_wt_lower"]),
                              _scalar(c.inp["pre_wt_alpha"]), ru, rl, m, g_w, wlo, whi, True)
    exact(ru, c.out["buf_wt_run_upper"], "run_upper")
    exact(rl, c.out["buf_wt_run_lower"], "run_lower")
    exact(F().rootq_wt_forward(dev(w), sw), c.out["qw"], "qw")
    dw, gr = F().rootq_wt_backward(dev(w), dev(c.out["d_qw"]), sw)
    assert torch.allclose(dw.cpu(), c.out["grad_weight"], rtol=1e-5, atol=1e-8)      # north_star: 1e-5 relative
    floor = c.out["d_qw"].abs().sum() * whi * m * g_w
    red_close(gr[0], c.out["grad_wt_upper"], abs_sum=floor.reshape(1), rtol=1e-5)
    red_close(gr[1], c.out["grad_wt_lower"], abs_sum=floor.reshape(1), rtol=1e-5)
    red_close(gr[2], c.out["grad_wt_alpha"], abs_sum=(c.out["d_qw"].abs().sum() * 1e-3).reshape(1), rtol=1e-5)


@pytest.mark.parametrize("wbits,abits,mom,alpha", [(4, 4, 0.1, 0.25), (2, 3, 0.3, 0.6), (8, 8, 0.05, 1.7), (3, 4, 0.1, -0.2)])
def test_rootq_vs_oracle_large(wbits, abits, mom, alpha):
    """C1-sized tensors (ResNet-18 CIFAR: 128x64x32x32 activations, 512x512x3x3 weights scaled down)."""
    gen = torch.Generator().manual_seed(100 + wbits)
    x = torch.relu(torch.randn(16, 64, 32, 32, generator=gen)) * 1.3
    w = torch.randn(128, 256, 3, 3, generator=gen) * 0.03
    dyx, dyw = torch.randn(x.shape, generator=gen), torch.randn(w.shape, generator=gen)
    ilo, ihi = R.qrange(False, abits)
    wlo, whi = R.qrange(False, wbits)
    in_scale = R.rootq_act_init(x, ilo, ihi) * 0.9
    run_scale = in_scale * 1.05
    up, dn = R.rootq_wt_init(w, whi)
    up, dn = (up * 0.8).float(), (dn * 1.1).float()
    run_up, run_dn = up * 1.02, dn * 0.97
    a = torch.tensor(alpha)
    y, new_run, dx_ref, ds_ref = R.rootq_act_fwd_bwd(x, in_scale, run_scale, mom, ilo, ihi, dyx)
    g_i, g_w = 1 / math.sqrt(x.numel() * ihi), 1 / math.sqrt(w.numel() * whi)
    run = _scalar(run_scale)
    st = F().rootq_act_prepare(_scalar(in_scale), run, mom, g_i, ilo, ihi, True)
    exact(run, new_run, "run_scale")
    exact(F().rootq_act_forward(dev(x), st), y, "act fwd")
    dx, ds = F().rootq_act_backward(dev(x), dev(dyx), st)
    assert torch.equal(dx.cpu() == 0, dx_ref == 0) and torch.allclose(dx.cpu(), dx_ref, rtol=1e-6, atol=0)
    red_close(ds, ds_ref, abs_sum=(dyx.abs().sum() * ihi * mom * g_i).reshape(1))

    yw, nru, nrl, dw_ref, du, dl, da = R.rootq_wt_fwd_bwd(w, up, dn, a, run_up, run_dn, mom, wlo, whi, dyw)
    ru, rl = _scalar(run_up), _scalar(run_dn)
    sw = F().rootq_wt_prepare(_scalar(up), _scalar(dn), _scalar(a), ru, rl, mom, g_w, wlo, whi, True)
    exact(ru, nru, "run_upper")
    exact(rl, nrl, "run_lower")
    exact(F().rootq_wt_forward(dev(w), sw), yw, "wt fwd")
    dw, gr = F().rootq_wt_backward(dev(w), dev(dyw), sw)
    assert torch.allclose(dw.cpu(), dw_ref, rtol=1e-5, atol=1e-7)
    floor = (dyw.abs().sum() * whi * mom * g_w).reshape(1)
    red_close(gr[0], du, abs_sum=floor)
    red_close(gr[1], dl, abs_sum=floor)
    red_close(gr[2], da, abs_sum=(dyw.abs().sum() * 1e-3).reshape(1))


def test_rootq_clipping_special_values():
    c = ROOTQ["clipping_0_15"]
    # clipping(x, 15, 0) followed by round(x/1)*1 : use scale 1 so that y = round_pass(clip(x))
    run = torch.tensor(1.0).cuda()
    st = F().rootq_act_prepare(torch.tensor(1.0).cuda(), run, 0.1, 0.01, 0, 15, False)
    y = F().rootq_act_forward(dev(c.inp["x"]), st)
    ref, _ = R.rootq_act(c.inp["x"], torch.tensor(1.0), torch.tensor(1.0), 0.1, 0, 15, False)
    exact(y, ref, "rootq act on special values")


# --------------------------------------------------------------------------------------
OBS = load("observers")


def _kind(name):
    return name.split("_")[0] + "_" + name.split("_")[1]


@pytest.mark.parametrize("name", sorted(n for n in OBS if n.startswith("minmax_tensor") or n.startswith("minmax_channel")))
def test_golden_minmax(name):
    c = OBS[name]
    t = c.inp["t"]
    ax = c.meta.get("ch_axis") if name.startswith("minmax_channel") else None
    stats = F().obs_stats(dev(t), ch_axis=ax)
    s, o = F().minmax_from_stats(stats, c.meta["n_bits"], c.meta["signed"])
    exact(s, c.out["scale"].reshape(-1), "scale")
    exact(o, c.out["offset"].reshape(-1), "offset")


@pytest.mark.parametrize("name", sorted(n for n in OBS if n.startswith("l2loss_tensor")))
def test_golden_sweep_tensor(name):
    c = OBS[name]
    t = c.inp["t"]
    if c.meta["signed"]:
        pytest.skip("signed l2loss_tensor is the min/max answer (ops.py:37-40), covered by test_golden_minmax")
    s, o, picked = F().sweep_tensor(dev(t), c.meta["n_bits"])
    ref_s, ref_o, ref_pick = R.obs_l2loss_tensor(t, c.meta["n_bits"], False, return_index=True)
    assert c.meta["picked"] == ref_pick
    if int(picked) == ref_pick:
        exact(s, c.out["scale"].reshape(-1), "scale")
        exact(o, c.out["offset"].reshape(-1), "offset")
    else:   # near-tie between two candidates decided by summation order: losses must agree to 1e-5
        sse = F().sweep_tensor_sse(dev(t), F().obs_stats(dev(t)), c.meta["n_bits"]).cpu()
        assert abs(float(sse[int(picked)]) - float(sse[ref_pick])) <= 1e-5 * float(sse[ref_pick])


def _sweep_loss(row, scale, zp, qmax):
    r = row.double()
    q = (torch.round(r / float(scale)) + float(zp)).clamp(0, qmax)
    return float((((q - float(zp)) * float(scale)) - r).pow(2).sum())


def _sweep_rows_equivalent(rows, s, o, ref_s, ref_o, n_bits):
    """Rows must pick the reference's (scale, zero point); where they do not, the two candidates
    must be a genuine near-tie: for signed weights the search clamps every negative value to 0
    (reference quirk), so all 80 losses share one huge constant and differ in the 7th digit - the
    accept decision is then summation-order noise even between fp32 and fp64 on the CPU."""
    qmax = 2 ** n_bits - 1
    same = (s == ref_s) & (o == ref_o)
    for r in torch.nonzero(~same).flatten().tolist():
        mine, ref = _sweep_loss(rows[r], s[r], o[r], qmax), _sweep_loss(rows[r], ref_s[r], ref_o[r], qmax)
        assert abs(mine - ref) <= 2e-5 * abs(ref) + 1e-12, (r, mine, ref, float(s[r]), float(ref_s[r]))
    assert same.float().mean() >= 0.5, f"only {same.float().mean():.2f} of rows identical"


@pytest.mark.parametrize("name", sorted(n for n in OBS if n.startswith("l2loss_channel")))
def test_golden_sweep_channel(name):
    c = OBS[name]
    t = c.inp["t"]
    rows = t.reshape(t.shape[0], -1)
    s, o = F().sweep_channel(dev(rows), c.meta["n_bits"], c.meta["signed"])
    ref_s, ref_o = c.out["scale"].reshape(-1), c.out["offset"].reshape(-1)
    _sweep_rows_equivalent(rows, s.cpu(), o.cpu(), ref_s, ref_o, c.meta["n_bits"])


@pytest.mark.parametrize("name", sorted(n for n in OBS if n.startswith("l2norm_")))
def test_golden_l2norm(name):
    c = OBS[name]
    t = c.inp["t"]
    signed, bits = c.meta["signed"], c.meta["n_bits"]
    lo, hi = R.qrange(signed, bits)
    per_channel = name.startswith("l2norm_channel")
    rows = t.reshape(t.shape[0], -1) if per_channel else t.reshape(1, -1)
    stats = F().obs_stats(dev(rows), ch_axis=0 if per_channel else None)
    s0, o0 = F().minmax_from_stats(stats, bits, signed)
    s, iters, done = F().l2norm_fixed_point(dev(rows), s0, o0, lo, hi)
    assert done, "did not converge although the reference did"
    assert torch.allclose(s.cpu(), c.out["scale"].reshape(-1), rtol=2e-4), (s.cpu(), c.out["scale"].reshape(-1))


def test_sweep_tensor_vs_oracle_large():
    gen = torch.Generator().manual_seed(9)
    t = torch.relu(torch.randn(8, 32, 28, 28, generator=gen)) * 2 + 0.0
    for bits in (4, 8):
        s, o, picked = F().sweep_tensor(dev(t), bits)
        rs, ro, rp = R.obs_l2loss_tensor(t, bits, False, return_index=True)
        assert abs(int(picked) - rp) <= 1, (int(picked), rp)
        if int(picked) == rp:
            exact(s, rs.reshape(1), "scale")
            exact(o, ro.reshape(1).float(), "zero point")


def test_sweep_channel_vs_oracle_rows():
    """Signed weights (the search clamps to [0, qmax] - reference quirk) and shifted positive rows
    (exercise the aliasing of the running minimum), row lengths 27..4608 and > shared-memory cap."""
    gen = torch.Generator().manual_seed(10)
    for shape, kind in [((48, 27), "wt"), ((16, 576), "wt"), ((8, 4608), "wt"), ((6, 50), "shift"), ((3, 7000), "wt"),
                        ((5, 147), "shift")]:
        t = torch.randn(shape, generator=gen) * 0.02 if kind == "wt" else torch.rand(shape, generator=gen) * 3 + 0.75
        for signed in (True, False):
            s, o = F().sweep_channel(dev(t), 4, signed)
            rs, ro = R.obs_l2loss_channel(t.clone(), 4, signed)
            _sweep_rows_equivalent(t, s.cpu(), o.cpu(), rs.reshape(-1), ro.reshape(-1), 4)


def test_stats_nan_and_layouts():
    gen = torch.Generator().manual_seed(12)
    t = torch.randn(4, 6, 7, 7, generator=gen)
    st = F().obs_stats(dev(t), ch_axis=1).cpu()
    rows = t.transpose(0, 1).reshape(6, -1)
    assert torch.equal(st[:, 0], rows.min(1)[0]) and torch.equal(st[:, 1], rows.max(1)[0])
    assert torch.equal(st[:, 2], rows.abs().max(1)[0])
    assert torch.allclose(st[:, 3], rows.abs().sum(1), rtol=1e-5)
    t2 = t.clone()
    t2[1, 2, 3, 3] = float("nan")
    st = F().obs_stats(dev(t2), ch_axis=1).cpu()
    assert torch.isnan(st[2]).all() and not torch.isnan(st[[0, 1, 3, 4, 5]]).any()   # torch.min/max propagate NaN
    big = torch.randn((1 << 22) + 5, generator=gen)
    st = F().obs_stats(dev(big)).cpu()[0]
    assert st[0] == big.min() and st[1] == big.max() and st[2] == big.abs().max()
    assert abs(float(st[3]) - float(big.abs().double().sum())) <= 1e-5 * float(st[3])


def test_absmean_initialisers():
    gen = torch.Generator().manual_seed(13)
    x = torch.randn(64, 3, 3, 3, generator=gen) * 0.1
    stats = F().obs_stats(dev(x))
    lsq = F().absmean_from_stats(stats, x.numel(), 2.0, math.sqrt(7), 0).cpu()
    assert torch.allclose(lsq, R.lsq_init_scale(x, 7).reshape(1), rtol=1e-6)
    up = F().absmean_from_stats(stats, x.numel(), 2.0, math.sqrt(15), 1).cpu()
    assert torch.allclose(up, R.rootq_wt_init(x, 15)[0].reshape(1).float(), rtol=1e-6)


def test_grouped_matches_single_launches():
    """All weight tensors of a model in one launch == the per-tensor launches, bit for bit."""
    from dlmc_quant_b200.functional import GroupedFakeQuant
    gen = torch.Generator().manual_seed(14)
    shapes = [(64, 147), (64, 64), (128, 1152), (256, 2304), (512, 4608), (1000, 2048), (32, 9)]
    entries, singles = [], []
    for i, (c, k) in enumerate(shapes):
        per_channel = i % 2 == 0
        w = dev(torch.randn(c, k, generator=gen) * 0.03)
        dy = dev(torch.randn(c, k, generator=gen))
        nch = c if per_channel else 1
        scale = dev(torch.rand(nch, generator=gen) * 0.004 + 0.004)
        form = 3 if per_channel else 1
        g = 1 / math.sqrt(c * k * 7)
        e = dict(x=w, y=torch.empty_like(w), dy=dy, scale=scale, offset=None, dscale=torch.zeros(nch, device="cuda"),
                 channels=nch, inner=k if per_channel else c * k, form=form, lo=-7, hi=7, g=g)
        entries.append(e)
        singles.append((w, dy, scale, form, g, 0 if per_channel else None))
    grp = GroupedFakeQuant("cuda")
    grp.forward(entries)
    for e, (w, dy, scale, form, g, ax) in zip(entries, singles):
        assert torch.equal(e["y"], F().fq_forward(w, scale, None, -7, 7, form, g=g, ch_axis=ax))
    outs = [e["y"].clone() for e in entries]
    bentries = [dict(e, y=torch.empty_like(e["x"])) for e in entries]
    grp2 = GroupedFakeQuant("cuda")
    grp2.backward(bentries)
    for e, (w, dy, scale, form, g, ax) in zip(bentries, singles):
        dx, ds = F().fq_backward(w, dy, scale, None, -7, 7, form, g=g, ch_axis=ax)
        assert torch.equal(e["y"], dx)
        red_close(e["dscale"], ds, abs_sum=(dy.abs().sum() * 7).expand(ds.numel()) * (g if form == 1 else 1.0), rtol=1e-5)
    assert all(torch.equal(a, e["y"]) for a, e in zip(outs, entries))


def test_host_pipeline_matches_device_path():
    from dlmc_quant_b200.functional import HostFakeQuant
    gen = torch.Generator().manual_seed(15)
    n = (1 << 21) + 1000
    x = (torch.relu(torch.randn(n, generator=gen)) * 2).pin_memory()
    dy = torch.randn(n, generator=gen).pin_memory()
    y, dx = torch.empty(n).pin_memory(), torch.empty(n).pin_memory()
    hq = HostFakeQuant("cuda", chunk_elems=1 << 19)
    g = R.lsq_g(n, 15)
    ds = hq.forward_backward(x, dy, y, dx, 0.25, 0.0, 0, 15, form=1, g=g)
    s, o = dev(torch.tensor([0.25])), dev(torch.tensor([0.0]))
    assert torch.equal(y, F().fq_forward(dev(x), s, o, 0, 15, 1, g=g).cpu())
    dxd, dsd = F().fq_backward(dev(x), dev(dy), s, o, 0, 15, 1, g=g)
    assert torch.equal(dx, dxd.cpu())
    assert abs(ds - float(dsd)) <= 1e-5 * abs(float(dsd)) + 1e-7
    # async form: several tensors in flight, one synchronize
    outs = []
    for k in range(3):
        yk, dxk, dsk = torch.empty(n).pin_memory(), torch.empty(n).pin_memory(), torch.zeros(1).pin_memory()
        hq.forward_backward_async(x, dy, yk, dxk, dsk, 0.25 + 0.05 * k, 0.0, 0, 15, form=1, g=g)
        outs.append((yk, dxk, dsk, 0.25 + 0.05 * k))
    hq.synchronize()
    for yk, dxk, dsk, sk in outs:
        sd = dev(torch.tensor([sk]))
        assert torch.equal(yk, F().fq_forward(dev(x), sd, o, 0, 15, 1, g=g).cpu())
        dxd, dsd = F().fq_backward(dev(x), dev(dy), sd, o, 0, 15, 1, g=g)
        assert torch.equal(dxk, dxd.cpu()) and abs(float(dsk) - float(dsd)) <= 1e-5 * abs(float(dsd)) + 1e-7


def test_host_compact_wire_format_is_lossless():
    """dlmcq_host_ctx_fq_codes: packed integer codes + one keep bit per element come back over PCIe instead of y and dx
    (8.6 instead of 16 bytes per fp32 element); both reconstruct the full-precision results bit for bit:
    y == import_codes(codes) == fq_forward(x), dx == where(keep, dy, 0) == fq_backward(x, dy)."""
    import numpy as np
    from dlmc_quant_b200.functional import HostFakeQuant
    gen = torch.Generator().manual_seed(16)
    n = (1 << 20) + 1003                                   # ragged: not a multiple of 8, several chunks
    x = (torch.relu(torch.randn(n, generator=gen)) * 2).pin_memory()
    dy = torch.randn(n, generator=gen).pin_memory()
    hq = HostFakeQuant("cuda", chunk_elems=1 << 18)
    g = R.lsq_g(n, 15)
    s, o = dev(torch.tensor([0.23])), dev(torch.tensor([0.0]))
    y_ref = F().fq_forward(dev(x), s, o, 0, 15, 1, g=g).cpu()
    dx_ref, ds_ref = F().fq_backward(dev(x), dev(dy), s, o, 0, 15, 1, g=g)
    for pack4 in (True, False):
        codes = torch.zeros((n + 1) // 2 if pack4 else n, dtype=torch.uint8).pin_memory()
        keep = torch.zeros((n + 7) // 8, dtype=torch.uint8).pin_memory()
        ds = torch.zeros(1).pin_memory()
        hq.codes_async(x, dy, codes, keep, ds, 0.23, 0.0, 0, 15, form=1, g=g, pack4=pack4)
        hq.synchronize()
        want = F().export_codes(dev(x), s, o, 0, 15, 1, g=g, pack4=pack4).cpu().reshape(-1)
        assert torch.equal(codes, want)
        y = F().import_codes(dev(codes), (n,), s, o, 0, 15, 1, g=g, pack4=pack4).cpu()
        assert torch.equal(y, y_ref)
        bits = torch.from_numpy(np.unpackbits(keep.numpy(), bitorder="little")[:n].astype(bool))
        assert torch.equal(torch.where(bits, dy, torch.zeros(())), dx_ref.cpu())
        assert abs(float(ds) - float(ds_ref)) <= 1e-5 * abs(float(ds_ref)) + 1e-7
    # signed 8-bit weights, SYM form, forward only
    w = (torch.randn(70001, generator=gen) * 0.05).pin_memory()
    c8 = torch.zeros(70001, dtype=torch.int8).pin_memory()
    hq.codes_async(w, None, c8, None, None, 0.0011, 0.0, -127, 127, form=3)
    hq.synchronize()
    sw = dev(torch.tensor([0.0011]))
    assert torch.equal(c8, F().export_codes(dev(w), sw, None, -127, 127, 3).cpu().reshape(-1))
    # two contexts are independent; a context can be closed and another created
    hq2 = HostFakeQuant("cuda", chunk_elems=1 << 16)
    y2, dx2 = torch.empty(n).pin_memory(), torch.empty(n).pin_memory()
    assert abs(hq2.forward_backward(x, dy, y2, dx2, 0.23, 0.0, 0, 15, form=1, g=g) - float(ds_ref)) <= 1e-5 * abs(float(ds_ref)) + 1e-7
    assert torch.equal(y2, y_ref) and torch.equal(dx2, dx_ref.cpu())
    hq.close(); hq2.close()


# --------------------------------------------------------------------------------------
# geometry coverage of the observer kernels added in the second half of round 1
def test_sweep_channel_unstaged_rows_bf16_and_block_geometry():
    gen = torch.Generator().manual_seed(21)
    # a row longer than the shared-memory staging cap (200 KB) is swept from global memory
    t = torch.rand(2, 60000, generator=gen) * 3 + 0.5
    s, o = F().sweep_channel(dev(t), 4, False)
    rs, ro = R.obs_l2loss_channel(t.clone(), 4, False)
    _sweep_rows_equivalent(t, s.cpu(), o.cpu(), rs.reshape(-1), ro.reshape(-1), 4)
    # bf16 rows: converted while staging, fp32 arithmetic on the up-converted values
    tb = (torch.rand(24, 1152, generator=gen) * 2 + 0.25).to(torch.bfloat16)
    s, o = F().sweep_channel(dev(tb), 8, False)
    rs, ro = R.obs_l2loss_channel(tb.float(), 8, False)
    _sweep_rows_equivalent(tb.float(), s.cpu(), o.cpu(), rs.reshape(-1), ro.reshape(-1), 8)
    # one rank's block of rows, swept with the geometry of the whole matrix, gets the same bits as the
    # unsharded sweep (dist.rows_sharded relies on this)
    w = torch.randn(64, 2304, generator=gen) * 0.02
    s_all, o_all = F().sweep_channel(dev(w), 4, True)
    for lo_r, hi_r in ((0, 32), (32, 64), (5, 6)):
        s_b, o_b = F().sweep_channel(dev(w[lo_r:hi_r]), 4, True, geom_channels=64)
        assert torch.equal(s_b, s_all[lo_r:hi_r]) and torch.equal(o_b, o_all[lo_r:hi_r])


@pytest.mark.parametrize("shape", [(400, 6, 7, 7), (150, 6, 14, 14), (260, 5, 8, 8)])
def test_channel_major_kernels_with_several_batch_chunks(shape):
    """[B, C, h, w] activations with small planes and B*h*w > 8192: every channel is covered by several (channel,
    batch chunk) work items whose partial statistics / scale gradients are combined by the CTA-per-channel
    finalisers.  7x7: scalar accesses; 14x14 and 8x8: rows are whole 128-bit vectors (vectorised variant)."""
    gen = torch.Generator().manual_seed(22)
    x = torch.relu(torch.randn(shape, generator=gen)) * 1.5
    dy = torch.randn(x.shape, generator=gen)
    st = F().obs_stats(dev(x), ch_axis=1).cpu()
    rows = x.transpose(0, 1).reshape(shape[1], -1)
    assert torch.equal(st[:, 0], rows.min(1)[0]) and torch.equal(st[:, 1], rows.max(1)[0])
    assert torch.equal(st[:, 2], rows.abs().max(1)[0]) and torch.allclose(st[:, 3], rows.abs().sum(1), rtol=1e-5)
    xn = x.clone()
    xn[shape[0] - 1, 4, shape[2] - 1, shape[3] - 1] = float("nan")
    stn = F().obs_stats(dev(xn), ch_axis=1).cpu()
    others = [c for c in range(shape[1]) if c != 4]
    assert torch.isnan(stn[4]).all() and not torch.isnan(stn[others]).any()
    scale, off = R.obs_minmax_channel(x, 4, False, ch_axis=1)
    g = R.lsq_g(x.numel(), 15)
    xs, ss = x.clone().requires_grad_(True), scale.clone().requires_grad_(True)
    y_ref = R.fq_affine(xs, ss, off, 0, 15, g)
    dx_ref, ds_ref = torch.autograd.grad(y_ref, (xs, ss), dy)
    y = F().fq_forward(dev(x), dev(scale), dev(off), 0, 15, 1, g=g, ch_axis=1)
    exact(y, y_ref.detach(), "y")
    dx, ds = F().fq_backward(dev(x), dev(dy), dev(scale), dev(off), 0, 15, 1, g=g, ch_axis=1)
    assert torch.equal(dx.cpu() == 0, dx_ref == 0) and torch.allclose(dx.cpu(), dx_ref, rtol=1e-6, atol=0)
    red_close(ds, ds_ref.reshape(-1), abs_sum=dy.abs().sum(dim=(0, 2, 3)) * 15 * g)


@pytest.mark.parametrize("shape,dtype", [
    ((400, 8, 7, 7), torch.float32),        # G = 4 channels per 49-vector run, several batch chunks
    ((300, 12, 5, 5), torch.float32),       # 25-vector runs
    ((257, 16, 3, 3), torch.float32),       # 9-vector runs, ragged last pass
    ((1000, 64, 1, 1), torch.float32),      # inner == 1: a vector is four channels
    ((90, 6, 5, 10), torch.float32),        # inner % 4 == 2: G = 2
    ((3, 2048, 7, 7), torch.float32),       # fewer batch indices than rows per pass
    ((200, 16, 7, 7), torch.bfloat16),      # VEC = 8: G = 8, one channel per warp in the CTA fold
    ((130, 8, 3, 5), torch.bfloat16),       # inner = 15, G = 8, 15-vector runs
])
def test_slab_kernels_for_rows_that_are_not_whole_vectors(shape, dtype):
    """stats_slab_kernel / fq_slab_kernel (per-channel activations with short, unaligned rows read as 128-bit vectors
    across G adjacent channels): statistics, forward (AFFINE and ZP forms, codes too), backward and the NaN rule equal
    the oracle exactly as the scalar channel-major kernels did; a channel count that is not a multiple of G still takes
    the scalar kernels and gives the same bits."""
    gen = torch.Generator().manual_seed(hash(shape) % 1000)
    x = (torch.relu(torch.randn(shape, generator=gen)) * 1.5 - 0.1).to(dtype)
    dy = torch.randn(x.shape, generator=gen).to(dtype)
    xf, dyf = x.float(), dy.float()
    C = shape[1]
    st = F().obs_stats(dev(x), ch_axis=1).cpu()
    rows = xf.transpose(0, 1).reshape(C, -1)
    assert torch.equal(st[:, 0], rows.min(1)[0]) and torch.equal(st[:, 1], rows.max(1)[0])
    assert torch.equal(st[:, 2], rows.abs().max(1)[0]) and torch.allclose(st[:, 3], rows.abs().sum(1), rtol=1e-5)
    xn = x.clone()
    xn[shape[0] - 1, C - 3, shape[2] - 1, shape[3] - 1] = float("nan")
    stn = F().obs_stats(dev(xn), ch_axis=1).cpu()
    others = [c for c in range(C) if c != C - 3]
    assert torch.isnan(stn[C - 3]).all() and not torch.isnan(stn[others]).any()
    scale, off = R.obs_minmax_channel(xf, 4, False, ch_axis=1)
    g = R.lsq_g(x.numel(), 15)
    xs, ss = xf.clone().requires_grad_(True), scale.clone().requires_grad_(True)
    y_ref = R.fq_affine(xs, ss, off, 0, 15, g)
    dx_ref, ds_ref = torch.autograd.grad(y_ref, (xs, ss), dyf)
    y = F().fq_forward(dev(x), dev(scale), dev(off), 0, 15, 1, g=g, ch_axis=1)
    exact(y.float(), y_ref.detach().to(dtype).float(), "y")
    dx, ds = F().fq_backward(dev(x), dev(dy), dev(scale), dev(off), 0, 15, 1, g=g, ch_axis=1)
    # the reference's dx is (dy * s') / s' where in range: up to 1 ulp off dy (the kernels return dy itself)
    assert torch.equal(dx.float().cpu() == 0, dx_ref == 0) and torch.allclose(dx.float().cpu(), dx_ref, rtol=1e-6 if dtype is torch.float32 else 4e-3, atol=0)
    red_close(ds, ds_ref.reshape(-1), abs_sum=dyf.abs().sum(dim=(0, 2, 3)) * 15 * g)
    # zero-point form, with codes
    zp = torch.arange(C, dtype=torch.float32).reshape(1, C, 1, 1) % 5
    s2 = (scale.reshape(1, C, 1, 1) * 0.7 + 0.01)
    y2_ref, dx2_ref, ds2_ref = R.fq_zp_fwd_bwd(xf, s2, zp, 0, 15, dyf)[:3]
    y2 = F().fq_forward(dev(x), dev(s2.reshape(-1)), dev(zp.reshape(-1)), 0, 15, 2, ch_axis=1)
    exact(y2.float(), y2_ref.to(dtype).float(), "y zp")
    dx2, ds2 = F().fq_backward(dev(x), dev(dy), dev(s2.reshape(-1)), dev(zp.reshape(-1)), 0, 15, 2, ch_axis=1)
    assert torch.equal(dx2.float().cpu() == 0, dx2_ref == 0) and torch.allclose(dx2.float().cpu(), dx2_ref, rtol=1e-6 if dtype is torch.float32 else 4e-3, atol=0)
    red_close(ds2, ds2_ref.reshape(-1), abs_sum=dyf.abs().sum(dim=(0, 2, 3)) * 16)
    # odd channel count: the scalar channel-major kernels, same bits on the shared channels
    if C > 4:
        xo, dyo = x[:, :C - 1].contiguous(), dy[:, :C - 1].contiguous()
        so, oo = scale.reshape(-1)[:C - 1].contiguous(), off.reshape(-1)[:C - 1].contiguous()
        yo = F().fq_forward(dev(xo), dev(so), dev(oo), 0, 15, 1, g=g, ch_axis=1)
        exact(yo, y[:, :C - 1], "slab vs scalar channel-major forward")
        dxo, dso = F().fq_backward(dev(xo), dev(dyo), dev(so), dev(oo), 0, 15, 1, g=g, ch_axis=1)
        exact(dxo, dx[:, :C - 1], "slab vs scalar channel-major backward")
        red_close(dso, ds[:C - 1], abs_sum=dyf[:, :C - 1].abs().sum(dim=(0, 2, 3)) * 15 * g)
        assert torch.equal(F().obs_stats(dev(xo), ch_axis=1).cpu()[:, :3], st[:C - 1, :3])


def test_l2norm_per_channel_multi_cta_finalise():
    """More than 256 channels: the new scales, the global stopping rule and the done flag are produced by
    several finalising CTAs plus a last-ticket combination."""
    gen = torch.Generator().manual_seed(23)
    w = torch.randn(600, 96, generator=gen) * 0.05
    lo, hi = R.qrange(True, 4)
    rs, ro, ref_iters = R.obs_l2norm_channel(w, 4, True, return_iters=True)
    stats = F().obs_stats(dev(w), ch_axis=0)
    s0, o0 = F().minmax_from_stats(stats, 4, True)
    s, iters, done = F().l2norm_fixed_point(dev(w), s0, o0, lo, hi)
    assert done and abs(int(iters) - ref_iters) <= 2, (int(iters), ref_iters)
    assert torch.allclose(s.cpu(), rs.reshape(-1), rtol=2e-4)


# --------------------------------------------------------------------------------------
# percentile observer (north-star extension): exact order statistics == torch.kthvalue
@pytest.mark.parametrize("n", [1, 7, 1000, (1 << 20) + 13])
@pytest.mark.parametrize("kind", ["randn", "relu", "const", "special"])
def test_kth_values_equal_torch_kthvalue(n, kind):
    gen = torch.Generator().manual_seed(31 + n)
    x = torch.randn(n, generator=gen) * 3
    if kind == "relu":
        x = torch.relu(x)                          # half of the elements in one histogram bin
    elif kind == "const":
        x = torch.full((n,), -1.25)
    elif kind == "special":
        x[::5] = 0.0
        x[1::7] = -0.0
        if n > 20:
            x[3], x[4], x[11], x[12] = float("inf"), float("-inf"), 1e-45, -1e-45
    for dtype in (torch.float32, torch.bfloat16):
        xd = x.to(dtype)
        ranks = sorted({1, n, (n + 1) // 2, max(1, n - n // 1000), min(n, 1 + n // 1000)})
        for i in range(0, len(ranks), 2):
            pair = ranks[i:i + 2]
            got = F().kth_values(dev(xd), pair).cpu()
            want = torch.stack([xd.float().kthvalue(k)[0] for k in pair])
            assert torch.equal(got, want), (n, kind, dtype, pair, got, want)
            got_abs = F().kth_values(dev(xd), pair, abs_input=True).cpu()
            want_abs = torch.stack([xd.float().abs().kthvalue(k)[0] for k in pair])
            assert torch.equal(got_abs, want_abs), (n, kind, dtype, pair, got_abs, want_abs)


def test_kth_values_nan_sorts_last_and_multidim():
    x = torch.tensor([[3.0, float("nan")], [-2.0, 5.0]])
    got = F().kth_values(dev(x), [3, 4]).cpu()
    assert got[0] == 5.0 and torch.isnan(got[1])                       # like torch.sort: NaN is the largest
    t = torch.randn(4, 8, 14, 14, generator=torch.Generator().manual_seed(5))
    assert F().kth_values(dev(t), [100]).cpu()[0] == t.flatten().kthvalue(100)[0]


@pytest.mark.parametrize("signed,bits,pct", [(False, 4, 99.9), (False, 8, 99.99), (True, 4, 99.0), (True, 8, 100.0)])
def test_percentile_observer_vs_oracle(signed, bits, pct):
    from dlmc_quant_b200.scalar import ops
    gen = torch.Generator().manual_seed(41)
    t = torch.randn(16, 32, 28, 28, generator=gen) * 2
    if not signed:
        t = torch.relu(t) + 0.125
    s, o = ops.get_qparams_tensor(dev(t), "percentile_tensor", n_bits=bits, signed=signed, percentile=pct)
    rs, ro = R.obs_percentile_tensor(t, bits, signed, pct)
    exact(s.reshape(1), rs.reshape(1), "scale")
    exact(o.reshape(1), ro.reshape(1).float(), "offset")
    if pct == 100.0:                                                    # degenerates to the min/max observer
        ms, mo = ops.quantize_minmax_tensor(dev(t), bits, signed)
        assert torch.equal(ms, s) and torch.equal(mo.float(), o.float())


def test_grouped_rootq_matches_per_layer_launches():
    """One prepare launch for all quantizers and one forward / backward launch for all weight tensors give the
    per-layer entry points' results: states, running buffers, w_q and dw bit for bit, reduced gradients to 1e-5."""
    from dlmc_quant_b200 import functional as Fn
    gen = torch.Generator().manual_seed(51)
    lo, hi, mom = 0, 15, 0.1
    shapes = [(64, 3, 3, 3), (128, 64, 3, 3), (10, 512), (7,), (300, 33)]
    layers = []
    for shp in shapes:
        w = (torch.randn(shp, generator=gen) * 0.05).cuda()
        dy = torch.randn(shp, generator=gen).cuda()
        up, dn = R.rootq_wt_init(w.cpu(), hi)
        x = torch.relu(torch.randn(4, 8, 6, 6, generator=gen)).cuda()
        in_scale = R.rootq_act_init(x.cpu(), lo, hi).cuda()
        layers.append(dict(w=w, dy=dy, up=up.float().cuda(), dn=dn.float().cuda(), alpha=torch.tensor(0.3).cuda(),
                           in_scale=in_scale, g_w=1 / math.sqrt(w.numel() * hi), g_i=1 / math.sqrt(x.numel() * hi)))
    # per-layer reference path
    ref = []
    for L in layers:
        rup, rdn, run = L["up"].clone() * 0.9, L["dn"].clone() * 1.1, L["in_scale"].clone() * 0.8
        sa = Fn.rootq_act_prepare(L["in_scale"], run, mom, L["g_i"], lo, hi, True)
        sw = Fn.rootq_wt_prepare(L["up"], L["dn"], L["alpha"], rup, rdn, mom, L["g_w"], lo, hi, True)
        wq = Fn.rootq_wt_forward(L["w"], sw)
        dw, gw = Fn.rootq_wt_backward(L["w"], L["dy"], sw)
        ref.append(dict(sa=sa, sw=sw, wq=wq, dw=dw, gw=gw, rup=rup, rdn=rdn, run=run))
    # grouped path
    G = Fn.GroupedRootQ("cuda")
    qs, bufs = [], []
    for L in layers:
        rup, rdn, run = L["up"].clone() * 0.9, L["dn"].clone() * 1.1, L["in_scale"].clone() * 0.8
        bufs.append((rup, rdn, run))
        qs.append(dict(kind="act", in_scale=L["in_scale"], run_scale=run, momentum=mom, g=L["g_i"], lo=lo, hi=hi, training=True))
        qs.append(dict(kind="wt", upper=L["up"], lower=L["dn"], alpha=L["alpha"], run_upper=rup, run_lower=rdn,
                       momentum=mom, g=L["g_w"], lo=lo, hi=hi, training=True))
    states = G.prepare(qs)
    ent = [dict(w=L["w"], out=torch.empty_like(L["w"]), state=states[2 * i + 1]) for i, L in enumerate(layers)]
    G.wt_forward(ent)
    bent = [dict(w=L["w"], dy=L["dy"], out=torch.empty_like(L["w"]), state=states[2 * i + 1],
                 grads=torch.empty(3, device="cuda")) for i, L in enumerate(layers)]
    G.wt_backward(bent)
    for i, (L, r) in enumerate(zip(layers, ref)):
        assert torch.equal(states[2 * i][:5], r["sa"][:5]) and torch.equal(states[2 * i + 1], r["sw"]), i
        assert torch.equal(bufs[i][0], r["rup"]) and torch.equal(bufs[i][1], r["rdn"]) and torch.equal(bufs[i][2], r["run"])
        assert bits_equal(ent[i]["out"].cpu(), r["wq"].cpu()), i
        assert bits_equal(bent[i]["out"].cpu(), r["dw"].cpu()), i
        assert torch.allclose(bent[i]["grads"], r["gw"], rtol=1e-5, atol=1e-6), (i, bent[i]["grads"], r["gw"])


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_grouped_rootq_activations_match_per_tensor_launches(dtype):
    """dlmcq_rootq_act_forward_grouped / _backward_grouped: several activation tensors (ragged sizes, a misaligned
    view, an empty tensor, one that spans many work units, two quantizers reading the SAME tensor as a residual
    block's main and shortcut convolutions do) in one launch per direction give the per-tensor entries' x_q and dx
    bit for bit and d in_scale to 1e-5."""
    from dlmc_quant_b200 import functional as Fn
    gen = torch.Generator().manual_seed(77)
    lo, hi, mom = 0, 15, 0.1
    base = torch.randn(70_001, generator=gen)
    xs = [torch.relu(torch.randn(8, 16, 12, 12, generator=gen)) * 2, torch.randn(3, 5, generator=gen) * 4,
          torch.randn(1_000_003, generator=gen) * 3, base[1:], torch.empty(0), torch.randn(2048 * 3, generator=gen)]
    xs = [x.to(dtype).cuda() for x in xs]
    xs[3] = base.to(dtype).cuda()[1:]                       # not 16-byte aligned: scalar path
    xs.append(xs[0])                                        # second quantizer on the first tensor
    G = Fn.GroupedRootQ("cuda")
    qs, ref = [], []
    for i, x in enumerate(xs):
        in_scale = torch.tensor([0.05 + 0.07 * i], device="cuda")
        g = 1 / math.sqrt(max(x.numel(), 1) * hi)
        run = in_scale.clone() * 0.8
        sa = Fn.rootq_act_prepare(in_scale, run.clone(), mom, g, lo, hi, True)
        dy = torch.randn(x.shape, generator=gen).to(dtype).cuda()
        y = Fn.rootq_act_forward(x, sa) if x.numel() else x.clone()
        dx, ds = Fn.rootq_act_backward(x, dy, sa) if x.numel() else (x.clone(), torch.zeros(1, device="cuda"))
        ref.append(dict(y=y, dx=dx, ds=ds, dy=dy))
        qs.append(dict(kind="act", in_scale=in_scale, run_scale=run, momentum=mom, g=g, lo=lo, hi=hi, training=True))
    states = G.prepare(qs)
    fwd = [dict(w=x, out=torch.full_like(x, float("nan")), state=states[i]) for i, x in enumerate(xs)]
    G.act_forward(fwd, dtype)
    bwd = [dict(w=x, dy=ref[i]["dy"], out=torch.full_like(x, float("nan")), state=states[i],
                grads=torch.full((1,), float("nan"), device="cuda")) for i, x in enumerate(xs)]
    G.act_backward(bwd, dtype)
    for i, r in enumerate(ref):
        assert bits_equal(fwd[i]["out"].float().cpu(), r["y"].float().cpu()), i
        assert bits_equal(bwd[i]["out"].float().cpu(), r["dx"].float().cpu()), i
        want = r["ds"].reshape(-1)[:1]
        floor = 4e-7 * float(r["dy"].float().abs().sum()) * hi * float(states[i][2]) * float(states[i][3]) if xs[i].numel() else 0
        assert torch.allclose(bwd[i]["grads"], want, rtol=1e-5, atol=max(floor, 1e-9)), (i, bwd[i]["grads"], want)


# --------------------------------------------------------------------------------------
# full-size (2^26 elements), size-independent properties of the observers and of RootQ
def test_full_size_observer_and_rootq_properties():
    from dlmc_quant_b200 import functional as Fn
    n = 1 << 26
    torch.manual_seed(2333)
    x = torch.relu(torch.randn(n, device="cuda")) * 2
    half = n // 2
    # statistics of a concatenation = merge of the parts' statistics
    st, s0, s1 = Fn.obs_stats(x), Fn.obs_stats(x[:half]), Fn.obs_stats(x[half:])
    assert st[0, 0] == torch.minimum(s0[0, 0], s1[0, 0]) and st[0, 1] == torch.maximum(s0[0, 1], s1[0, 1])
    assert abs(float(st[0, 3]) - float(s0[0, 3]) - float(s1[0, 3])) <= 1e-5 * float(st[0, 3])
    # the 80 sweep sums are additive over a split of the tensor (same candidates: the whole tensor's statistics)
    sse = Fn.sweep_tensor_sse(x, st, 8).double()
    parts = Fn.sweep_tensor_sse(x[:half], st, 8).double() + Fn.sweep_tensor_sse(x[half:], st, 8).double()
    assert torch.allclose(sse, parts, rtol=1e-5)
    # ... and equal to the eager evaluation of one candidate on the GPU (ops.py:53-61), candidate 17
    r = torch.tensor(1.0 - 0.01 * 17, dtype=torch.float32, device="cuda")
    c_hi, c_lo = r * st[0, 1], r * st[0, 0]
    sc = (c_hi - c_lo) / 255
    zp = torch.round(-c_lo / sc)
    xq = ((torch.round(x / sc) + zp).clamp(0, 255) - zp) * sc
    want = float(((xq - x) ** 2).double().sum())
    assert abs(float(sse[17]) - want) <= 2e-5 * want
    # exact order statistics against a full sort
    ranks = [n // 1000, n - n // 1000]
    srt = torch.sort(x).values
    assert torch.equal(Fn.kth_values(x, ranks), torch.stack([srt[k - 1] for k in ranks]))
    del srt, xq
    # RootQ: the quantised weights lie on the 16-level grid {L + j*delta} - plus the 15 interval midpoints, which
    # the reference produces for inputs exactly on a midpoint (sgn(0) = 0, RootQ/function.py:58-67; a handful of
    # the 6.7e7 samples) - and re-quantising changes nothing
    w = torch.randn(n, device="cuda") * 0.05
    up, lo_b = torch.tensor(0.12, device="cuda"), torch.tensor(-0.11, device="cuda")
    state = Fn.rootq_wt_prepare(up, lo_b, torch.tensor(0.3, device="cuda"), up.clone(), lo_b.clone(), 0.1,
                                1 / math.sqrt(n * 15), 0, 15, False)
    wq = Fn.rootq_wt_forward(w, state)
    assert torch.unique(wq).numel() <= 31
    assert torch.equal(Fn.rootq_wt_forward(wq, state), wq)
    # RootQ activations: idempotent, bounded by [0, run_scale * 15], backward linear in dy
    sa = Fn.rootq_act_prepare(torch.tensor(0.5, device="cuda"), torch.tensor(0.5, device="cuda"), 0.1,
                              1 / math.sqrt(n * 15), 0, 15, False)
    y = Fn.rootq_act_forward(x, sa)
    assert torch.equal(Fn.rootq_act_forward(y, sa), y) and float(y.min()) >= 0 and float(y.max()) <= 7.5 + 1e-6
    dy = torch.randn(n, device="cuda")
    dx1, g1 = Fn.rootq_act_backward(x, dy, sa)
    dx2, g2 = Fn.rootq_act_backward(x, dy * 2, sa)
    assert torch.equal(dx2, dx1 * 2) and abs(float(g2) - 2 * float(g1)) <= 1e-5 * abs(float(g2)) + 1e-7


# --------------------------------------------------------------------------------------
# bf16 tensors (API extension, SURVEY.md A.8 vi): reference(x.float()) rounded once to bf16; reductions in fp32
def test_bf16_rootq_and_observers():
    from dlmc_quant_b200 import functional as Fn
    gen = torch.Generator().manual_seed(61)
    bf = torch.bfloat16
    x = (torch.relu(torch.randn(8, 32, 16, 16, generator=gen)) * 1.3).to(bf)
    w = (torch.randn(64, 96, 3, 3, generator=gen) * 0.03).to(bf)
    dyx, dyw = torch.randn(x.shape, generator=gen).to(bf), torch.randn(w.shape, generator=gen).to(bf)
    lo, hi, mom = 0, 15, 0.1
    in_scale = R.rootq_act_init(x.float(), lo, hi) * 0.9
    run_scale = in_scale * 1.05
    up, dn = R.rootq_wt_init(w.float(), hi)
    up, dn = (up * 0.8).float(), (dn * 1.1).float()
    a = torch.tensor(0.4)
    # activations
    y_ref, _, dx_ref, ds_ref = R.rootq_act_fwd_bwd(x.float(), in_scale, run_scale, mom, lo, hi, dyx.float())
    g_i = 1 / math.sqrt(x.numel() * hi)
    st = Fn.rootq_act_prepare(_scalar(in_scale), _scalar(run_scale), mom, g_i, lo, hi, True)
    y = Fn.rootq_act_forward(dev(x), st)
    assert y.dtype == bf and bits_equal(y.float().cpu(), y_ref.to(bf).float())
    dx, ds = Fn.rootq_act_backward(dev(x), dev(dyx), st)
    assert dx.dtype == bf and bits_equal(dx.float().cpu(), dx_ref.to(bf).float())
    red_close(ds, ds_ref, abs_sum=(dyx.float().abs().sum() * hi * mom * g_i).reshape(1))
    # weights
    yw_ref, _, _, dw_ref, du, dl, da = R.rootq_wt_fwd_bwd(w.float(), up, dn, a, up * 1.02, dn * 0.97, mom, lo, hi, dyw.float())
    g_w = 1 / math.sqrt(w.numel() * hi)
    sw = Fn.rootq_wt_prepare(_scalar(up), _scalar(dn), _scalar(a), _scalar(up * 1.02), _scalar(dn * 0.97), mom, g_w,
                             lo, hi, True)
    yw = Fn.rootq_wt_forward(dev(w), sw)
    assert yw.dtype == bf and bits_equal(yw.float().cpu(), yw_ref.to(bf).float())
    dw, gr = Fn.rootq_wt_backward(dev(w), dev(dyw), sw)
    assert torch.allclose(dw.float().cpu(), dw_ref, rtol=2 ** -7, atol=1e-6)      # one bf16 rounding of the result
    floor = (dyw.float().abs().sum() * hi * mom * g_w).reshape(1)
    red_close(gr[0], du, abs_sum=floor)
    red_close(gr[1], dl, abs_sum=floor)
    # observers on bf16 data == observers on the up-converted data
    t = (torch.relu(torch.randn(6, 24, 14, 14, generator=gen)) * 2).to(bf)
    for ch_axis in (None, 1):
        sb = Fn.obs_stats(dev(t), ch_axis=ch_axis).cpu()
        sf = Fn.obs_stats(dev(t.float()), ch_axis=ch_axis).cpu()
        assert torch.equal(sb[:, :3], sf[:, :3]) and torch.allclose(sb[:, 3], sf[:, 3], rtol=1e-6)
    s, o, picked = Fn.sweep_tensor(dev(t), 8)
    rs, ro, rp = R.obs_l2loss_tensor(t.float(), 8, False, return_index=True)
    assert abs(int(picked) - rp) <= 1
    if int(picked) == rp:
        exact(s, rs.reshape(1), "scale")
    rows = t.reshape(6, -1)
    st4 = Fn.obs_stats(dev(rows), ch_axis=0)
    s0, o0 = Fn.minmax_from_stats(st4, 4, False)
    sb, itb, doneb = Fn.l2norm_fixed_point(dev(rows), s0, o0, 0, 15, max_iters=200)
    sf, itf, donef = Fn.l2norm_fixed_point(dev(rows.float()), s0, o0, 0, 15, max_iters=200)
    assert doneb == donef and torch.allclose(sb, sf, rtol=1e-5)


def _sweep_plan(rows2d):
    """dlmcq_obs_sweep_channel_plan for a [channels, inner] matrix: the launch geometry sweep_channel gives it."""
    import ctypes as C
    from dlmc_quant_b200 import _lib
    ch, inner = rows2d.shape
    it = _lib.SweepItem(channels=ch, inner=inner)
    _lib.check(_lib.lib().dlmcq_obs_sweep_channel_plan(C.byref(it), ch))
    return it


def _sweep_channel_with_wpr(rows2d, n_bits, signed, wpr):
    """sweep_channel of one fp32 matrix through dlmcq_obs_sweep_channel_grouped, with `wpr` warps per row set by hand
    instead of the plan's choice (8 warps per CTA: 8 / wpr rows per CTA, each staged in row_floats floats)."""
    import ctypes as C
    from dlmc_quant_b200 import _lib
    ch = rows2d.shape[0]
    out = torch.empty(2, ch, dtype=torch.float32, device=rows2d.device)
    it = _sweep_plan(rows2d)
    assert it.staged == 1
    it.x, it.scale, it.offset = rows2d.data_ptr(), out[0].data_ptr(), out[1].data_ptr()
    it.n_bits, it.is_signed, it.wpr = n_bits, int(signed), wpr
    it.ctas = (ch * wpr + 7) // 8
    it.smem_bytes = (8 // wpr) * it.row_floats * 4
    tab = torch.frombuffer(bytearray(bytes(it)), dtype=torch.uint8).to(rows2d.device)
    pre = torch.zeros(1, dtype=torch.int64, device=rows2d.device)
    _lib.check(_lib.lib().dlmcq_obs_sweep_channel_grouped(C.c_void_p(tab.data_ptr()), C.c_void_p(pre.data_ptr()), 1,
                                                          it.ctas, _lib.F32, it.smem_bytes, None))
    torch.cuda.synchronize()
    return out[0], out[1]


def test_reductions_are_deterministic_run_to_run():
    """Every reduction on the path is fixed-order (no floating-point atomics): repeated launches on the same input
    return the same bits - also a race detector for the multi-warp channel sweep (shared-memory exchange + named
    barriers) under every warps-per-row setting."""
    from dlmc_quant_b200 import functional as Fn
    gen = torch.Generator().manual_seed(71)
    for inner, wpr in ((100, 1), (300, 2), (700, 4), (2304, 8)):     # the plan's warps per row for 96 rows of `inner`
        w = dev(torch.randn(96, inner, generator=gen) * 0.02)
        assert _sweep_plan(w).wpr == wpr, inner
        first = Fn.sweep_channel(w, 4, True)
        for _ in range(10):
            again = Fn.sweep_channel(w, 4, True)
            assert torch.equal(first[0], again[0]) and torch.equal(first[1], again[1]), wpr
    x = dev(torch.relu(torch.randn(1 << 22, generator=gen)) * 2)
    dy = dev(torch.randn(1 << 22, generator=gen))
    xa = dev(torch.relu(torch.randn(64, 48, 14, 14, generator=gen)))
    dya = dev(torch.randn(64, 48, 14, 14, generator=gen))
    st = Fn.obs_stats(x)
    scale, off = Fn.minmax_from_stats(st, 4, False)
    ref = (Fn.fq_backward(x, dy, scale, off, 0, 15, 1, g=1e-3)[1], Fn.sweep_tensor_sse(x, st, 8), Fn.obs_stats(x),
           Fn.kth_values(x, [1000, 4000000]))
    sa, oa = Fn.minmax_from_stats(Fn.obs_stats(xa, ch_axis=1), 4, False)
    ref_a = Fn.fq_backward(xa, dya, sa, oa, 0, 15, 1, g=1e-3, ch_axis=1)[1]
    for _ in range(10):
        got = (Fn.fq_backward(x, dy, scale, off, 0, 15, 1, g=1e-3)[1], Fn.sweep_tensor_sse(x, st, 8), Fn.obs_stats(x),
               Fn.kth_values(x, [1000, 4000000]))
        assert all(torch.equal(a, b) for a, b in zip(ref, got))
        assert torch.equal(ref_a, Fn.fq_backward(xa, dya, sa, oa, 0, 15, 1, g=1e-3, ch_axis=1)[1])


def test_sweep_channel_edge_rows_under_every_geometry():
    """NaN rows, constant rows (zero scale: literal chain), all-zero rows, single-element rows and rows shorter than
    the number of lanes, with 1..8 warps per row (warps without elements must still take part in the exchange)."""
    from dlmc_quant_b200 import functional as Fn
    gen = torch.Generator().manual_seed(81)
    cases = []
    for inner, wpr in ((100, 1), (300, 2), (700, 4), (1100, 8)):     # the plan's warps per row for 6 rows of `inner`
        t = torch.rand(6, inner, generator=gen) * 3 + 0.5
        t[1, 13] = float("nan")
        t[2] = 1.75
        t[3] = 0.0
        t[4, ::2] = 0.0
        assert _sweep_plan(t).wpr == wpr, inner
        cases.append(t)
    short = [torch.rand(5, 1, generator=gen) + 0.1, torch.rand(3, 5, generator=gen) * 2,
             torch.randn(4, 33, generator=gen) * 0.02]
    # the plan gives these short rows one warp each; more warps per row only through a hand-set geometry
    runs = [(t, None) for t in cases + short] + [(t, wpr) for t in short for wpr in (2, 4, 8)]
    for t, wpr in runs:
        for signed in (False, True):
            if wpr is None:
                s, o = Fn.sweep_channel(dev(t), 4, signed)
            else:
                s, o = _sweep_channel_with_wpr(dev(t), 4, signed, wpr)
            rs, ro = R.obs_l2loss_channel(t.clone(), 4, signed)
            rs, ro = rs.reshape(-1), ro.reshape(-1).float()
            s, o = s.cpu(), o.cpu()
            nan_rows = torch.isnan(rs)
            assert torch.equal(torch.isnan(s), nan_rows) and torch.equal(torch.isnan(o), torch.isnan(ro)), (wpr, t.shape)
            ok = ~nan_rows
            _sweep_rows_equivalent(t[ok], s[ok], o[ok], rs[ok], ro[ok], 4)


def test_grouped_channel_sweep_is_bit_identical_to_per_tensor_sweeps():
    """dlmcq_obs_sweep_channel_grouped: all weight tensors of a model in one launch per shared-memory class; every
    tensor keeps its own launch geometry, so (scale, offset) equal the per-tensor sweeps bit for bit - and
    calibrate.init_weight_quantizers gives the same state as the lazy per-layer initialisation."""
    import copy
    from dlmc_quant_b200 import functional as Fm
    gen = torch.Generator().manual_seed(321)
    shapes = [(64, 147), (64, 64), (64, 576), (256, 64), (512, 4608), (2048, 512), (1000, 2048), (48, 27), (7, 13),
              (96, 864), (3, 20000)]
    rows = [(torch.randn(s, generator=gen) * 0.05).cuda() for s in shapes]
    for signed in (True, False):
        got = Fm.sweep_channel_grouped(rows, 4, signed)
        for r, (s, o) in zip(rows, got):
            s1, o1 = Fm.sweep_channel(r, 4, signed)
            assert torch.equal(s, s1) and torch.equal(o, o1), (tuple(r.shape), signed)
    rows_bf = [r.bfloat16() for r in rows[:6]]
    for r, (s, o) in zip(rows_bf, Fm.sweep_channel_grouped(rows_bf, 8, True)):
        s1, o1 = Fm.sweep_channel(r, 8, True)
        assert torch.equal(s, s1) and torch.equal(o, o1)

    from dlmc_quant_b200 import quantize_model
    from dlmc_quant_b200.calibrate import init_weight_quantizers
    cfg = {"weight": {"enable": True, "type": "l2loss_channel", "args": {"n_bits": 4, "signed": True, "ch_axis": 0}},
           "input": {"enable": True, "type": "minmax_tensor", "args": {"n_bits": 8, "signed": False}},
           "exclude_layers": [], "override_options": [], "momentum": 0.1}
    torch.manual_seed(5)
    net = torch.nn.Sequential(torch.nn.Conv2d(3, 16, 3, padding=1), torch.nn.ReLU(), torch.nn.Conv2d(16, 24, 3, padding=1),
                              torch.nn.AdaptiveAvgPool2d(1), torch.nn.Flatten(), torch.nn.Linear(24, 10)).cuda()
    for family in (None, "FSPTQ"):
        a, b = copy.deepcopy(net), copy.deepcopy(net)
        quantize_model(a, copy.deepcopy(cfg), None, quantization_type=family)
        quantize_model(b, copy.deepcopy(cfg), None, quantization_type=family)
        assert init_weight_quantizers(b) == 3 and init_weight_quantizers(b) == 0
        x = torch.rand(4, 3, 8, 8, device="cuda")
        with torch.no_grad():
            ya, yb = a(x), b(x)
        assert torch.equal(ya, yb)
        for (n, p), (_, q) in zip(a.state_dict().items(), b.state_dict().items()):
            assert torch.equal(p, q), (family, n)


def test_resident_l2norm_matches_the_stepwise_loop_and_the_oracle():
    """dlmcq_obs_l2norm_resident: the whole fixed point of ops.py:71-83 / 198-215 in one cooperative launch on rows
    staged in shared memory.  Same arithmetic per iteration as the step-wise kernels (summation order differs):
    converged scales within 1e-5 of them and of the oracle loop; large tensors report "not resident" and fall back."""
    from dlmc_quant_b200 import functional as Fm
    gen = torch.Generator().manual_seed(77)
    for shape, bits, signed in [((64, 576), 4, True), ((512, 4608), 4, True), ((1000, 2048), 8, True), ((1, 300000), 4, True),
                                ((7, 13), 4, True), ((96, 864), 8, True), ((1, 1 << 20), 4, True)]:
        w = (torch.randn(shape, generator=gen) * 0.05)
        if not signed:
            w = w.abs()
        wd = w.cuda()
        st = Fm.obs_stats(wd, ch_axis=0)
        s0, o0 = Fm.minmax_from_stats(st, bits, signed)
        lo, hi = R.qrange(signed, bits)
        s_res, it_res, done_res = Fm.l2norm_fixed_point(wd, s0, o0, lo, hi, max_iters=300, resident=True)
        s_stp, it_stp, done_stp = Fm.l2norm_fixed_point(wd, s0, o0, lo, hi, max_iters=300, resident=False)
        assert done_res and done_stp, (shape, it_res, it_stp)
        assert torch.allclose(s_res, s_stp, rtol=2e-5, atol=0), (shape, float((s_res / s_stp - 1).abs().max()))
        assert abs(it_res - it_stp) <= 3, (shape, it_res, it_stp)
        if shape[0] > 1:
            rs, _ = R.obs_l2norm_channel(w, bits, signed, ch_axis=0)
        else:
            rs, _ = R.obs_l2norm_tensor(w.reshape(-1), bits, signed)
        # the loop stops when ONE step moves the scale VECTOR by <= 1e-5 in relative 2-norm (ops.py:209): single rows may
        # still move by 1e-5 * sqrt(C), so two implementations are compared in the norm the criterion itself uses
        rel = float((s_res.cpu() - rs.reshape(-1)).norm() / rs.norm())
        assert rel <= 3e-4, (shape, rel)
    # run-to-run deterministic
    a = Fm.l2norm_fixed_point(wd, s0, o0, lo, hi, resident=True)[0]
    b = Fm.l2norm_fixed_point(wd, s0, o0, lo, hi, resident=True)[0]
    assert torch.equal(a, b)
    # not resident: 2^25 elements cannot be staged on chip -> the step-wise loop runs instead (same API, same answer)
    big = (torch.randn(1, 1 << 25, generator=gen) * 0.05).cuda()
    sb, ob = Fm.minmax_from_stats(Fm.obs_stats(big, ch_axis=0), 4, True)
    s1, _, d1 = Fm.l2norm_fixed_point(big, sb, ob, -7, 7, resident=True)
    s2, _, d2 = Fm.l2norm_fixed_point(big, sb, ob, -7, 7, resident=False)
    assert d1 and d2 and torch.equal(s1, s2)
    # bounded: the reference's loop never terminates on some inputs; max_iters stops the resident loop too
    _, it, done = Fm.l2norm_fixed_point(wd, s0, o0, lo, hi, max_iters=2, resident=True)
    assert it == 2 and not done


def test_one_read_kth_value_survives_a_missed_bracket():
    """The sample positions are a fixed hash of the index: plant values there that misplace the bracket for the rank
    asked (all samples huge, the tensor otherwise small): status must report the miss and the values must still equal
    torch.kthvalue - for one rank, two ranks, |x| and bf16."""
    import ctypes as C
    from dlmc_quant_b200 import _lib
    n = 1_500_001
    gen = torch.Generator().manual_seed(3)
    x = torch.randn(n, generator=gen)
    i = torch.arange(16384, dtype=torch.int64)
    hsh = (i * 2654435761 + 0x9e3779b9) & 0xffffffff
    idx = (hsh * n) >> 32
    x[idx] = 1000.0 + torch.arange(16384, dtype=torch.float32)           # every sample lies above the true quantiles
    h = _lib.lib()
    for dtype in (torch.float32, torch.bfloat16):
        xd = x.to(dtype).cuda()
        srt = xd.float().cpu().sort()[0]
        asrt = xd.float().cpu().abs().sort()[0]
        nws = h.dlmcq_obs_kth_fast_workspace_bytes(n)
        ws = torch.empty(nws, dtype=torch.uint8, device="cuda")
        for ranks, flags, ref in (((n // 2, 0), 0, srt), ((n // 4, 3 * n // 4), 0, srt), ((n // 2, n - 20000), 1, asrt)):
            vals = torch.zeros(2, device="cuda")
            status = torch.full((1,), 7, dtype=torch.int32, device="cuda")
            _lib.check(h.dlmcq_obs_kth_fast(C.c_void_p(xd.data_ptr()), n, 0 if dtype is torch.float32 else 1, flags,
                                            ranks[0], ranks[1], C.c_void_p(vals.data_ptr()),
                                            C.c_void_p(status.data_ptr()), C.c_void_p(ws.data_ptr()), nws, None))
            torch.cuda.synchronize()
            assert int(status) == 0, (dtype, ranks)
            for j, k in enumerate(ranks):
                if k:
                    assert vals[j].cpu() == ref[k - 1], (dtype, ranks, j, vals, ref[k - 1])


@pytest.mark.parametrize("kind", ["randn", "relu", "relu6", "const", "sorted", "periodic", "heavy_tail"])
def test_one_read_kth_value_is_exact(kind):
    """dlmcq_obs_kth_fast (sample bracket -> one counting / collecting read -> exact select among the candidates) equals
    torch.kthvalue on every rank asked, and reports status 1 on ordinary data; where the bracket cannot hold the same
    launch runs the full three-digit select in-kernel (status 0) and the value is exact all the same."""
    n = 3_000_017
    gen = torch.Generator().manual_seed(11)
    x = torch.randn(n, generator=gen) * 2
    if kind == "relu":
        x = torch.relu(x)
    elif kind == "relu6":
        x = torch.clamp(torch.relu(x * 3), max=6.0)              # two values (0, 6) hold most of the tensor
    elif kind == "const":
        x = torch.full((n,), 0.75)
    elif kind == "sorted":
        x = x.sort()[0]
    elif kind == "periodic":
        x = torch.sin(torch.arange(n, dtype=torch.float32) * (2 * 3.14159265 / 4096)) * 3
    elif kind == "heavy_tail":
        x = x * torch.exp(torch.randn(n, generator=gen) * 2)
    xd = x.cuda()
    srt = x.sort()[0]
    asrt = x.abs().sort()[0]
    for p in (99.99, 99.9, 99.0, 50.0, 0.01):
        k_hi = min(n, max(1, int(-(-p * n // 100))))
        k_lo = n + 1 - k_hi
        got = F().kth_values(xd, sorted({k_lo, k_hi})).cpu()
        want = torch.stack([srt[k - 1] for k in sorted({k_lo, k_hi})])
        assert torch.equal(got, want), (kind, p, got, want)
        ga = F().kth_values(xd, [k_hi], abs_input=True).cpu()
        assert ga[0] == asrt[k_hi - 1], (kind, p)
    # the fast path's own verdict, through the C ABI
    import ctypes as C
    from dlmc_quant_b200 import _lib
    h = _lib.lib()
    nws = h.dlmcq_obs_kth_fast_workspace_bytes(n)
    ws = torch.zeros(nws, dtype=torch.uint8, device="cuda")
    vals = torch.zeros(2, device="cuda")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    k = int(0.999 * n)
    _lib.check(h.dlmcq_obs_kth_fast(C.c_void_p(xd.data_ptr()), n, 0, 0, k, 0, C.c_void_p(vals.data_ptr()),
                                    C.c_void_p(status.data_ptr()), C.c_void_p(ws.data_ptr()), nws, None))
    torch.cuda.synchronize()
    assert vals[0].cpu() == srt[k - 1], kind          # exact whether the bracket held (1) or the in-kernel full select ran (0)
    assert int(status) == 1 or kind in ("sorted",), kind          # pseudo-random sample positions: only exotic orders miss
    bf = x[:1_000_003].bfloat16()
    assert F().kth_values(bf.cuda(), [999_000]).cpu()[0] == bf.float().sort()[0][999_000 - 1]
