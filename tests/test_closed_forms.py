"""CPU tests: the closed-form RootQ gradients (SURVEY.md A.5) that rootq_kernels.cu implements and
tests/rootq_terms.py restates in float64.

1. All inputs in float64: the terms, summed and chained (m * g for in_scale, wt_upper and wt_lower; the alpha clamp's
   mask for wt_alpha), equal torch.autograd of the oracle chain (oracle/restate.py::rootq_act_fwd_bwd,
   rootq_wt_fwd_bwd) to 1e-12 relative; dw and dx element by element to the same bar; the forward values are
   identical.  The inputs include the points where the chain's relus and floor switch: w exactly at L and at U,
   w on an interval midpoint (z = 0), x exactly at the clipping bound, and alpha at and beyond both clamp edges.
2. fp32 inputs: rootq_terms gives the plain-C oracle's (oracle/fq_oracle.c) forward values bit for bit and its
   float64 gradient sums to 1e-12 relative."""
import math

import numpy as np
import pytest
import torch

from oracle import c_oracle as CO
from oracle import restate as R
from tests.golden_io import bits_equal
from tests.rootq_terms import act_terms, wt_terms

LO, HI, MOM = 0, 15, 0.1
ALPHAS = (1e-4, 1.0, 1.3, -0.2, 0.25)   # at the lower clamp edge, at the upper, beyond each, inside


def rel_ok(got, want, what, rtol=1e-12):
    got, want = torch.as_tensor(got, dtype=torch.float64), torch.as_tensor(want, dtype=torch.float64)
    err = (got - want).abs()
    assert bool((err <= rtol * want.abs()).all()), f"{what}: worst relative error {float((err / want.abs()).max()):.3g}"


def act_inputs(dtype, seed):
    gen = torch.Generator().manual_seed(seed)
    x = torch.relu(torch.randn(4, 8, 9, 9, generator=gen)) * 2 - 0.05
    dy = torch.randn(x.shape, generator=gen)
    in_scale = R.rootq_act_init(x, LO, HI) * 0.5             # about a tenth of the elements clip at the top
    run = in_scale * 1.1
    x, dy, in_scale, run = (t.to(dtype) for t in (x, dy, in_scale, run))
    # the effective scale this step will use; put elements exactly on the clipping bound and on zero
    _, rs = R.rootq_act(x, in_scale, run, MOM, LO, HI, True)
    xf = x.reshape(-1)
    xf[:5] = rs * (HI - LO)
    xf[5], xf[6] = 0.0, -0.0
    return x, dy, in_scale, run


def wt_inputs(dtype, seed, shrink):
    """Weights whose bounds clip a share of them (shrink < 1), with elements exactly at L, at U and on
    interval midpoints of the bounds the step will use."""
    gen = torch.Generator().manual_seed(seed)
    w = torch.randn(16, 8, 3, 3, generator=gen) * 0.03
    dy = torch.randn(w.shape, generator=gen)
    up, dn = R.rootq_wt_init(w, HI)
    up, dn = (up * shrink).to(dtype), (dn * shrink * 0.8).to(dtype)
    rup, rdn = up * 1.05, dn * 0.9
    w, dy = w.to(dtype), dy.to(dtype)
    _, U, L = R.rootq_wt(w, up, dn, torch.tensor(0.5, dtype=dtype), rup, rdn, MOM, LO, HI, True)
    delta = (U - L) / torch.tensor(HI - LO, dtype=dtype)
    wf = w.reshape(-1)
    wf[:3], wf[3:6] = L, U
    for j in range(HI - LO):
        wf[6 + j] = (j + 0.5) * delta + L
    return w, dy, up, dn, rup, rdn


@pytest.mark.parametrize("seed", [1, 2])
def test_act_closed_form_equals_autograd_fp64(seed):
    x, dy, in_scale, run = act_inputs(torch.float64, seed)
    y, rs, dx, ds = R.rootq_act_fwd_bwd(x, in_scale, run, MOM, LO, HI, dy)
    a = act_terms(x, dy, rs, HI - LO)
    assert bits_equal(a.y, y)
    g = 1 / math.sqrt(x.numel() * HI)
    rel_ok(MOM * g * a.terms.sum(), ds.reshape(()), "d in_scale")
    assert torch.equal(dx == 0, ~a.keep)
    rel_ok(torch.where(a.keep, dy, 0.0)[a.keep], dx[a.keep], "dx")
    clip = (x >= rs * (HI - LO)) & (x > 0)
    assert 0.02 < float(clip.double().mean()) < 0.3 and bool(a.keep[x == rs * (HI - LO)].all())


@pytest.mark.parametrize("alpha", ALPHAS)
@pytest.mark.parametrize("shrink", [1.0, 0.4])
def test_wt_closed_form_equals_autograd_fp64(alpha, shrink):
    w, dy, up, dn, rup, rdn = wt_inputs(torch.float64, 3, shrink)
    a = torch.tensor(alpha, dtype=torch.float64)
    y, U, L, dw, du, dl, da = R.rootq_wt_fwd_bwd(w, up, dn, a, rup, rdn, MOM, LO, HI, dy)
    t = wt_terms(w, dy, U, L, a, HI - LO)
    assert bits_equal(t.y, y)
    z = w.reshape(-1)[6:6 + HI - LO] - ((torch.arange(HI - LO, dtype=torch.float64) + 0.5) * t.delta + L)
    assert int((z == 0).sum()) >= 8, "the midpoint inputs must hit z = 0"
    assert t.amask == (1.0 if 1e-4 <= alpha <= 1.0 else 0.0)
    g = 1 / math.sqrt(w.numel() * HI)
    s = t.terms.sum(1)
    rel_ok(MOM * g * s[0], du.reshape(()), "d wt_upper")
    rel_ok(MOM * g * s[1], dl.reshape(()), "d wt_lower")
    if t.amask:
        rel_ok(s[2], da.reshape(()), "d wt_alpha")
    else:
        assert float(da) == 0.0
    rel_ok(t.dw, dw, "dw")
    if shrink < 1:
        assert bool((t.dw == 0).any()), "some weights must clip"


@pytest.mark.parametrize("seed", [4, 5])
def test_act_terms_match_c_oracle_fp32(seed):
    x, dy, in_scale, run = act_inputs(torch.float32, seed)
    _, rs = R.rootq_act(x, in_scale, run, MOM, LO, HI, True)
    a = act_terms(x, dy, rs, HI - LO)
    y, dx, d = CO.rootq_act(x.numpy(), dy.numpy(), float(rs), np.float32(rs) * np.float32(HI - LO), HI - LO)
    assert bits_equal(torch.from_numpy(y).reshape(x.shape), a.y)
    assert bits_equal(torch.from_numpy(dx).reshape(x.shape), torch.where(a.keep, dy, 0.0))
    rel_ok(a.terms.sum(), d, "d in_scale terms")


@pytest.mark.parametrize("alpha", ALPHAS)
@pytest.mark.parametrize("shrink", [1.0, 0.4])
def test_wt_terms_match_c_oracle_fp32(alpha, shrink):
    w, dy, up, dn, rup, rdn = wt_inputs(torch.float32, 6, shrink)
    a = torch.tensor(alpha, dtype=torch.float32)
    _, U, L = R.rootq_wt(w, up, dn, a, rup, rdn, MOM, LO, HI, True)
    t = wt_terms(w, dy, U, L, a, HI - LO)
    y, dw, gr = CO.rootq_wt(w.numpy(), dy.numpy(), float(U), float(L), float(a), HI - LO)
    assert bits_equal(torch.from_numpy(y).reshape(w.shape), t.y)
    dwc = torch.from_numpy(dw).double().reshape(w.shape)
    assert bool(((dwc - t.dw).abs() <= 2.0 ** -24 * t.dw.abs()).all()), "dw beyond one fp32 rounding"
    for j, name in enumerate(("dU", "dL", "dalpha")):
        rel_ok(t.terms[j].sum(), gr[j], name + " terms")


@pytest.mark.parametrize("alpha", [0.25, 1.0])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_wt_level_sign_when_bounds_cross(alpha, dtype):
    """U < L makes delta and k negative, so b = k|z| + 1e-5 can be negative: the reference's level sign
    sgn(pow(b, alpha) * sg) is then 0 (pow is NaN) for a fractional alpha and -sign(z) for alpha == 1, not sign(z).
    rootq_terms and the C oracle follow the reference's forward value."""
    gen = torch.Generator().manual_seed(7)
    w = (torch.randn(300, generator=gen) * 0.05).to(dtype)
    up, dn, a = torch.tensor(-0.05, dtype=dtype), torch.tensor(0.05, dtype=dtype), torch.tensor(alpha, dtype=dtype)
    y, U, L = R.rootq_wt(w, up, dn, a, up.clone(), dn.clone(), MOM, LO, HI, True)
    assert float(U) < float(L)
    t = wt_terms(w, torch.ones_like(w), U, L, a, HI - LO)
    assert bits_equal(t.y, y)
    if dtype == torch.float32:
        yc, _, _ = CO.rootq_wt(w.numpy(), None, float(U), float(L), alpha, HI - LO)
        assert bits_equal(torch.from_numpy(yc), y)
