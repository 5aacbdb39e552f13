"""CPU checks of tests/adaround_terms.py: the float64 AdaRound terms against autograd of the oracle's chain, their
masks against the fp32 eager chain, and the row-vectorised MSE sweep against the oracle's double loop on rows of
every C3 and C4 weight shape (profiles/calibration_c3_c4.py)."""
import math

import pytest
import torch

from oracle import restate as R
from profiles.calibration_c3_c4 import mobileone_s0_layers, repvgg_a0_layers
from tests.adaround_terms import ada_terms, l2loss_channel_rows

LN11 = math.log(11.0)


def ada_inputs(c, k, dtype, seed, lo, hi):
    """Weights 0.03 N(0,1) with a few on multiples of s and past the clamp, alpha from the initialiser with some
    elements saturated on each side and some on 0 and +-ln 11."""
    gen = torch.Generator().manual_seed(seed)
    w = (torch.randn(c, k, generator=gen, dtype=torch.float64) * 0.03).to(dtype)
    s = (w.abs().amax(1, keepdim=True) / hi + 1e-6).to(dtype)
    w[:, 0] = s[:, 0] * 3
    w[:, 1] = s[:, 0] * (hi + 1.5)
    w[:, 2] = -s[:, 0] * (hi + 2.5)
    alpha = R.adaround_init_alpha(w, s).to(dtype)
    alpha.view(-1)[::7] = 6.0
    alpha.view(-1)[3::7] = -6.0
    alpha.view(-1)[5::11] = 0.0
    alpha.view(-1)[6::13] = LN11
    alpha.view(-1)[8::13] = -LN11
    dy = torch.randn(c, k, generator=gen, dtype=torch.float64).to(dtype)
    return w, s, alpha, dy


@pytest.mark.parametrize("bits", [4, 8])
def test_terms_equal_autograd_in_float64(bits):
    lo, hi = R.qrange(True, bits)
    w, s, alpha, dy = ada_inputs(16, 300, torch.float64, 5 + bits, lo, hi)
    alpha[0, 4] = float("nan")                     # autograd's d alpha is NaN there: 0 * sigmoid'(NaN)
    y, ds, da = R.fq_adaround_fwd_bwd(w, s, alpha, lo, hi, dy)
    t = ada_terms(w, alpha, s, dy, lo, hi)
    assert torch.allclose(t.y, y, rtol=1e-12, atol=0, equal_nan=True)
    assert torch.allclose(t.ds.sum(1, keepdim=True), ds, rtol=1e-12, atol=1e-300, equal_nan=True)
    assert torch.allclose(t.da, da, rtol=1e-12, atol=0, equal_nan=True)
    assert torch.equal(t.da.isnan(), da.isnan()) and int(da.isnan().sum()) == 1
    assert torch.equal(t.da != 0, da != 0)
    assert bool(t.mask.any()) and bool((~t.mask).any())
    assert bool((t.q > hi).any()) and bool((t.q < lo).any()), "the outer clamp must act on both sides"


@pytest.mark.parametrize("bits", [4, 8])
def test_masks_equal_fp32_eager_chain(bits):
    lo, hi = R.qrange(True, bits)
    w, s, alpha, dy = ada_inputs(32, 500, torch.float32, 17 + bits, lo, hi)
    t = ada_terms(w, alpha, s, dy, lo, hi)
    y32, _, da32 = R.fq_adaround_fwd_bwd(w, s, alpha, lo, hi, torch.ones_like(w))
    assert torch.equal(t.fl, torch.floor(w / s))
    near = t.near_pre | t.near_q
    assert torch.equal((da32 != 0)[~near], t.mask[~near])
    assert bool(t.near_pre.any()) and bool(t.near_q.any())          # the +-ln 11 and clamp-edge elements
    assert bool(t.mask[~near].any()) and bool((~t.mask[~near]).any())
    # the fp32 chain's soft forward is within a few ulp of the float64 one
    assert bool(((y32.double() - t.y).abs() <= 2.0 ** -22 * t.y.abs() + 2.0 ** -21 * s.double()).all())


def test_boundary_flags():
    """Elements placed on each edge are flagged, interior ones are not."""
    lo, hi = -7, 7
    s = torch.tensor([[0.25]])
    w = torch.tensor([[0.25 * 3, 0.25 * 3 + 0.1, -0.25 * 8, 0.25 * 7.0, 0.1]])
    alpha = torch.tensor([[0.0, 0.0, LN11, 0.0, -LN11]])
    t = ada_terms(w, alpha, s, torch.ones_like(w), lo, hi)
    assert t.near_int.tolist() == [[True, False, True, True, False]]
    assert t.near_pre[0, 2] and t.near_pre[0, 4] and not t.near_pre[0, 0]
    assert bool(t.near_q[0, 2]) and not bool(t.near_q[0, 0]) and not bool(t.near_q[0, 4])   # -8 + h(ln 11) ~ lo


def sweep_rows_sample(shape, gen, signed_rows):
    c = shape[0]
    k = math.prod(shape[1:])
    pick = torch.randperm(c, generator=gen)[:12]
    w = torch.randn(c, k, generator=gen) * 0.03
    rows = w[pick].contiguous()
    if not signed_rows:
        rows = rows.abs() + 0.01 * torch.rand(rows.shape[0], 1, generator=gen)
    return rows


@pytest.mark.parametrize("signed", [True, False], ids=["signed", "unsigned"])
@pytest.mark.parametrize("bits", [4, 8])
def test_vectorised_sweep_matches_oracle_loop(bits, signed):
    """Every distinct weight shape of C3 and C4 (row lengths 9 to 1728), signed weights and shifted positive rows;
    the oracle sees the same rows one at a time."""
    gen = torch.Generator().manual_seed(31 + bits)
    shapes = sorted({w for _, w in repvgg_a0_layers() + mobileone_s0_layers()})
    assert any(math.prod(w[1:]) == 9 for w in shapes)
    for shape in shapes:
        for signed_rows in (True, False):
            rows = sweep_rows_sample(shape, gen, signed_rows)
            s, o = l2loss_channel_rows(rows, bits, signed)
            rs, ro = R.obs_l2loss_channel(rows.clone(), bits, signed)
            assert torch.equal(s, rs.reshape(-1)), (shape, signed_rows)
            assert torch.equal(o, ro.reshape(-1)), (shape, signed_rows)
