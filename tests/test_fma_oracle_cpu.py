"""CPU: oracle/restate.py::fma_f32 (the single-rounding fp32 fma the fused BatchNorm tests compare against) against
exact rational arithmetic, on random triples and on hand-made cases where the float64 sum lands on an fp32 midpoint."""
from fractions import Fraction

import numpy as np
import torch

from oracle import restate as R


def _round_f32(v):
    """Correctly rounded (nearest, ties to even) fp32 of the rational v."""
    r0 = np.float32(float(v))                 # within one fp32 ulp of the answer
    cands = [np.nextafter(r0, np.float32(-np.inf)), r0, np.nextafter(r0, np.float32(np.inf))]
    best = None
    for c in cands:
        if not np.isfinite(c):
            continue
        d = abs(Fraction(float(c)) - v)
        key = (d, int(np.array(c, dtype=np.float32).view(np.uint32)) & 1)     # ties: the even significand
        if best is None or key < best[0]:
            best = (key, c)
    return best[1]


def _check(a, b, c):
    a, b, c = (np.asarray(v, dtype=np.float32) for v in (a, b, c))
    got = R.fma_f32(torch.from_numpy(a), torch.from_numpy(b), torch.from_numpy(c)).numpy()
    for i in range(a.size):
        exact = Fraction(float(a.flat[i])) * Fraction(float(b.flat[i])) + Fraction(float(c.flat[i]))
        want = _round_f32(exact)
        assert got.flat[i].view(np.uint32) == np.float32(want).view(np.uint32), \
            (float(a.flat[i]), float(b.flat[i]), float(c.flat[i]), float(got.flat[i]), float(want))


def test_fma_f32_random_triples():
    rng = np.random.default_rng(7)
    n = 3000
    a = (rng.standard_normal(n) * 2.0 ** rng.integers(-30, 30, n)).astype(np.float32)
    b = (rng.standard_normal(n) * 2.0 ** rng.integers(-30, 30, n)).astype(np.float32)
    c = (rng.standard_normal(n) * 2.0 ** rng.integers(-60, 60, n)).astype(np.float32)
    # near-cancellation: c close to -a*b, so the result's bits come from far below the product's leading bit
    k = n // 3
    c[:k] = (-(a[:k].astype(np.float64) * b[:k].astype(np.float64))).astype(np.float32)
    # BatchNorm-like operands: (x - mean) * (gamma * invstd) + beta
    t = rng.standard_normal(n).astype(np.float32)
    A = (rng.random(n) + 0.5).astype(np.float32)
    beta = (rng.standard_normal(n) * 0.3).astype(np.float32)
    _check(a, b, c)
    _check(t, A, beta)


def test_fma_f32_double_rounding_ties():
    """a*b = 1 + 2^-11 + 2^-24 is exactly the midpoint of two fp32 neighbours; a c below half a float64 ulp leaves the
    float64 sum on that midpoint, and only its sign decides the fp32 result (an fp32 tie rounds to even)."""
    h = np.float32(1 + 2.0 ** -12)
    cases = []
    for sa in (1.0, -1.0):
        for sc in (2.0 ** -60, -(2.0 ** -60), 0.0, 2.0 ** -140):
            for scale in (1.0, 2.0 ** 20, 2.0 ** -20):
                cases.append((np.float32(sa * h * scale), h, np.float32(sc * scale)))
    # the midpoint of 2^30 + 128 (odd significand) and 2^30 + 256: naive rounding of the float64 sum gives the even
    # neighbour whichever side the exact value lies
    cases.append((np.float32(1 + 2.0 ** -23), np.float32(64 * (1 - 2.0 ** -23)), np.float32(2.0 ** 30 + 128)))
    cases.append((np.float32(1 + 2.0 ** -12), np.float32(1 + 2.0 ** -12), np.float32(-(2.0 ** -70))))
    a, b, c = (np.array(v, dtype=np.float32) for v in zip(*cases))
    _check(a, b, c)
    # and the helper does differ from the naive rounding on the first case (so the test above has teeth)
    naive = (torch.tensor([float(h)]).double() * float(h) + 2.0 ** -60).float()
    fixed = R.fma_f32(torch.tensor([float(h)]), torch.tensor([float(h)]), torch.tensor([2.0 ** -60], dtype=torch.float32))
    assert not torch.equal(naive, fixed)


def test_fma_f32_non_finite():
    a = torch.tensor([float("inf"), float("nan"), 3e38, 1.0, -float("inf")])
    b = torch.tensor([2.0, 1.0, 10.0, 1.0, 0.5])
    c = torch.tensor([1.0, 0.0, 0.0, float("inf"), 1.0])
    got = R.fma_f32(a, b, c)
    assert got[0] == float("inf") and bool(torch.isnan(got[1])) and got[2] == float("inf")
    assert got[3] == float("inf") and got[4] == -float("inf")
