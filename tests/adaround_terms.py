"""Float64 reference of the AdaRound soft rounding (FSPTQuant/base.py:69-79,136-141,151-152) and a row-vectorised
restatement of the per-channel MSE sweep (ops.py:169-196), as device-agnostic torch functions.

floor(w / s) is formed in the inputs' dtype with the reference's own division, as the reference's fp32 tensors form
it; everything after that is evaluated in float64.  The constants zeta - gamma and gamma are the values the inputs'
dtype holds (1.2f and -0.1f for fp32, the Python doubles for float64), because that is what the reference's
`tensor * 1.2000000000000002` multiplies by.  The per-element terms are un-chained: d scale of a channel is the sum
of `ds` over its elements, d alpha is `da` itself."""
from collections import namedtuple

import torch

from oracle import restate as R

AdaTerms = namedtuple("AdaTerms", "y fl sg pre q ds da mask near_pre near_q near_int")

BOUNDARY = 2.0 ** -22          # distance to a mask edge below which fp32 and float64 may decide differently


def ada_terms(w, alpha, s, dy, lo, hi):
    """w, alpha, dy of one shape (fp32 or float64), s broadcastable to it (the per-channel scale).
    -> y (float64 soft forward), fl (floor(w / s), inputs' dtype), sg (float64 sigmoid(alpha)), pre / q (float64
    soft target before its clamp, and floor + h before the outer clamp), ds (float64 d scale terms dy * clamp(q)),
    da (float64 d alpha dy * s * (zeta - gamma) * sigma (1 - sigma) where both clamps pass), mask (both clamps pass), and per element
    whether it lies within BOUNDARY of a mask edge (pre near 0 or 1, q near lo or hi) or w / s within one ulp of
    an integer."""
    dt = w.dtype
    zg = float(torch.tensor(R.ADAROUND_ZETA - R.ADAROUND_GAMMA, dtype=dt))
    gm = float(torch.tensor(R.ADAROUND_GAMMA, dtype=dt))
    v = w / s
    fl = torch.floor(v)
    sg = torch.sigmoid(alpha.double())
    pre = sg * zg + gm
    h = pre.clamp(0.0, 1.0)
    q = fl.double() + h
    s64 = s.double()
    y = q.clamp(lo, hi) * s64
    d = dy.double()
    ds = d * q.clamp(lo, hi)
    in_q = (q >= lo) & (q <= hi)
    in_h = (pre >= 0.0) & (pre <= 1.0)
    mask = in_q & in_h
    da = torch.where(mask, d * s64 * zg, 0.0) * (sg * (1.0 - sg))       # a NaN alpha gives NaN, as in autograd
    near_pre = (pre.abs() <= BOUNDARY) | ((pre - 1.0).abs() <= BOUNDARY)
    near_q = ((q - lo).abs() <= BOUNDARY * max(1, abs(lo))) | ((q - hi).abs() <= BOUNDARY * max(1, abs(hi)))
    ulp = (torch.nextafter(v.abs(), torch.full_like(v, float("inf"))) - v.abs()).double()
    near_int = (v.double() - v.double().round()).abs() <= ulp
    return AdaTerms(y, fl, sg, pre, q, ds, da, mask, near_pre, near_q, near_int)


def l2loss_channel_rows(rows, n_bits, signed):
    """R.obs_l2loss_channel on a [channels, inner] matrix with the 80 candidates run in sequence for all rows at once.
    The reference's running minimum aliases the offset vector (ops.py:172,192): a row that accepts a candidate moves
    its own minimum, and only its own, so a per-row `where` reproduces the aliasing exactly.  The scalar divisions
    divide by a tensor, which is the IEEE quotient on every device (eager CUDA would multiply a Python-int divisor's
    reciprocal; the library divides, DESIGN.md §2).  -> (scale [C], offset [C])."""
    dt, dev = rows.dtype, rows.device
    if signed:
        scale = rows.abs().max(dim=1)[0] / torch.tensor(float(2 ** (n_bits - 1) - 1), dtype=dt, device=dev)
        offset = torch.zeros_like(scale)
    else:
        mn = rows.min(dim=1)[0]
        scale = (rows.max(dim=1)[0] - mn) / torch.tensor(float(2 ** n_bits - 1), dtype=dt, device=dev)
        offset = mn.clone()
    qmax = 2 ** n_bits - 1
    qm = torch.tensor(float(qmax), dtype=dt, device=dev)
    hi = offset + scale * qmax
    best = torch.full_like(scale, float(R.SWEEP_MIN_LOSS))
    for i in range(R.N_SWEEP):
        r = 1 - 0.01 * i
        c_lo, c_hi = r * offset, r * hi                   # offset is the aliased minimum
        c_scale = (c_hi - c_lo) / qm
        c_zp = torch.round(-c_lo / c_scale)
        q = torch.round(rows / c_scale[:, None])
        q = (q + c_zp[:, None]).clamp(0, qmax)
        q = (q - c_zp[:, None]) * c_scale[:, None]
        loss = ((rows - q) ** 2).sum(axis=1)              # l2_loss of one row: the mean over one row is the sum
        take = best > loss
        scale = torch.where(take, c_scale, scale)
        offset = torch.where(take, c_zp, offset)
        best = torch.where(take, loss, best)
    return scale, offset
