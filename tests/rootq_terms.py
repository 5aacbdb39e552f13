"""Float64 reference of the RootQ closed-form gradients (SURVEY.md A.5), as device-agnostic torch functions.

The forward values are formed in the inputs' dtype with the reference's own operations (RootQ/function.py:15-32,
58-67, RootQ/base.py:109-111,146-155): fp32 inputs give the fp32 values the kernels and the eager chain compute.
From those values the per-element gradient terms are evaluated in float64, with the arithmetic of
oracle/fq_oracle.c::orc_rootq_act / orc_rootq_wt.  The terms are un-chained: the gradient of in_scale, wt_upper
and wt_lower is m * g * sum(terms), the gradient of wt_alpha is amask * sum(terms) (base.py:95,97,137-140,
function.py:25-26)."""
from collections import namedtuple

import torch
import torch.nn.functional as F

ActTerms = namedtuple("ActTerms", "y keep terms")
WtTerms = namedtuple("WtTerms", "y dw terms amask alpha delta")


def act_terms(x, dy, rs, q):
    """Activation quantizer with effective scale rs (0-dim, after EMA and gradient mix) and Q = hi - lo levels.
    -> y (x's dtype), keep (dx = dy where keep, else 0), terms (float64, the d in_scale terms
    dy * ((I - v) + Q * 1[x1 > up]) before the m * g chain)."""
    up = rs * q
    nl = 0.0 - x
    x1 = x + F.relu(nl)
    ov = x1 - up
    xq = x1 - F.relu(ov)
    v = xq / rs
    i = (v.round() - v) + v                                  # round_pass value, utils.py:29-32
    y = i * rs
    clip = ov > 0
    keep = (nl <= 0) & (ov <= 0)                             # relu's gradient passes NaN: dx(NaN) = 0
    terms = dy.double() * ((i.double() - v.double()) + torch.where(clip, float(q), 0.0).double())
    return ActTerms(y, keep, terms)


def wt_terms(w, dy, U, L, alpha, q):
    """Weight quantizer with mixed running bounds U, L (0-dim), raw alpha (0-dim) and Q = hi - lo.
    -> y (w's dtype), dw (float64), terms [3, n] (float64: d U, d L, d alpha' per element), amask (1.0 where the
    alpha clamp passes the gradient, else 0.0), the clamped alpha and delta (w's dtype)."""
    dt = w.dtype
    lw = L - w
    x1 = w + F.relu(lw)
    ov = x1 - U
    c = x1 - F.relu(ov)                                      # clipping by the relu trick, function.py:15-20
    delta = (U - L) / torch.tensor(q, dtype=dt, device=w.device)   # IEEE quotient (see DESIGN §2)
    r1 = F.relu(1e-4 - alpha)                               # function.py:25-26
    a1 = alpha + r1
    r2 = F.relu(a1 - 1)
    a2 = a1 - r2
    amask = 1.0 if not (bool(r1 > 0) or bool(r2 > 0)) else 0.0
    k = 2 / delta
    t = (c - L) / delta
    i = (t.floor() - t) + t                                  # floor_pass value, utils.py:34-37
    mi = (i + 0.5) * delta + L
    z = c - mi
    sig = (torch.pow(k * z.abs() + 1e-5, a2) * (z / (z.abs() + 1e-5))).sgn()   # function.py:22-32,58
    y = ((sig + 1) / 2 + i) * delta + L
    # float64 from here on
    d, k, hd, a = dy.double(), float(k), float(delta) * 0.5, float(a2)
    s = torch.where(z > 0, 1.0, torch.where(z < 0, -1.0, 0.0)).double()   # d|z|/dz
    m_lo, m_hi = lw > 0, ov > 0
    dcw = (~(m_lo | m_hi)).double()
    cu, cl = m_hi.double(), (m_lo & ~m_hi).double()
    az = z.double().abs()
    den = az + 1e-5
    sg = z.double() / den
    b = k * az + 1e-5
    pw = b.pow(a)
    dpdz = a * pw / b * k * s * sg + pw * 1e-5 / (den * den)
    dpdd = -(a * pw / b * k * az * sg) / float(delta)
    dpda = pw * b.log() * sg
    lvl = (sig.double() + 1.0) * 0.5 + i.double()
    iq, td = 1.0 / q, t.double()
    terms = torch.stack([
        d * (hd * (dpdz * cu + dpdd * iq) + (cu - td * iq) + lvl * iq),
        d * (hd * (dpdz * cl - dpdd * iq) + (cl - 1.0 + td * iq) - lvl * iq + 1.0),
        d * (hd * dpda)])
    dw = d * dcw * (1.0 + hd * dpdz)
    return WtTerms(y, dw, terms.reshape(3, -1), amask, a2, delta)
