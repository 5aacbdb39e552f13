"""The fused BatchNorm (+ residual) (+ ReLU) -> fake-quant kernels (csrc/bnq_kernels.cu) at the sizes ResNet-50 QAT
training launches them, against exact and float64 references.

The entries `dlmcq_bnq_forward` / `dlmcq_bnq_backward` are called through ctypes, so the test owns every buffer.
Before each call every output is poisoned with NaN and sits between two guard bands that must come back untouched,
and the workspace is filled with 0xFF bytes (the header promises it needs no initialisation).

What is compared with what:
  * batch statistics: save_mean / save_invstd / the running buffers against float64 statistics of the same input,
    with a bar from the longest fp32 chain of bnq_stats_kernel (see `stats_bars`), and bit for bit against the
    kernel's fixed summation order and finalisation formula (`stats_fixed_order`);
  * the plain output a: bit for bit, from the kernel's own saved fp32 mean / invstd, as t = x - mean, A = gamma*invstd,
    z = fma(t, A, beta) (R.fma_f32, one rounding), + identity, ReLU, rounded to storage;
  * a_q: bit for bit against the stand-alone kernel `fq_forward(a)`;
  * dz (residual form): bit for bit - mask * (in-range d_q + d_a), rounded to storage;
  * dbeta, dgamma, dscale: against the float64 sum of the kernel's own fp32 terms, bar 1e-5 |exact| + L 2^-24 sum|t|
    with L the longest fp32 chain of the reduce kernel's geometry, and dbeta / dgamma also bit for bit against the
    reduce kernel's fixed summation order (per thread over its tiles, over the thread rows, then the per-CTA partials
    in double in warp-strided order; `fixed_order_sums`);
  * dx: per element, gamma*invstd * ((dz - mean(dz)) - xhat * mean(dz*xhat)) in float64, with a bar of five fp32
    roundings of |A| (|dz| + |c1| + |xhat c2|) plus the propagated reduction bars of c1, c2.
Inputs whose sums are exact in any order (test_exact_sums) make dbeta, dgamma, dscale and the statistics exact."""
import ctypes as C
import math
import time

import numpy as np
import pytest
import torch

from oracle import restate as R
from tests.golden_io import bits_equal, first_mismatch

pytestmark = pytest.mark.gpu

THREADS = 256
FOLD_WARPS = 16            # bnq_fold_partials: warp w adds partials w, w + 16, ... in double, then warp 0 adds the warps
SAFE = 2.0 ** 20           # kBnqSafe: the packed fast path's bound on |x|, |identity| and the channel constants
ULP = 2.0 ** -24
GUARD = 64                 # guard elements on each side of every output
SENTINEL = 0x5A
LO, HI = 0, 15

WORST = {}                 # bar -> worst measured error / tolerance over the module


def _lib():
    from dlmc_quant_b200 import _lib as L
    return L


def F():
    from dlmc_quant_b200 import functional
    return functional


@pytest.fixture(scope="module", autouse=True)
def _module_report():
    torch.cuda.reset_peak_memory_stats()
    t0 = time.time()
    yield
    print(f"\n[bnq training] wall {time.time() - t0:.1f} s, peak allocated "
          f"{torch.cuda.max_memory_allocated() / 2 ** 30:.2f} GiB")
    for k in sorted(WORST):
        print(f"[bnq training] worst error / tolerance  {k:8s} {WORST[k]:.3e}")


def same(a, b, what):
    assert bits_equal(a, b), f"{what}: {first_mismatch(a, b)}"


def within(err, tol, what):
    """err <= tol elementwise (float64 tensors; a zero error passes a zero bar); records the worst ratio."""
    ratio = torch.where(err == 0, torch.zeros_like(err), torch.nan_to_num(err / tol, nan=math.inf, posinf=math.inf))
    worst = float(ratio.max())
    WORST[what] = max(WORST.get(what, 0.0), worst)
    if worst > 1.0:
        i = int(ratio.flatten().argmax())
        raise AssertionError(f"{what}: error/tolerance {worst:.3g} at {i} (err {float(err.flatten()[i])!r}, "
                             f"tol {float(tol.flatten()[i])!r})")


# ---------------------------------------------------------------------------------------------------------------
# geometry: make_bnq_geom / apply_grid restated
# ---------------------------------------------------------------------------------------------------------------
class Geom:
    def __init__(self, rows, ch, dtype):
        self.rows, self.C = rows, ch
        self.vn = 4 if dtype is torch.float32 else 8
        self.nsm = torch.cuda.get_device_properties(0).multi_processor_count
        self.cv = ch // self.vn
        self.txw = max(min(self.cv, THREADS), 1)
        self.ty = max(THREADS // self.txw, 1)
        self.gy = -(-self.cv // self.txw)
        passes = self.tiles(4)
        self.nbx = max(min(passes, max(self.nsm * 4 // self.gy, 1), max(rows // 16, 1)), 1)

    def tiles(self, u):
        """row tiles of ty * u rows, the ragged one included"""
        return -(-self.rows // (self.ty * u))

    def apply_grid(self, u=4, per_cta=8):
        passes = self.tiles(u)
        return max(min(max(passes // per_cta, self.nsm * 8 // self.gy), passes), 1)

    def chain_stats(self):
        """longest fp32 chain of a statistics sum: the thread's tiles x 4 rows, the fold over ty thread rows, and the
        rounding of d = x - k"""
        return -(-self.tiles(4) // self.nbx) * 4 + self.ty + 1

    def chain_reduce(self, u):
        """longest fp32 chain of dbeta / dgamma (the products dz * xhat are exact inside the fma), + 1 for the double
        fold of the partials"""
        return -(-self.tiles(u) // self.nbx) * u + self.ty + 1

    def chain_scale(self, u):
        """longest fp32 chain of the scale gradient: per thread two chains over u * VN / 2 elements a tile (one more
        add a vector on the generic path), the two chains and the generic sum added, then block_sum's two 5-level
        warp trees"""
        return -(-self.tiles(u) // self.nbx) * u * (self.vn // 2 + 1) + 2 + 10


def fixed_order_sums(geo, u, add_t, fa, fb):
    """float64 [C]: sum(add_t) and sum(fa * fb) per channel in the fused kernels' fixed order.  Thread row r of CTA b
    adds, in fp32, the rows r + j * ty (j < u) of its tiles b, b + nbx, ... (sum: +=, product sum: fma), then the ragged
    tile if b = nfull % nbx owns it; the CTA folds its ty thread rows in fp32 in order; bnq_fold_partials adds the nbx
    partials in double, warp w taking w, w + 16, ... and warp 0 adding the 16 warp sums in order.
    This restates an implementation choice, not a requirement: dbeta / dgamma are held to it bit for bit because only
    an order-exact check sees a tile that moved to another CTA (which merely reorders the sum).  A deliberate change to
    the reduce kernel's summation order, tile ownership or partial folding must update this restatement; such a change
    still has to pass the derived bars in check_backward, which do not depend on the order."""
    rows, ch, ty, nbx = geo.rows, geo.C, geo.ty, geo.nbx
    tr = ty * u
    nfull = rows // tr
    s1 = torch.zeros(nbx, ty, ch, dtype=torch.float32, device=add_t.device)
    s2 = torch.zeros_like(s1)
    va = add_t[:nfull * tr].view(nfull, u, ty, ch)
    pa = fa[:nfull * tr].view(nfull, u, ty, ch)
    pb = fb[:nfull * tr].view(nfull, u, ty, ch)
    for i0 in range(0, nfull, nbx):
        m = min(nbx, nfull - i0)
        for j in range(u):
            s1[:m] += va[i0:i0 + m, j]
            s2[:m] = R.fma_f32(pa[i0:i0 + m, j], pb[i0:i0 + m, j], s2[:m])
    if nfull * tr < rows:
        own = nfull % nbx
        for j in range(u):
            r0 = nfull * tr + j * ty
            n = min(ty, rows - r0)
            if n <= 0:
                break
            s1[own, :n] += add_t[r0:r0 + n]
            s2[own, :n] = R.fma_f32(fa[r0:r0 + n], fb[r0:r0 + n], s2[own, :n])
    p1 = torch.zeros(nbx, ch, dtype=torch.float32, device=add_t.device)
    p2 = torch.zeros_like(p1)
    for r in range(ty):
        p1 += s1[:, r]
        p2 += s2[:, r]
    w1 = torch.zeros(FOLD_WARPS, ch, dtype=torch.float64, device=add_t.device)
    w2 = torch.zeros_like(w1)
    for b0 in range(0, nbx, FOLD_WARPS):
        m = min(FOLD_WARPS, nbx - b0)
        w1[:m] += p1[b0:b0 + m].double()
        w2[:m] += p2[b0:b0 + m].double()
    t1 = torch.zeros(ch, dtype=torch.float64, device=add_t.device)
    t2 = torch.zeros_like(t1)
    for w in range(FOLD_WARPS):
        t1 += w1[w]
        t2 += w2[w]
    return t1, t2


# ---------------------------------------------------------------------------------------------------------------
# buffers and calls
# ---------------------------------------------------------------------------------------------------------------
class Guarded:
    """`t` is a [*shape] view into a buffer with GUARD elements of SENTINEL bytes on each side."""

    def __init__(self, shape, dtype):
        n = int(np.prod(shape))
        self.base = torch.empty(n + 2 * GUARD, dtype=dtype, device="cuda")
        self.base.view(torch.uint8).fill_(SENTINEL)
        self.n = n
        self.t = self.base[GUARD:GUARD + n].view(*shape)

    def poison(self):
        self.t.fill_(float("nan"))

    def check(self, what):
        b = self.base.view(torch.uint8)
        es = self.base.element_size()
        assert bool((b[:GUARD * es] == SENTINEL).all()) and bool((b[(GUARD + self.n) * es:] == SENTINEL).all()), \
            f"{what}: write outside the output"


def qparams(scale, offset, g):
    L = _lib()
    return L.QParams(L.FORM_AFFINE, LO, HI, float(g), scale.data_ptr(), offset.data_ptr())


class Case:
    """One BatchNorm site: inputs, guarded outputs and the two C-ABI calls."""

    def __init__(self, x, gamma, beta, rm0, rv0, *, identity=None, relu=True, quant=None, training=True, eps=1e-5,
                 momentum=0.1, d_a=None, d_q=None):
        L = _lib()
        self.x, self.idn, self.gamma, self.beta = x, identity, gamma, beta
        self.rows, self.C = x.shape
        self.dtype = x.dtype
        self.relu, self.training, self.eps, self.momentum = relu, training, eps, momentum
        self.quant = quant                                   # (scale, offset, g) or None
        self.rm0, self.rv0 = rm0, rv0
        self.d_a, self.d_q = d_a, d_q
        self.geo = Geom(self.rows, self.C, self.dtype)
        flags = (L.BNQ_TRAINING if training else 0) | (L.BNQ_RELU if relu else 0) | \
            (L.BNQ_RESIDUAL if identity is not None else 0)
        self.desc = L.BnqDesc(self.rows, self.C, F()._dtype_code(x), flags, float(eps), float(momentum))
        self.ws_bytes = L.lib().dlmcq_bnq_workspace_bytes(C.byref(self.desc))
        assert self.ws_bytes > 0
        self.ws = Guarded((self.ws_bytes,), torch.uint8)
        shp, ch = (self.rows, self.C), (self.C,)
        self.rm, self.rv = Guarded(ch, torch.float32), Guarded(ch, torch.float32)
        self.mean, self.invstd = Guarded(ch, torch.float32), Guarded(ch, torch.float32)
        self.a, self.aq = Guarded(shp, self.dtype), Guarded(shp, self.dtype)
        self.dx, self.dz = Guarded(shp, self.dtype), Guarded(shp, self.dtype)
        self.dgamma, self.dbeta = Guarded(ch, torch.float32), Guarded(ch, torch.float32)
        self.dscale = Guarded((1,), torch.float32)
        self.qp = qparams(*quant) if quant is not None else None
        self.outs = [self.mean, self.invstd, self.a, self.aq, self.dx, self.dz, self.dgamma, self.dbeta, self.dscale]

    def reset(self):
        """NaN in every output, 0xFF in the workspace, the running buffers back to their initial values"""
        for o in self.outs:
            o.poison()
        self.ws.t.fill_(0xFF)
        self.rm.t.copy_(self.rm0)
        self.rv.t.copy_(self.rv0)

    def check_guards(self):
        for name in ("ws", "rm", "rv", "mean", "invstd", "a", "aq", "dx", "dz", "dgamma", "dbeta", "dscale"):
            getattr(self, name).check(name)

    def launch_forward(self, want_a=True, want_q=True):
        p = F()._ptr
        q = want_q and self.quant is not None
        _lib().check(_lib().lib().dlmcq_bnq_forward(
            p(self.x), p(self.idn), p(self.gamma), p(self.beta), p(self.rm.t), p(self.rv.t), p(self.mean.t),
            p(self.invstd.t), p(self.a.t) if want_a else p(None), p(self.aq.t) if q else p(None), C.byref(self.desc),
            C.byref(self.qp) if q else None, p(self.ws.t), self.ws_bytes, F()._stream_ptr()))

    def launch_backward(self, use_da, use_dq, want_dx=True):
        p = F()._ptr
        resid = self.idn is not None
        q = use_dq and self.quant is not None
        _lib().check(_lib().lib().dlmcq_bnq_backward(
            p(self.x), p(self.a.t) if resid else p(None), p(self.d_a) if use_da else p(None),
            p(self.d_q) if q else p(None), p(self.gamma), p(self.beta), p(self.mean.t), p(self.invstd.t),
            p(self.dx.t) if want_dx else p(None), p(self.dz.t) if resid else p(None), p(self.dgamma.t),
            p(self.dbeta.t), p(self.dscale.t) if q else p(None), C.byref(self.desc), C.byref(self.qp) if q else None,
            p(self.ws.t), self.ws_bytes, F()._stream_ptr()))

    def forward(self, want_a=True, want_q=True):
        self.reset()
        self.launch_forward(want_a, want_q)
        torch.cuda.synchronize()
        self.check_guards()

    def backward(self, use_da, use_dq, want_dx=True):
        """needs the forward's mean / invstd (and a, for the residual form) in place"""
        for o in (self.dx, self.dz, self.dgamma, self.dbeta, self.dscale):
            o.poison()
        self.ws.t.fill_(0xFF)
        self.launch_backward(use_da, use_dq, want_dx)
        torch.cuda.synchronize()
        self.check_guards()


# ---------------------------------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------------------------------
def stats_bars(c):
    """Training statistics against float64 statistics of the same input.  With k = x[0] (the kernel's shift),
    S1 = sum(x - k), S2 = sum((x - k)^2) carry at most L 2^-24 sum|x - k| and (L + 1) 2^-24 sum (x - k)^2 (the fp32
    rounding of x - k, doubled by the square), L = chain_stats().  Then
        |mean - mean64|     <= dS1 / n + 2^-24 |mean64|                          (last: the fp32 store)
        dvar                 = dS2 / n + (2 |m1| + dS1 / n) dS1 / n,  m1 = mean64 - k
        |invstd - invstd64| <= dvar / 2 (var64 + eps - dvar)^(-3/2) + 2^-24 invstd64
        running_mean, running_var: momentum * (dS1 / n, dvar * n / (n - 1)) + 2^-24 |value|."""
    geo, n = c.geo, c.rows
    x = c.x.double()
    k = x[0]
    d = x - k
    a1, a2 = d.abs().sum(0), (d * d).sum(0)
    del d
    mean = x.mean(0)
    var = ((x - mean) ** 2).mean(0)
    del x
    L = geo.chain_stats()
    ds1, ds2 = L * ULP * a1, (L + 1) * ULP * a2
    eps = float(np.float32(c.eps))
    dvar = ds2 / n + (2 * (mean - k).abs() + ds1 / n) * ds1 / n
    inv = 1 / torch.sqrt(var + eps)
    tiny = 1e-12 * (mean.abs() + a1 / n)                         # float64 evaluation of the reference itself
    within((c.mean.t.double() - mean).abs(), ds1 / n + ULP * mean.abs() + tiny, "mean")
    den = (var + eps - dvar).clamp(min=1e-300)
    within((c.invstd.t.double() - inv).abs(), 0.5 * dvar * den ** -1.5 + ULP * inv + 1e-12 * inv, "invstd")
    mo = float(np.float32(c.momentum))
    rm = (1 - mo) * c.rm0.double() + mo * mean
    rv = (1 - mo) * c.rv0.double() + mo * var * (n / (n - 1))
    within((c.rm.t.double() - rm).abs(), mo * ds1 / n + ULP * rm.abs() + tiny, "running")
    within((c.rv.t.double() - rv).abs(), mo * dvar * n / (n - 1) + ULP * rv.abs() + 1e-12 * rv, "running")


def stats_fixed_order(c):
    """save_mean / save_invstd / running buffers bit for bit: the sums in the kernel's order (fixed_order_sums), then
    bnq_stats_finalize_kernel's float64 formula in its order, rounded once.  The divisions take n as a tensor: torch
    divides by a host scalar as a multiplication by its reciprocal, which is not the correctly rounded quotient."""
    xf = c.x.float()
    k = xf[0]
    d = xf - k
    t1, t2 = fixed_order_sums(c.geo, 4, d, d, d)
    del d
    n = float(c.rows)
    nt = torch.full_like(t1, n)
    m1 = t1 / nt
    mean = k.double() + m1
    var = (t2 / nt - m1 * m1).clamp(min=0.0)
    same(c.mean.t, mean.float(), "save_mean (fixed order)")
    same(c.invstd.t, (1.0 / torch.sqrt(var + float(np.float32(c.eps)))).float(), "save_invstd (fixed order)")
    mo = float(np.float32(c.momentum))
    same(c.rm.t, ((1.0 - mo) * c.rm0.double() + mo * mean).float(), "running_mean (fixed order)")
    unb = var * (n / (n - 1.0)) if n > 1 else var
    same(c.rv.t, ((1.0 - mo) * c.rv0.double() + mo * unb).float(), "running_var (fixed order)")


def eval_stats(c):
    same(c.mean.t, c.rm0, "eval save_mean")
    v = c.rv0 + float(np.float32(c.eps))                         # fp32 add; sqrt and 1/ each rounded once
    same(c.invstd.t, (1.0 / torch.sqrt(v.double()).float().double()).float(), "eval save_invstd")
    same(c.rm.t, c.rm0, "eval running_mean untouched")
    same(c.rv.t, c.rv0, "eval running_var untouched")


def ref_act(c):
    """the plain output bit for bit from the kernel's saved statistics, rounded to storage"""
    mean, inv = c.mean.t, c.invstd.t
    A = c.gamma * inv
    out = torch.empty(c.rows, c.C, dtype=c.dtype, device="cuda")
    step = max(1, (1 << 24) // c.C)
    for r0 in range(0, c.rows, step):
        xs = c.x[r0:r0 + step].float()
        z = R.fma_f32(xs - mean, A, c.beta)
        if c.idn is not None:
            z = z + c.idn[r0:r0 + step].float()
        if c.relu:
            z = torch.where(z > 0, z, torch.where(torch.isnan(z), z, torch.zeros_like(z)))
        out[r0:r0 + step] = z.to(c.dtype)
    return out


def check_forward(c, a_ref):
    same(c.a.t, a_ref, "a")
    if c.quant is not None:
        s, o, g = c.quant
        same(c.aq.t, F().fq_forward(a_ref, s, o, LO, HI, F().FORM_AFFINE, g=g), "a_q vs fq_forward(a)")


def quant_terms(c, act):
    """fp32 in-range mask and the float64 scale-gradient terms d_q * (inside ? code - u : code), u = (act - off) / s'"""
    s, o, g = c.quant
    g32 = float(np.float32(g))
    sg = s * g32
    sp = (s - sg) + sg
    u = (act - o) / sp
    inside = (u >= LO) & (u <= HI)
    code = u.clamp(LO, HI).round()
    term = c.d_q.double() * torch.where(inside, code.double() - u.double(), code.double())
    return inside, term, g32


def check_backward(c, a_ref, use_da, use_dq, want_dx, what):
    resid = c.idn is not None
    q = use_dq and c.quant is not None
    geo, n = c.geo, c.rows
    u = 2 if resid else 4                                           # rows in flight of the reduce kernel
    act = (c.a.t if resid else a_ref).float()
    dz = torch.zeros(c.rows, c.C, dtype=torch.float32, device="cuda")
    if q:
        inside, sterm, g32 = quant_terms(c, act)
        dz = torch.where(inside, c.d_q.float(), dz)
        del inside
    if use_da:
        dz = dz + c.d_a.float()
    if c.relu:
        dz = torch.where(act > 0, dz, torch.zeros_like(dz))
    del act
    if resid:
        dz = dz.to(c.dtype).float()
        same(c.dz.t, dz.to(c.dtype), f"{what}: dz")
    xh = (c.x.float() - c.mean.t) * c.invstd.t                      # the kernel's fp32 xhat
    # reductions against the float64 sums of the kernel's terms
    prod = dz.double() * xh.double()
    db, dg = dz.double().sum(0), prod.sum(0)
    adb, adg = dz.double().abs().sum(0), prod.abs().sum(0)
    del prod
    Lr = geo.chain_reduce(u)
    bar_db = 1e-5 * db.abs() + Lr * ULP * adb
    bar_dg = 1e-5 * dg.abs() + Lr * ULP * adg
    within((c.dbeta.t.double() - db).abs(), bar_db, "dbeta")
    within((c.dgamma.t.double() - dg).abs(), bar_dg, "dgamma")
    fb, fg = fixed_order_sums(geo, u, dz, dz, xh)
    same(c.dbeta.t, fb.float(), f"{what}: dbeta (fixed order)")
    same(c.dgamma.t, fg.float(), f"{what}: dgamma (fixed order)")
    del xh
    if q:
        ss, sa = sterm.sum(), sterm.abs().sum()
        del sterm
        Ls = geo.chain_scale(u)
        within((c.dscale.t.double() - g32 * ss).abs().reshape(1),
               (g32 * (1e-5 * ss.abs() + Ls * ULP * sa)).reshape(1), "dscale")
    if want_dx:
        A = (c.gamma * c.invstd.t).double()
        c1 = db / n if c.training else torch.zeros_like(db)
        c2 = dg / n if c.training else torch.zeros_like(dg)
        dc1 = (bar_db / n + ULP * c1.abs()) if c.training else torch.zeros_like(db)
        dc2 = (bar_dg / n + ULP * c2.abs()) if c.training else torch.zeros_like(dg)
        step = max(1, (1 << 23) // c.C)
        for r0 in range(0, c.rows, step):
            xhat = (c.x[r0:r0 + step].double() - c.mean.t.double()) * c.invstd.t.double()
            d = dz[r0:r0 + step].double()
            ref = A * ((d - c1) - xhat * c2)
            tol = 5 * ULP * A.abs() * (d.abs() + c1.abs() + (xhat * c2).abs()) + A.abs() * (dc1 + xhat.abs() * dc2)
            if c.dtype is torch.bfloat16:
                tol = tol + 2.0 ** -8 * (ref.abs() + tol)         # the bf16 store: unit roundoff of an 8-bit significand
            tol = tol + 1e-300
            within((c.dx.t[r0:r0 + step].double() - ref).abs(), tol, "dx")
    else:
        assert bool(torch.isnan(c.dx.t.float()).all()), f"{what}: dx written although dx == NULL"


# ---------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------
KINDS = {
    # kind: (residual, relu, quantizer, backward variants (name, d_a, d_q, dx))
    "stem": (False, True, False, [("plain", True, False, True), ("nodx", True, False, False)]),
    "plain": (False, False, False, [("plain", True, False, True)]),
    "into": (False, True, True, [("masked", False, True, True), ("quant_da", True, True, True),
                                 ("nodx", False, True, False)]),
    "resid": (True, True, True, [("resid_q", True, True, True), ("resid_noq", True, False, True),
                                 ("nodx", True, True, False)]),
}


def random_case(rows, ch, dtype, kind, training=True, seed=0, eps=1e-5, scale=0.21, offset=None):
    resid, relu, quant, _ = KINDS[kind]
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = (torch.randn(rows, ch, generator=g, device="cuda") * 1.7 + 0.4).to(dtype)
    idn = torch.relu(torch.randn(rows, ch, generator=g, device="cuda")).to(dtype) if resid else None
    gamma = torch.rand(ch, generator=g, device="cuda") + 0.5
    beta = torch.randn(ch, generator=g, device="cuda") * 0.3
    rm0 = torch.randn(ch, generator=g, device="cuda") * 0.1
    rv0 = torch.rand(ch, generator=g, device="cuda") + 0.5
    d_a = torch.randn(rows, ch, generator=g, device="cuda").to(dtype)
    d_q = torch.randn(rows, ch, generator=g, device="cuda").to(dtype) if quant else None
    q = None
    if quant:
        off = 0.0 if offset is None else offset
        q = (torch.tensor([scale], device="cuda"), torch.tensor([off], device="cuda"),
             float(np.float32(R.lsq_g(rows * ch, HI))))
    return Case(x, gamma, beta, rm0, rv0, identity=idn, relu=relu, quant=q, training=training, eps=eps, d_a=d_a,
                d_q=d_q)


def run_and_check(c, kind):
    """forward (+ the q-only forward), statistics, then every backward variant of the kind"""
    c.forward()
    if c.training:
        stats_bars(c)
        stats_fixed_order(c)
    else:
        eval_stats(c)
    a_ref = ref_act(c)
    check_forward(c, a_ref)
    if c.quant is not None and c.idn is None:                      # bn_act_into: a_q alone, a_out == NULL
        aq = c.aq.t.clone()
        c.forward(want_a=False)
        same(c.aq.t, aq, "a_q without a_out")
        assert bool(torch.isnan(c.a.t.float()).all()), "a written although a_out == NULL"
        c.forward()
    for name, use_da, use_dq, want_dx in KINDS[kind][3]:
        c.backward(use_da, use_dq, want_dx)
        check_backward(c, a_ref, use_da, use_dq, want_dx, name)
    return a_ref


# ---------------------------------------------------------------------------------------------------------------
# 1. the geometries ResNet-50 QAT launches at per-GPU batch 128 (and one at 32), 224 x 224
# ---------------------------------------------------------------------------------------------------------------
f32, bf16 = torch.float32, torch.bfloat16
SITES = [
    ("stem_bn1", 1605632, 64, f32, "stem"),                 # 25 088 tiles, apply grid 3136, stats nbx 592
    ("l1_bn1_f32", 401408, 64, f32, "into"),
    ("l1_bn1_bf16", 401408, 64, bf16, "into"),
    ("l1_bn3_f32", 401408, 256, f32, "resid"),
    ("l1_bn3_bf16", 401408, 256, bf16, "resid"),
    ("l4_bn3_f32", 6272, 2048, f32, "resid"),               # gy = 2, ty = 1, CTAs with unequal tile counts
    ("ragged_64_f32", 401408 + 37, 64, f32, "into"),
    ("ragged_64_bf16", 401408 + 37, 64, bf16, "into"),
    ("ragged_512_f32", 100352 + 3, 512, f32, "resid"),
    ("ragged_512_bf16", 100352 + 3, 512, bf16, "resid"),
    ("idle_1028_f32", 50001, 1028, f32, "resid"),           # cv = 257: one active column in the second y-block
    ("idle_12_f32", 1000003, 12, f32, "plain"),             # txw = 3, ty = 85: one idle thread
    ("idle_8_bf16", 1000005, 8, bf16, "into"),              # txw = 1, ty = 256
    ("b32_l1_bn1_bf16", 100352, 64, bf16, "into"),          # per-GPU batch 32
]
EVAL = ["l1_bn1_f32", "ragged_512_bf16", "l4_bn3_f32", "idle_8_bf16"]


@pytest.mark.parametrize("site", SITES, ids=[s[0] for s in SITES])
def test_training_geometry(site):
    name, rows, ch, dtype, kind = site
    c = random_case(rows, ch, dtype, kind, training=True, seed=SITES.index(site))
    geo = c.geo
    if name == "stem_bn1":
        assert (geo.tiles(4), geo.apply_grid(), geo.nbx) == (25088, 3136, 592)
    run_and_check(c, kind)


@pytest.mark.parametrize("name", EVAL)
def test_eval_geometry(name):
    _, rows, ch, dtype, kind = next(s for s in SITES if s[0] == name)
    c = random_case(rows, ch, dtype, kind, training=False, seed=11)
    run_and_check(c, kind)


# ---------------------------------------------------------------------------------------------------------------
# 3. inputs that make every sum exact in any order
# ---------------------------------------------------------------------------------------------------------------
EXACT = [
    ("stem", 1605632, 64, f32, "stem"),
    ("into_f32", 401408, 64, f32, "into"),
    ("into_bf16_ragged", 401408 + 38, 64, bf16, "into"),
    ("resid_f32_ragged", 100352 + 2, 512, f32, "resid"),
]


@pytest.mark.parametrize("site", EXACT, ids=[s[0] for s in EXACT])
def test_exact_sums(site):
    """Per channel x is 0.5 +- 1 in equal numbers, shuffled over the rows, and eps = 0: mean = 0.5, invstd = 1 and
    xhat = +-1 exactly.  gamma in {1.5, 9, -1.5, 0.75}, beta = 0.25 and an identity in {0, 0.25, 0.5} keep a on a
    quarter grid; scale 0.5 with g = 2^-12 gives s' == s, so u = 2a and every scale-gradient term is a multiple of
    d_q / 2; d_q, d_a are small integers.  Every partial sum is then an fp32-exact dyadic number, whatever the order,
    and dbeta, dgamma, dscale / g, save_mean, save_invstd must equal their exact values."""
    _, rows, ch, dtype, kind = site
    resid, relu, quant, _ = KINDS[kind]
    g = torch.Generator(device="cuda").manual_seed(5)
    up = torch.rand(rows, ch, generator=g, device="cuda").argsort(0) < rows // 2
    x = torch.where(up, 1.5, -0.5).to(dtype)
    del up
    gamma = torch.tensor([1.5, 9.0, -1.5, 0.75], device="cuda").repeat(ch // 4)
    beta = torch.full((ch,), 0.25, device="cuda")
    idn = (torch.randint(0, 3, (rows, ch), generator=g, device="cuda") * 0.25).to(dtype) if resid else None
    d_a = torch.randint(-2, 3, (rows, ch), generator=g, device="cuda").to(dtype)
    d_q = torch.randint(-3, 4, (rows, ch), generator=g, device="cuda").to(dtype) if quant else None
    rm0 = torch.randn(ch, generator=g, device="cuda") * 0.1
    rv0 = torch.rand(ch, generator=g, device="cuda") + 0.5
    q = None
    if quant:
        s32, g32 = np.float32(0.5), np.float32(2.0 ** -12)
        sg = np.float32(s32 * g32)
        assert np.float32(np.float32(s32 - sg) + sg) == s32            # s' == s
        q = (torch.tensor([0.5], device="cuda"), torch.zeros(1, device="cuda"), float(g32))
    c = Case(x, gamma, beta, rm0, rv0, identity=idn, relu=relu, quant=q, training=True, eps=0.0, d_a=d_a, d_q=d_q)
    a_ref = run_and_check(c, kind)
    # statistics: exact
    assert bool((c.mean.t == 0.5).all()) and bool((c.invstd.t == 1.0).all()), "exact statistics"
    n, mo = float(rows), float(np.float32(c.momentum))
    rm = ((1.0 - mo) * rm0.double() + mo * 0.5).float()
    rv = ((1.0 - mo) * rv0.double() + mo * (1.0 * (n / (n - 1.0)))).float()
    same(c.rm.t, rm, "running_mean (exact)")
    same(c.rv.t, rv, "running_var (exact)")
    # every backward variant once more, against the exact sums
    xh = torch.where(x.float() > 0.5, 1.0, -1.0).double()
    for name, use_da, use_dq, want_dx in KINDS[kind][3]:
        c.backward(use_da, use_dq, want_dx)
        act = (c.a.t if resid else a_ref).float()
        dz = torch.zeros(rows, ch, dtype=torch.float64, device="cuda")
        qq = use_dq and quant
        if qq:
            inside, sterm, g32 = quant_terms(c, act)
            dz = torch.where(inside, c.d_q.double(), dz)
        if use_da:
            dz = dz + c.d_a.double()
        if relu:
            dz = torch.where(act > 0, dz, torch.zeros_like(dz))
        assert float(dz.abs().sum(0).max()) < 2 ** 24
        db, dg = dz.sum(0), (dz * xh).sum(0)
        assert bool((c.dbeta.t.double() == db).all()), f"{name}: dbeta is not exact"
        assert bool((c.dgamma.t.double() == dg).all()), f"{name}: dgamma is not exact"
        if qq:
            ss = sterm.sum()
            assert abs(float(ss)) < 2 ** 22 and bool((sterm * 2 == (sterm * 2).round()).all())
            assert float(c.dscale.t[0]) == g32 * float(ss), f"{name}: dscale {float(c.dscale.t[0])} != {g32 * float(ss)}"


# ---------------------------------------------------------------------------------------------------------------
# 4. the packed fast path against the guarded generic path
# ---------------------------------------------------------------------------------------------------------------
def outlier_positions(geo, u, count_cols=3):
    """(rows, cols) of single elements in tiles 0, 1, 7, nfull / 2, nfull - 1 and the ragged tile (u-row tiles)"""
    tr = geo.ty * u
    nfull = geo.rows // tr
    tiles = sorted({0, 1, 7, nfull // 2, nfull - 1})
    rows = [t * tr + (t * 5) % tr for t in tiles if t < nfull]
    if nfull * tr < geo.rows:
        rows.append(geo.rows - 1)
    rows = [r for r in rows if r != 0]                             # row 0 is the statistics shift
    cols = [(r * 7) % geo.C for r in rows]
    return torch.tensor(rows, device="cuda"), torch.tensor(cols, device="cuda")


@pytest.mark.parametrize("site", [("ragged_512_f32", 100352 + 3, 512, f32, "resid"),
                                  ("ragged_64_bf16", 401408 + 37, 64, bf16, "into")], ids=lambda s: s[0])
def test_outliers_training(site):
    """|x| = 2^21 (and a 2^21 identity) in scattered tiles, the ragged one included: those threads' tiles take the
    generic path; every element must still match the bit-exact reference and the reductions their bars."""
    name, rows, ch, dtype, kind = site
    c = random_case(rows, ch, dtype, kind, seed=3)
    r, col = outlier_positions(c.geo, 4)
    c.x[r, col] = torch.where(r % 2 == 0, 2.0 ** 21, -(2.0 ** 21)).to(dtype)
    if c.idn is not None:
        r2, col2 = outlier_positions(c.geo, 2)
        c.idn[r2, (col2 + 1) % ch] = 2.0 ** 21
    run_and_check(c, kind)


@pytest.mark.parametrize("dtype", [f32, bf16])
def test_special_values_eval(dtype):
    """Eval mode with +-inf, NaN and 2^21 in scattered tiles (the ragged one included): the reference holds on every
    element, and every other element is bit-identical to the run without them."""
    rows, ch = 401408 + 37, 64
    clean = random_case(rows, ch, dtype, "into", training=False, seed=9)
    clean.forward()
    a0, q0 = clean.a.t.clone(), clean.aq.t.clone()
    c = clean
    r, col = outlier_positions(c.geo, 4)
    vals = torch.tensor([float("inf"), -float("inf"), float("nan"), 2.0 ** 21, -(2.0 ** 21), float("nan")],
                        device="cuda")
    c.x[r, col] = vals[torch.arange(r.numel(), device="cuda") % vals.numel()].to(dtype)
    c.forward()
    eval_stats(c)
    a_ref = ref_act(c)
    check_forward(c, a_ref)
    keep = torch.ones(rows, ch, dtype=torch.bool, device="cuda")
    keep[r, col] = False
    same(c.a.t[keep], a0[keep], "a away from the special values")
    same(c.aq.t[keep], q0[keep], "a_q away from the special values")
    assert bool(torch.isnan(c.a.t[r, col].float()).any()) and bool(torch.isinf(c.a.t[r, col].float()).any())


def test_generic_channel_constants():
    """A constant channel with eps = 1e-14 has gamma * invstd = 1e7 > 2^20: every thread holding it runs the generic
    path on all its tiles, in the forward, the reduction and the dx pass."""
    for dtype in (f32, bf16):
        c = random_case(401408 + 37, 64, dtype, "into", seed=4, eps=1e-14)
        c.x[:, 5] = 0.75
        c.forward()
        A = c.gamma * c.invstd.t
        assert float(A[5]) > SAFE and float(A.abs().max()) == float(A[5])
        run_and_check(c, "into")


@pytest.mark.parametrize("scale,offset", [(2.0 ** -41, 0.0), (0.21, -(2.0 ** 21 + 0.5))], ids=["tiny_scale", "offset"])
def test_generic_quantizer(scale, offset):
    """A scale below 2^-40 (the quantizer's reciprocal path is off) or |offset| > 2^20 (the packed path is off) sends
    every thread to the generic path: a_q must still equal fq_forward(a), and the backward its references."""
    for kind, site in (("into", (401408 + 37, 64, bf16)), ("resid", (100352 + 3, 512, f32))):
        rows, ch, dtype = site
        c = random_case(rows, ch, dtype, kind, seed=6, scale=scale, offset=offset)
        run_and_check(c, kind)


# ---------------------------------------------------------------------------------------------------------------
# 5. repeatability and graph capture, at layer1's residual site
# ---------------------------------------------------------------------------------------------------------------
def _outputs(c):
    return [o.t.clone() for o in (c.mean, c.invstd, c.rm, c.rv, c.a, c.aq, c.dx, c.dz, c.dgamma, c.dbeta, c.dscale)]


def _eager(c):
    c.reset()
    c.launch_forward()
    c.launch_backward(True, True, True)
    torch.cuda.synchronize()
    c.check_guards()
    return _outputs(c)


def test_repeatable_and_graph_replay():
    c = random_case(401408, 256, f32, "resid", seed=21)
    e1, e2 = _eager(c), _eager(c)
    for i, (u, v) in enumerate(zip(e1, e2)):
        same(u, v, f"eager run-to-run output {i}")
    del e2
    c.reset()
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            c.launch_forward()
            c.launch_backward(True, True, True)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.Generator(device="cuda").manual_seed(22)
    for rep in range(2):
        c.x.copy_((torch.randn(c.rows, c.C, generator=g, device="cuda") * (1.3 + rep) - 0.2))
        c.idn.copy_(torch.relu(torch.randn(c.rows, c.C, generator=g, device="cuda")))
        c.d_a.copy_(torch.randn(c.rows, c.C, generator=g, device="cuda"))
        c.d_q.copy_(torch.randn(c.rows, c.C, generator=g, device="cuda"))
        c.reset()
        graph.replay()
        torch.cuda.synchronize()
        c.check_guards()
        got = _outputs(c)
        want = _eager(c)
        for i, (u, v) in enumerate(zip(got, want)):
            same(u, v, f"replay {rep} output {i}")
        assert not bits_equal(got[0], e1[0]), "the replay read the new inputs"
