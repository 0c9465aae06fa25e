"""The fused BatchNorm training kernels (pygho_b200/csrc/fused_mlp.cu, ticket.cuh) against a float64
reference, at every work split they use.

u = 2^-24.  A launch splits the rows into CTAs of ``ty`` row lanes; each thread adds at most
``k = rows_per_block / ty`` rows (``bn_geom`` below).  n is the number of valid rows.  Every
reference is float64 and is built from the inputs; a later pass is judged from the kernel's own
outputs of the earlier passes (mean, rstd, sums), so each kernel is judged on its own.  Bounds are
per channel or per element, never scaled by a global maximum:

* bn_stats.  d = y - y[0] over the valid rows (the kernel shifts by row 0 of the tensor).  A thread
  sums <= k rounded terms in fp32, the CTA adds ty lanes in fp32, and a group sum is rounded to fp32
  once, so
      |S - sum d|   <= Sb = 1.01 (k + ty + 2) u sum |d|
      |Q - sum d^2| <= Qb = 1.01 (k + ty + 3) u sum d^2
      mean:  Sb / n + 1.01 u |mean|
      var:   dvar = (Qb + (2 |S/n| + Sb/n) Sb) / n
      rstd:  rstd ((1 - dvar / (var + eps))^-1/2 - 1) + 2.01 u rstd   (1/2 rstd dvar/(var + eps) to
             first order)
  running_mean / running_var follow torch, (1 - m) r + m x with the unbiased variance (the biased
  one at n = 1): bound m dx + 3u (|(1 - m) r| + |m x|).  num_batches_tracked grows by exactly 1.
  bn_stats_local: mean as above, M2 within n dvar + 1.01 u M2, count exact.  With n = 0: mean 0,
  rstd = fl(1/sqrt(eps)), M2 = count = 0, and the running statistics keep their values.
* bn_sync_finalize: Chan's merge in rank order in float64 (count-0 ranks skipped); every output
  within 2u of it (nvcc may contract the double expressions into FMAs, so not bit for bit).
* bn_act_fwd.  t = (y - m) r g + b, z = act(t) (+ res).  |t~ - t| <= et = 1.01 (2u |x^ g| + u |t|).
  Identity and ReLU: |dz| <= et.  SiLU (Lipschitz 1.1): 1.1 et + 1.01 |z| es, where
  es = 2 (3 + 1.173 |t|) u e/(1+e) + 3u, e = exp(-t): the __expf error of the CUDA C++ Programming
  Guide (2 + floor(|1.173 x|) ulp, an ulp <= 2u relative) plus 1 + e and the division.  Where
  e > 2^126 (__expf overflows) es = 1.  A residual adds 1.01 u |z|.  Pad rows are exactly 0.
* bn_act_bwd_reduce.  S1 = sum dz act'(t), S2 = sum dz act'(t) x^.  Per term: act' of ReLU is
  exact (its mask is restated with the kernel's own rounding, t32 = f64(x^32 g) + b with
  x^32 = f32(f32(y - m) r): the product is exact in float64 and rounding keeps the sign); SiLU' is
  off by 0.5 et (|SiLU''| <= 0.5) + s (1 + |t|) (2 es + 4u), bounded by the size of its
  intermediates because SiLU' has a root near t = -1.278; the product dz act' adds u |dz act'|,
  x^ adds 2.01 u |x^| to the S2 term.  The sum adds 1.01 (k + ty + 2) u sum |term|.  dbeta and
  dgamma equal the rows of ``sums`` bit for bit; accumulating, after == f32(before + S) bit for bit.
* bn_act_bwd_apply.  dy = g r (G - S1 inv - x^ S2 inv) with G = dz act'(t), from the kernel's own
  sums and inv = inv_n (or 1/n).  Bound 1.01 |g r| (eG + c u (|G| + |S1 inv| + |x^ S2 inv|)), eG
  the per-term error of G above, c = 7 roundings (8 when the kernel forms 1/(float)n itself).
  dbias against the float64 sum of the kernel's own dy over the valid rows, within
  1.01 (k + ty + 2) u sum |dy|.  Pad rows of dy are exactly 0.  Accumulation as for the reduce.
* sum_slabs: fixed order, nothing fused, restated exactly in numpy float32 and compared bit for bit.

Every case asserts the split it reaches; every launch runs twice with the same bits; tuning keys
2, 3 and 5 change only the work split, so 3 and 5 must not change a bit.
"""
import math
from collections import namedtuple

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu
DEV = "cuda"
U = 2.0 ** -24
EPS, MOM = 1e-5, 0.1
EPS32, MOM32 = float(np.float32(EPS)), float(np.float32(MOM))
SAT = 126 * math.log(2.0)         # e^-t > 2^126: __expf overflows or its reciprocal flushes


@pytest.fixture(autouse=True)
def _default_knobs():
    """Tuning is process-global: put keys 2, 3 and 5 back to their defaults after every test."""
    from pygho_b200 import _lib
    try:
        yield
    finally:
        for key in (2, 3, 5):
            _lib.call("pgh_set_tuning", key, 0)


@pytest.fixture(scope="module")
def ops():
    import pygho_b200.ops  # noqa: F401  (registers torch.ops.pygho_b200)
    return torch.ops.pygho_b200


def set_knob(key, value):
    from pygho_b200 import _lib
    _lib.call("pgh_set_tuning", key, value)


# ------------------------------------------------------------------------------ geometry
# Restates bn_geom() and pgh_bn_ws_bytes() of pygho_b200/csrc/fused_mlp.cu (kSMs from common.cuh,
# kBnThreads, kBnMaxGroups).  Keep this in step with the C source.
K_SMS, K_BN_THREADS, K_BN_MAX_GROUPS = 148, 256, 63
Geom = namedtuple("Geom", "c4 ty rows_per_block blocks grp ngroups k")


def bn_geom(rows, C, ctas_per_sm=4):
    c4 = C // 4
    ty = max(K_BN_THREADS // c4, 1)
    rpb = max(-(-rows // (K_SMS * ctas_per_sm)), 8 * ty)
    rpb = -(-rpb // ty) * ty
    blocks = -(-rows // rpb)
    grp = 16
    while -(-blocks // grp) > K_BN_MAX_GROUPS:
        grp *= 2
    ngroups = -(-blocks // grp)
    return Geom(c4, ty, rpb, blocks, grp, ngroups, rpb // ty)


def ws_bytes(g, C):
    return g.blocks * 2 * C * 4 + 256 + g.ngroups * 2 * C * 4


TY = {4: 256, 12: 85, 16: 64, 128: 8, 384: 2, 516: 1, 1024: 1}


def split_rows(C):
    """rows -> (blocks, ngroups) for the splits every width must reach; all have k = 8."""
    cta = 8 * TY[C]
    out = {1: (1, 1), TY[C] - 1: (1, 1), cta: (1, 1), cta + 1: (2, 1), 16 * cta - 1: (16, 1),
           16 * cta + 1: (17, 2), 592 * cta - 3: (592, 37)}
    out.pop(0, None)
    return out


# name -> (rows, C, (blocks, ngroups, k)): the split each case must reach
CASES = {f"C{C}_r{rows}": (rows, C, (b, g, 8)) for C in TY for rows, (b, g) in split_rows(C).items()}
ZINC = {"zinc_C128": (230147, 128, (588, 37, 49)),          # ZINC-scale batches
        "zinc_C384": (230147, 384, (591, 37, 195)),
        "C1024_r100000": (100000, 1024, (592, 37, 169))}
KNOB2 = {1: (148, 10, 16, 195), 8: (1151, 36, 32, 25), 16: (2213, 35, 64, 13)}  # blocks ngroups grp k
ROWS_DEV_CAPS = {12: 16 * 680 + 1, 128: 592 * 64 - 3, 1024: 17 * 8}


def test_geometry_restatement_matches_workspace_size():
    """Ties bn_geom above to the C code: the workspace size it implies equals pgh_bn_ws_bytes for
    every case of this file, at every key-2 setting used; needs no device."""
    from pygho_b200 import _lib
    lib = _lib.load()
    shapes = [(r, C, 0) for r, C, _ in list(CASES.values()) + list(ZINC.values())]
    shapes += [(230147, 128, cps) for cps in KNOB2] + [(cap, C, 0) for C, cap in ROWS_DEV_CAPS.items()]
    shapes += [(r, C, cps) for cps in (1, 2, 8, 16, 64) for r in (1, 777, 230147, 4_000_000)
               for C in (4, 12, 128, 384, 1024)]
    for rows, C, cps in shapes:
        set_knob(2, cps)
        g = bn_geom(rows, C, cps or 4)
        assert ws_bytes(g, C) == int(lib.pgh_bn_ws_bytes(rows, C)), (rows, C, cps, g)
        assert g.ngroups <= K_BN_MAX_GROUPS and g.blocks <= g.grp * g.ngroups
    for rows, C, (blocks, ngroups, k) in list(CASES.values()) + list(ZINC.values()):
        g = bn_geom(rows, C)
        assert (g.ty, g.blocks, g.ngroups, g.k) == (TY[C], blocks, ngroups, k), (rows, C, g)
    for cps, (blocks, ngroups, grp, k) in KNOB2.items():
        assert bn_geom(230147, 128, cps)[3:] == (blocks, grp, ngroups, k)
    assert bn_geom(5000, 12).c4 * bn_geom(5000, 12).ty == 255


# ------------------------------------------------------------------------------ data
def make_inputs(rows, C, cap, seed, gb="affine"):
    """y (cap, C): columns cycle through four kinds -- standard normal; mean 1e3 with std 1e-2 (needs
    the shift); standard normal with row 0 a 50-sigma outlier; constant 0.7.  dz = N(0.3, 1), so
    S1 / n is not small.  Rows past ``rows`` hold junk (x100).  gamma / beta: "affine" (beta 0 on the
    constant columns: an exact ReLU tie at t = 0), "none", or "extreme" (beta = +-90 on two kinds:
    SiLU at |t| ~ 90, where __expf overflows)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    y = torch.randn((cap, C), device=DEV, generator=g)
    kind = torch.arange(C, device=DEV) % 4
    y[:, kind == 1] = y[:, kind == 1] * 1e-2 + 1e3
    y[0, kind == 2] = 50.0
    y[:, kind == 3] = 0.7
    dz = torch.randn((cap, C), device=DEV, generator=g) + 0.3
    if cap > rows:
        y[rows:] = torch.randn((cap - rows, C), device=DEV, generator=g) * 100.0
        dz[rows:] = torch.randn((cap - rows, C), device=DEV, generator=g) * 100.0
    res = torch.randn((cap, C), device=DEV, generator=g)
    gamma = beta = None
    if gb != "none":
        gamma = (torch.rand(C, device=DEV, generator=g) + 0.5) * torch.where(
            torch.rand(C, device=DEV, generator=g) < 0.3, -1.0, 1.0)
        beta = torch.randn(C, device=DEV, generator=g) * 0.5
        beta[kind == 3] = 0.0
        if gb == "extreme":
            beta[kind == 0], beta[kind == 1] = 90.0, -90.0
    return y, dz, res, gamma, beta


# ------------------------------------------------------------------------------ checks
def same_bits(x, y):
    return x.shape == y.shape and torch.equal(x.contiguous().view(torch.int32),
                                              y.contiguous().view(torch.int32))


def assert_within(got, want, bound, what):
    err = (got.double() - want).abs()
    bad = ~(err <= bound)                            # NaN counts as bad
    if bool(bad.any()):
        i = tuple(int(v) for v in bad.nonzero()[0])
        raise AssertionError(
            f"{what}: {int(bad.sum())} of {bad.numel()} outside the bound; first at {i}: got "
            f"{float(got[i])!r} want {float(want[i])!r} bound {float(bound[i]):.3g}")


def assert_zero_bits(t, what):
    assert bool((t.contiguous().view(torch.int32) == 0).all()), f"{what}: not +0.0"


def twice(fn):
    a, b = fn(), fn()
    for x, y in zip(a, b):
        assert same_bits(x, y), "two launches differ"
    return a


def affine64(gamma, beta, C):
    g = gamma.double() if gamma is not None else torch.ones(C, dtype=torch.float64, device=DEV)
    b = beta.double() if beta is not None else torch.zeros(C, dtype=torch.float64, device=DEV)
    return g, b


def silu_es(t):
    """Relative error of the kernel's sigmoid s~ = 1 / (1 + __expf(-t)) (module docstring)."""
    e = torch.exp(-t)
    es = 2.0 * (3.0 + 1.173 * t.abs()) * U * e / (1.0 + e) + 3.0 * U
    return torch.where(-t > SAT, torch.ones_like(es), es)


class Pointwise:
    """float64 x^, t, act(t), act'(t) over the first n rows, from the kernel's mean / rstd, with
    the per-element error bounds of the module docstring."""

    def __init__(self, y, mean, rstd, gamma, beta, act, n):
        C = y.shape[1]
        g, b = affine64(gamma, beta, C)
        yv = y[:n]
        self.x = (yv.double() - mean.double()) * rstd.double()
        xg = self.x * g
        t = xg + b
        self.et = 1.01 * U * (2.0 * xg.abs() + t.abs())
        if act == 0:
            self.z, self.ez = t, self.et
            self.ap, self.eap = torch.ones_like(t), torch.zeros_like(t)
        elif act == 2:
            self.z, self.ez = t.clamp(min=0.0), self.et
            x32 = (yv - mean) * rstd                                # f32(f32(y - m) * r)
            self.ap = ((x32.double() * g + b) > 0).double()         # the kernel's exact mask
            self.eap = torch.zeros_like(t)
        else:
            s, es = torch.sigmoid(t), silu_es(t)
            self.z = t * s
            self.ez = 1.1 * self.et + 1.01 * self.z.abs() * es
            self.ap = s * (1.0 + t * (1.0 - s))
            self.eap = 0.5 * self.et + s * (1.0 + t.abs()) * (2.0 * es + 4.0 * U)
        self.gr = g * rstd.double()


def check_stats(ops, y, rows_dev, n, geo, what):
    """bn_stats (with running statistics and num_batches_tracked) and bn_stats_local; -> (mean, rstd)."""
    C = y.shape[1]
    gen = torch.Generator(device=DEV).manual_seed(C + n)
    rm0 = torch.randn(C, device=DEV, generator=gen)
    rv0 = torch.rand(C, device=DEV, generator=gen) + 0.5
    runs = []
    for _ in range(2):
        rm, rv = rm0.clone(), rv0.clone()
        nbt = torch.tensor(41, dtype=torch.int64, device=DEV)
        mean, rstd = ops.bn_stats(y, EPS, MOM, rm, rv, rows_dev, nbt)
        runs.append((mean, rstd, rm, rv))
        assert int(nbt) == 42, f"{what}: num_batches_tracked"
    for a, b in zip(*runs):
        assert same_bits(a, b), f"{what}: two bn_stats launches differ"
    mean, rstd, rm, rv = runs[0]
    nbt = torch.tensor(5, dtype=torch.int64, device=DEV)
    local = twice(lambda: (ops.bn_stats_local(y, rows_dev, nbt),))[0]
    assert int(nbt) == 7, f"{what}: num_batches_tracked (local)"
    assert bool((local[2] == float(n)).all()), f"{what}: count"
    if n == 0:
        assert_zero_bits(mean, what + " mean")
        assert bool((rstd == float(np.float32(1.0 / math.sqrt(EPS32)))).all()), what + " rstd"
        assert same_bits(rm, rm0) and same_bits(rv, rv0), f"{what}: running statistics moved"
        assert_zero_bits(local, what + " local")
        return mean, rstd
    yv = y[:n].double()
    d = yv - yv[0]
    S, A, Q = d.sum(0), d.abs().sum(0), (d * d).sum(0)
    m = yv[0] + S / n
    var = ((yv - m) ** 2).sum(0) / n
    kk = geo.k + geo.ty
    Sb, Qb = 1.01 * (kk + 2) * U * A, 1.01 * (kk + 3) * U * Q
    bm = Sb / n + 1.01 * U * m.abs()
    dvar = (Qb + (2.0 * S.abs() / n + Sb / n) * Sb) / n
    assert_within(mean, m, bm, what + " mean")
    r = 1.0 / torch.sqrt(var + EPS32)
    rel = dvar / (var + EPS32)
    br = r * ((1.0 - rel).clamp(min=1e-300).rsqrt() - 1.0) + 2.01 * U * r
    assert_within(rstd, r, br, what + " rstd")
    assert_within(local[0], m, bm, what + " local mean")
    assert_within(local[1], var * n, n * dvar + 1.01 * U * var * n, what + " local M2")
    unb, dunb = (var * n / (n - 1), dvar * n / (n - 1)) if n > 1 else (var, dvar)
    keep = 1.0 - MOM32
    for got, old, x, dx, name in ((rm, rm0, m, bm, "running_mean"),
                                  (rv, rv0, unb, dunb + 1.01 * U * unb, "running_var")):
        old = old.double()
        assert_within(got, keep * old + MOM32 * x,
                      MOM32 * dx + 3.0 * U * ((keep * old).abs() + (MOM32 * x).abs()), f"{what} {name}")
    return mean, rstd


def check_fwd(ops, y, mean, rstd, gamma, beta, act, res, rows_dev, n, what, pw):
    z = twice(lambda: (ops.bn_act_fwd(y, mean, rstd, gamma, beta, act, res, rows_dev),))[0]
    assert_zero_bits(z[n:], what + " fwd pad rows")
    want, bound = pw.z, pw.ez
    if res is not None:
        want = want + res[:n].double()
        bound = bound + 1.01 * U * (want.abs() + bound)
    assert bool(torch.isfinite(z).all()), what + " fwd not finite"
    assert_within(z[:n], want, bound, what + " fwd")


def reduce_terms(dz, n, pw):
    """float64 terms G = dz act'(t) and their per-element errors eG."""
    dzv = dz[:n].double()
    G = dzv * pw.ap
    eG = 1.01 * (dzv.abs() * pw.eap + U * G.abs())
    return G, eG


def check_reduce(ops, dz, y, mean, rstd, gamma, beta, act, rows_dev, n, geo, what, pw, acc):
    sums, dgamma, dbeta = twice(lambda: ops.bn_act_bwd_reduce(dz, y, mean, rstd, gamma, beta, act,
                                                              rows_dev, None, None))
    assert bool(torch.isfinite(sums).all()), what + " sums not finite"
    assert same_bits(dbeta, sums[0]) and same_bits(dgamma, sums[1]), what + " dbeta / dgamma"
    G, eG = reduce_terms(dz, n, pw)
    x = pw.x
    T2 = G * x
    eT2 = 1.01 * eG * x.abs() + 2.01 * U * T2.abs()
    red = 1.01 * (geo.k + geo.ty + 2) * U
    assert_within(sums[0], G.sum(0), eG.sum(0) + red * G.abs().sum(0), what + " S1")
    assert_within(sums[1], T2.sum(0), eT2.sum(0) + red * T2.abs().sum(0), what + " S2")
    if acc:
        C = y.shape[1]
        g0 = torch.randn(C, device=DEV)
        b0 = torch.randn(C, device=DEV)
        ga, ba = g0.clone(), b0.clone()
        s2, _, _ = ops.bn_act_bwd_reduce(dz, y, mean, rstd, gamma, beta, act, rows_dev, ga, ba)
        assert same_bits(s2, sums), what + " sums (accumulating)"
        assert same_bits(ba, b0 + sums[0]) and same_bits(ga, g0 + sums[1]), what + " accumulate"
    return sums, G, eG


def check_apply(ops, dz, y, mean, rstd, gamma, beta, sums, inv_n, act, rows_dev, n, geo, what, pw,
                G, eG, acc):
    dy, dbias = twice(lambda: ops.bn_act_bwd_apply(dz, y, mean, rstd, gamma, beta, sums, inv_n, act,
                                                   rows_dev, True, None))
    assert_zero_bits(dy[n:], what + " dy pad rows")
    assert bool(torch.isfinite(dy).all()), what + " dy not finite"
    if n:
        if inv_n is not None:
            inv, c = inv_n.double(), 7.0
        else:
            inv, c = 1.0 / n, 8.0
        s1, s2 = sums[0].double() * inv, sums[1].double() * inv
        x = pw.x
        want = pw.gr * (G - s1 - x * s2)
        bound = 1.01 * pw.gr.abs() * (eG + c * U * (G.abs() + s1.abs() + (x * s2).abs()))
        assert_within(dy[:n], want, bound, what + " dy")
    dyv = dy[:n].double()
    assert_within(dbias, dyv.sum(0), 1.01 * (geo.k + geo.ty + 2) * U * dyv.abs().sum(0),
                  what + " dbias")
    if acc:
        b0 = torch.randn(y.shape[1], device=DEV)
        ba = b0.clone()
        dy2, _ = ops.bn_act_bwd_apply(dz, y, mean, rstd, gamma, beta, sums, inv_n, act, rows_dev,
                                      True, ba)
        assert same_bits(dy2, dy) and same_bits(ba, b0 + dbias), what + " dbias accumulate"


def check_chain(ops, rows, C, cap, rows_dev, geo, seed, what, acts=(0, 1, 2),
                gbs=("affine", "none", "extreme")):
    """Statistics, then for every activation and gamma / beta form the forward apply, the backward
    reduce and the backward apply, each against float64."""
    n = rows if rows_dev is None else min(max(int(rows_dev), 0), cap)
    for gb in gbs:
        y, dz, res, gamma, beta = make_inputs(n, C, cap, seed, gb)
        if gb == gbs[0]:
            mean, rstd = check_stats(ops, y, rows_dev, n, geo, what)
        for act in acts:
            tag = f"{what} {gb} act={act}"
            pw = Pointwise(y, mean, rstd, gamma, beta, act, n)
            check_fwd(ops, y, mean, rstd, gamma, beta, act, None, rows_dev, n, tag, pw)
            if gb != "none":
                check_fwd(ops, y, mean, rstd, gamma, beta, act, res, rows_dev, n, tag + " res", pw)
            sums, G, eG = check_reduce(ops, dz, y, mean, rstd, gamma, beta, act, rows_dev, n, geo,
                                       tag, pw, acc=gb == "affine")
            inv_n = None
            if gb == "extreme" and n:
                inv_n = torch.tensor([1.0 / n], dtype=torch.float32, device=DEV)
            check_apply(ops, dz, y, mean, rstd, gamma, beta, sums, inv_n, act, rows_dev, n, geo, tag,
                        pw, G, eG, acc=gb == "affine")
            del pw, G, eG


# ------------------------------------------------------------------------------ tests
@gpu
@pytest.mark.parametrize("name", list(CASES) + list(ZINC))
def test_batchnorm_chain_vs_fp64(ops, name):
    """Every width (ty 256, 85, 64, 8, 2, 1; C = 1024 has more finalize than reduce shared memory)
    at one row, fewer rows than lanes, one full CTA, one more row, 16 CTAs, 17 CTAs (a second
    group with one CTA of one row), 592 CTAs in 37 groups, and ZINC-scale batches (k = 49, 195,
    169)."""
    rows, C, split = {**CASES, **ZINC}[name]
    geo = bn_geom(rows, C)
    assert (geo.blocks, geo.ngroups, geo.k) == split
    check_chain(ops, rows, C, rows, None, geo, seed=rows + C, what=name)


@gpu
@pytest.mark.parametrize("cps", list(KNOB2))
def test_ctas_per_sm_knob_splits(ops, cps):
    """Key 2 at 1, 8 and 16 CTAs per SM: 10 groups of 16, groups of 32 and groups of 64."""
    set_knob(2, cps)
    geo = bn_geom(230147, 128, cps)
    blocks, ngroups, grp, k = KNOB2[cps]
    assert (geo.blocks, geo.ngroups, geo.grp, geo.k) == (blocks, ngroups, grp, k)
    check_chain(ops, 230147, 128, 230147, None, geo, seed=cps, what=f"ctas/sm={cps}",
                gbs=("affine", "extreme"))


ROWS_DEV = {"0": lambda cap: 0, "1": lambda cap: 1, "cap-1": lambda cap: cap - 1,
            "cap": lambda cap: cap, "above": lambda cap: cap + 5, "negative": lambda cap: -3}


@gpu
@pytest.mark.parametrize("C", list(ROWS_DEV_CAPS))
@pytest.mark.parametrize("rd", list(ROWS_DEV))
def test_rows_dev_vs_fp64(ops, C, rd):
    """Device-side row counts on a padded tensor with junk pad rows: 0 and negative (no valid row),
    1, capacity - 1, capacity, and above capacity (clamped)."""
    cap = ROWS_DEV_CAPS[C]
    geo = bn_geom(cap, C)
    rows_dev = torch.tensor([ROWS_DEV[rd](cap)], dtype=torch.int32, device=DEV)
    check_chain(ops, cap, C, cap, rows_dev, geo, seed=C, what=f"C={C} rows_dev={rd}",
                gbs=("affine", "extreme"))


@gpu
def test_zero_valid_rows_leave_running_statistics(ops):
    """A batch without valid rows (rows_dev <= 0, or all SyncBN ranks with count 0) gives mean 0 and
    rstd 1/sqrt(eps) and must not move the running statistics; num_batches_tracked still counts
    the call, as torch counts training forward calls."""
    C = 128
    y = torch.randn(300, C, device=DEV)
    rm0, rv0 = torch.randn(C, device=DEV), torch.rand(C, device=DEV) + 0.5
    rstd0 = float(np.float32(1.0 / math.sqrt(EPS32)))
    for v in (0, -3):
        rd = torch.tensor([v], dtype=torch.int32, device=DEV)
        rm, rv, nbt = rm0.clone(), rv0.clone(), torch.tensor(3, dtype=torch.int64, device=DEV)
        mean, rstd = ops.bn_stats(y, EPS, MOM, rm, rv, rd, nbt)
        assert same_bits(rm, rm0) and same_bits(rv, rv0), f"bn_stats rows_dev={v}"
        assert int(nbt) == 4 and not bool(mean.any()) and bool((rstd == rstd0).all())
    gathered = torch.zeros(3, 3, C, device=DEV)
    gathered[:, 0] = torch.randn(3, C, device=DEV)             # means of empty ranks: ignored
    rm, rv = rm0.clone(), rv0.clone()
    mean, rstd, inv_n = ops.bn_sync_finalize(gathered, EPS, MOM, rm, rv)
    assert same_bits(rm, rm0) and same_bits(rv, rv0), "bn_sync_finalize with no rows"
    assert not bool(mean.any()) and bool((rstd == rstd0).all()) and float(inv_n) == 0.0
    # the GEMM with the statistics epilogue finishes through the same function
    x = torch.randn(256, 128, device=DEV)
    w = torch.randn(128, 128, device=DEV) / 128 ** 0.5
    rm, rv, nbt = rm0.clone(), rv0.clone(), torch.tensor(3, dtype=torch.int64, device=DEV)
    zero = torch.zeros(1, dtype=torch.int32, device=DEV)
    yl, mean, rstd = ops.linear_stats(x, w, torch.randn(128, device=DEV), EPS, MOM, rm, rv, zero, nbt,
                                      False)
    assert same_bits(rm, rm0) and same_bits(rv, rv0), "linear_stats rows_dev=0"
    assert int(nbt) == 4 and not bool(mean.any()) and bool((rstd == rstd0).all())


def chan_reference(g64):
    world = g64.shape[0]
    n = torch.zeros_like(g64[0, 0])
    m, m2 = n.clone(), n.clone()
    for r in range(world):
        nb, mb, m2b = g64[r, 2], g64[r, 0], g64[r, 1]
        use = nb > 0
        tot = n + nb
        delta = mb - m
        m = torch.where(use, m + delta * (nb / tot), m)
        m2 = torch.where(use, m2 + m2b + delta * delta * (n * nb / tot), m2)
        n = torch.where(use, tot, n)
    return n, m, m2


@gpu
@pytest.mark.parametrize("counts", [[7], [5, 0, 1, 1000], [0, 1], [1, 1, 1], [3000, 0, 0, 2, 250000]])
def test_sync_finalize_vs_chan(ops, counts):
    """Chan's merge of float (mean, M2, count) triples in rank order, including a rank with count 0,
    a rank with count 1 and world = 1, over 130 channels (two thread blocks)."""
    C, world = 130, len(counts)
    gen = torch.Generator(device=DEV).manual_seed(world)
    g = torch.empty(world, 3, C, device=DEV)
    cnt = torch.tensor(counts, dtype=torch.float32, device=DEV)[:, None]
    g[:, 0] = torch.randn(world, C, device=DEV, generator=gen) * 3.0 + 100.0
    g[:, 1] = torch.rand(world, C, device=DEV, generator=gen) * (cnt - 1).clamp(min=0) * 4.0
    g[:, 2] = cnt
    rm0, rv0 = torch.randn(C, device=DEV, generator=gen), torch.rand(C, device=DEV, generator=gen)
    runs = []
    for _ in range(2):
        rm, rv = rm0.clone(), rv0.clone()
        runs.append(ops.bn_sync_finalize(g, EPS, MOM, rm, rv) + (rm, rv))
    for a, b in zip(*runs):
        assert same_bits(a, b), "two bn_sync_finalize launches differ"
    mean, rstd, inv_n, rm, rv = runs[0]
    n, m, m2 = chan_reference(g.double())
    var = m2 / n
    tiny = 1e-13 * g[:, 0].double().abs().max()
    assert_within(mean, m, 2 * U * m.abs() + tiny, "mean")
    r = 1.0 / torch.sqrt(var + EPS32)
    assert_within(rstd, r, 2 * U * r + r * 1e-13, "rstd")
    assert_within(inv_n, 1.0 / n[:1], 2 * U / n[:1], "inv_n")
    unb = m2 / (n - 1) if counts and float(n[0]) > 1 else var
    keep = 1.0 - MOM32
    for got, old, x, name in ((rm, rm0, m, "running_mean"), (rv, rv0, unb, "running_var")):
        old = old.double()
        want = keep * old + MOM32 * x
        assert_within(got, want, 3 * U * ((keep * old).abs() + (MOM32 * x).abs()) + MOM32 * (
            2 * U * x.abs() + tiny), name)


@gpu
def test_unroll_knobs_are_bit_identical(ops):
    """Keys 3 (rows in flight of the backward passes) and 5 (elements in flight of the forward apply)
    change neither a thread's row order nor any element-wise formula: every output keeps its bits."""
    shapes = [(230147, 128, None), (ROWS_DEV_CAPS[12], 12, ROWS_DEV_CAPS[12] - 7), (1001, 1024, 1000)]
    for rows, C, valid in shapes:
        y, dz, res, gamma, beta = make_inputs(rows if valid is None else valid, C, rows, 5, "extreme")
        rd = None if valid is None else torch.tensor([valid], dtype=torch.int32, device=DEV)

        def run_all():
            mean, rstd = ops.bn_stats(y, EPS, MOM, None, None, rd)
            out = [mean, rstd]
            for act in (0, 1, 2):
                out.append(ops.bn_act_fwd(y, mean, rstd, gamma, beta, act, res, rd))
                sums, _, _ = ops.bn_act_bwd_reduce(dz, y, mean, rstd, gamma, beta, act, rd, None, None)
                out += [sums, *ops.bn_act_bwd_apply(dz, y, mean, rstd, gamma, beta, sums, None, act, rd,
                                                    True, None)]
            return out

        base = run_all()
        for key, values in ((3, (2, 4)), (5, (1, 2, 4))):
            for v in values:
                set_knob(key, v)
                got = run_all()
                set_knob(key, 0)
                for i, (a, b) in enumerate(zip(base, got)):
                    assert same_bits(a, b), f"rows={rows} C={C} key {key}={v}: output {i} changed"


# ------------------------------------------------------------------------------ sum_slabs
def slabs_reference(part, out0, accumulate):
    """Lane y (0..7) adds slabs y, y+8, ... in ascending order from +0.0; then
    out = (accumulate ? out : 0) + lane 0 + ... + lane 7, idle lanes contributing +0.0."""
    lanes = []
    for y in range(8):
        a = np.zeros(part.shape[1], np.float32)
        for k in range(y, part.shape[0], 8):
            a = a + part[k]
        lanes.append(a)
    r = out0.copy() if accumulate else np.zeros(part.shape[1], np.float32)
    for a in lanes:
        r = r + a
    return r


@gpu
@pytest.mark.parametrize("n", [4, 132, 128 * 384])
@pytest.mark.parametrize("slabs", [1, 7, 8, 9, 63, 64])
def test_sum_slabs_bitwise(ops, n, slabs):
    rng = np.random.default_rng(n + slabs)
    part = (rng.standard_normal((slabs, n)) * 10.0 ** rng.uniform(-3, 3, (slabs, n))).astype(np.float32)
    out0 = rng.standard_normal(n).astype(np.float32)
    part_d = torch.from_numpy(part).to(DEV)
    for accumulate in (False, True):
        outs = []
        for _ in range(2):
            out = torch.tensor(out0, device=DEV)
            ops.sum_slabs(part_d, out, accumulate)
            outs.append(out)
        assert same_bits(outs[0], outs[1])
        want = slabs_reference(part, out0, accumulate)
        got = outs[0].cpu().numpy()
        assert np.array_equal(got.view(np.int32), want.view(np.int32)), \
            f"accumulate={accumulate}: {int((got != want).sum())} elements differ"
    if n == 128 * 384 and slabs == 64:                   # the order is visible at this size
        plain = np.zeros(n, np.float32)
        for k in range(slabs):
            plain = plain + part[k]
        assert not np.array_equal(plain, slabs_reference(part, out0, False))


# ------------------------------------------------------------------------------ host rejections
@gpu
def test_host_rejects_before_launch(ops):
    """Calls the host side refuses raise KernelError naming the op and leave the outputs and the
    running statistics untouched."""
    from pygho_b200._lib import KernelError, call
    C = 128
    good = torch.randn(64, C, device=DEV)
    mean, rstd = torch.zeros(C, device=DEV), torch.ones(C, device=DEV)
    rm, rv = torch.randn(C, device=DEV), torch.rand(C, device=DEV) + 0.5
    nbt = torch.tensor(9, dtype=torch.int64, device=DEV)
    acc = [torch.randn(C, device=DEV) for _ in range(3)]
    keep = [t.clone() for t in [rm, rv, nbt] + acc]
    store = torch.zeros(64 * C + 4, device=DEV)
    shifted = store[1:1 + 64 * C].view(64, C)            # one float past a 16-byte boundary
    assert shifted.data_ptr() % 16 == 4
    bad_shapes = [torch.empty(0, C, device=DEV)] + [torch.randn(16, c, device=DEV) for c in (2, 6, 1028)]
    for y in bad_shapes + [shifted]:
        c = y.shape[1]
        m, r = torch.zeros(c, device=DEV), torch.ones(c, device=DEV)
        with pytest.raises(KernelError, match="bn_stats"):
            ops.bn_stats(y, EPS, MOM, rm if c == C else None, rv if c == C else None, None,
                         nbt if c == C else None)
        with pytest.raises(KernelError, match="bn_stats"):
            ops.bn_stats_local(y, None, nbt if c == C else None)
        with pytest.raises(KernelError, match="bn_act_fwd"):
            ops.bn_act_fwd(y, m, r, None, None, 1)
        if c == C:
            with pytest.raises(KernelError, match="bn_act_bwd_reduce"):
                ops.bn_act_bwd_reduce(y, y, m, r, None, None, 1, None, acc[0], acc[1])
            sums = torch.zeros(2, c, device=DEV)
            with pytest.raises(KernelError, match="bn_act_bwd_apply"):
                ops.bn_act_bwd_apply(y, y, m, r, None, None, sums, None, 1, None, True, acc[2])
    sums = torch.zeros(2, C, device=DEV)
    with pytest.raises(KernelError, match="bn_act_fwd: act"):
        ops.bn_act_fwd(good, mean, rstd, None, None, 3)
    with pytest.raises(KernelError, match="bn_act_bwd_reduce: act"):
        ops.bn_act_bwd_reduce(good, good, mean, rstd, None, None, 3, None, acc[0], acc[1])
    with pytest.raises(KernelError, match="bn_act_bwd_apply: act"):
        ops.bn_act_bwd_apply(good, good, mean, rstd, None, None, sums, None, 3, None, True, acc[2])
    with pytest.raises(KernelError, match="bn_sync_finalize"):
        ops.bn_sync_finalize(torch.zeros(0, 3, C, device=DEV), EPS, MOM, rm, rv)
    out = torch.randn(8, device=DEV)
    out_keep = out.clone()
    with pytest.raises(KernelError, match="sum_slabs"):
        ops.sum_slabs(torch.randn(65, 8, device=DEV), out, True)
    with pytest.raises(KernelError, match="sum_slabs"):       # (the op cannot index an empty part)
        call("pgh_sum_slabs_f32", out.data_ptr(), 0, 8, out.data_ptr(), 1, None)
    out6 = torch.randn(6, device=DEV)
    out6_keep = out6.clone()
    with pytest.raises(KernelError, match="sum_slabs"):
        ops.sum_slabs(torch.randn(3, 6, device=DEV), out6, True)
    torch.cuda.synchronize()
    for a, b in zip([rm, rv, nbt] + acc, keep):
        assert torch.equal(a, b), "a rejected call wrote its outputs"
    assert same_bits(out, out_keep) and same_bits(out6, out6_keep)
