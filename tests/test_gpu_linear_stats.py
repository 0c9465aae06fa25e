"""The Linear layer with the BatchNorm statistics in its epilogue (pygho_b200/csrc/linear_stats.cu,
ticket.cuh) against a float64 reference, at every work split it uses.  The bound of its eval
instantiation is derived here too; tests/test_gpu_eval.py checks the eval kernel with it.

    training:  y = x W^T + b;  mean, rstd (+ running statistics, or the SyncBN triple) of y over the
               first n = clamp(rows_dev, 0, M) rows
    eval:      z = act((x W^T + b - rm) * gamma / sqrt(rv + eps) + beta) (+ residual), 0 past row n

u = 2^-24.  References are float64, built on the device from the inputs.  Bounds are per element or
per channel, never scaled by a global maximum; ``mag`` is the float64 sum_k |x_k| |w_k| of an output:

* GEMM (TF32 tcgen05, fp32 accumulation): ``|y - y64| <= (2^-9 + 2^-20 + 1.01 K 2^-23) mag +
  u |y64|``: at most 2^-10 of truncation per TF32 operand (2^-9 + 2^-20 per product), one
  truncating fp32 addition per K position, and the rounding of ``+ b``.  Whether the hardware
  truncates or rounds the operands, and the accumulator's internal order, are not measured; the
  bound holds for either.  With integer x, w, b in [-4, 4] every product and partial sum is an
  integer below 2^24, exact in TF32 and fp32 whatever the order: y equals y64 bit for bit.
* Statistics.  The epilogue sums v = acc (without the bias; the bias is the shift) over 32-row
  warp quarters by a 5-level fp32 transpose-reduce (the squares are rounded once before it),
  accumulates the quarter sums of a CTA's tiles in double, rounds each warp's total to float, adds
  the 4 warps in fp32 (3 additions) into the CTA's partial row, and the combine adds those rows in
  double, rounding each group's sum to float once when there is more than one group.  Every term
  passes at most 5 + 1 + 3 = 9 fp32 roundings into the partial (10 for a square) and one more into
  a group sum; the double additions (at most 13 tiles + 16 + 10 rows) stay below 2^-47 relative
  and are covered by the factor 1.01.  The reference takes d = y - b from the kernel's own y, so
  v = d +- du with du = u |y| (0 without a bias): y = fl(v + b).  With A = sum (|d| + du) and
  A2 = sum (|d| + du)^2 over the rows concerned:
      CTA partial:  |S - sum d|   <= 1.01 * 9 u A  + sum du
                    |Q - sum d^2| <= 1.01 * 10 u A2 + sum (2 |d| du + du^2)
      whole batch:  Sb, Qb the same with 10 and 11 roundings
      mean:  Sb / n + 1.01 u |mean|
      var:   dvar = (Qb + (2 |S/n| + Sb/n) Sb) / n  (m2 = Q - S S / n in double)
      rstd:  rstd ((1 - dvar / (var + eps))^-1/2 - 1) + 2.01 u rstd
  Q carries 11 u of sum d^2 = n (mean_d^2 + var): where |mean_d| / std is 10 to 30 (the post-SiLU
  family; the kernel shifts only by the bias) this cancellation term dominates dvar.  Running
  statistics follow torch (unbiased variance, the biased one at n = 1) within m dx + 3u (|(1-m) r|
  + |m x|); num_batches_tracked grows by exactly 1; the SyncBN triple has the mean bound, M2 within
  n dvar + 1.01 u M2 and the count exact.  n = 0: mean 0, rstd = fl(1/sqrt(eps)), running
  statistics unchanged.
  On top of the bounds, the combine and the finalize are restated exactly from the kernel's own
  CTA partials: the group rows and the mean bit for bit, rstd and M2 within 1 ulp (nvcc may
  contract Q - S * ms into an FMA).  With x, w in {-1, 0, 1}, K = 32 and integer b, the test checks
  that sum |v| and sum v^2 stay below 2^24 per channel, so every fp32 partial (a sum over a subset
  of rows) is exact: the CTA partials equal the integer sums, and mean and rstd are within 1 ulp
  of float64 from the exact sums.
* Eval.  s = fl(gamma rsqrtf(fl(rv + eps))) is within es = 5.5 u |s| (the sum's rounding, 0.5 u
  after the root; rsqrtf 2 ulp <= 4 u; the product u); shift = fma(fl(b - rm), s, beta) within
  |b - rm| es + u |b - rm| |s| + u |shift|; t = fma(v, s, shift) within |s| eg + |y64 - b| es +
  eshift + u |t| (eg the GEMM bound without the bias term); all times 1.01.  Identity and ReLU
  pass that error on; SiLU gives 1.1 et + 1.01 |z| es(t), with the __expf model of
  tests/test_gpu_batchnorm.py; a residual adds 1.01 u (|z| + bound).  Pad rows are exactly 0 and the
  running statistics keep their bits.

Every launch runs twice with the same bits, and a third time with the same bits with programmatic
dependent launch off (tuning key 8 = 0).  Each case asserts the split it reaches through the
restatement of ls_geom / ls_grid / pgh_linear_stats_ws_bytes below, tied to the device by direct
launches into a NaN-filled workspace with a zeroed ticket buffer of the test's own: exactly ``grid``
partial rows written, ``ngroups`` group rows when there is more than one group and none otherwise,
every ticket back to 0, and each CTA's partial row equal (within the bound) to the sums over the
tiles that CTA owns.
"""
import math
import os
from collections import namedtuple

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu
DEV = "cuda"
U = 2.0 ** -24
NAN, INF = float("nan"), float("inf")
EPS, MOM = 1e-5, 0.1
EPS32, MOM32 = float(np.float32(EPS)), float(np.float32(MOM))
SAT = 126 * math.log(2.0)         # e^-t > 2^126: __expf overflows or its reciprocal flushes
RATIOS = {}                       # family -> worst |error| / bound (printed after the module)


@pytest.fixture(autouse=True)
def _reset_knobs():
    """Key 8 (programmatic dependent launch) is process-global: back to its default."""
    try:
        yield
    finally:
        if torch.cuda.is_available():
            set_pdl(True)


@pytest.fixture(scope="module", autouse=True)
def _report_ratios():
    yield
    if RATIOS:
        print("\nworst |error| / bound: " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(RATIOS.items())))


@pytest.fixture(scope="module")
def ops():
    import pygho_b200.ops  # noqa: F401  (registers torch.ops.pygho_b200)
    return torch.ops.pygho_b200


def call(name, *args):
    from pygho_b200 import _lib
    _lib.call(name, *args)


def ptr(t):
    return None if t is None else t.data_ptr()


def stream_of(s=None):
    from pygho_b200._lib import stream_ptr
    if s is None:
        return stream_ptr(torch.device(DEV))
    return s.cuda_stream


def cdiv(a, b):
    return -(-a // b)


# ------------------------------------------------------------------------------ geometry
# Restates ls_grid, ls_geom, LsCfg and pgh_linear_stats_ws_bytes / pgh_linear_stats_supported of
# pygho_b200/csrc/linear_stats.cu (kSMs from common.cuh).  Keep this in step with the C source.
K_SMS, BM, BK, GRP, MAX_N, MAX_K = 148, 128, 32, 16, 384, 4096
STAGES = {1: 5, 2: 3, 3: 3}        # NT = N / 128 -> shared-memory ring stages
ACC_BUFS = {1: 2, 2: 2, 3: 1}      # NT -> TMEM accumulator buffers
Geom = namedtuple("Geom", "tiles grid grp ngroups")


def ls_geom(M):
    tiles = cdiv(M, BM)
    grid = min(tiles, K_SMS)
    return Geom(tiles, grid, GRP, cdiv(grid, GRP))


def part2_offset(g, N):
    """Byte offset of the group rows: the CTA partials (grid x 2N floats, the launch's own N)
    rounded up to 256 bytes."""
    return cdiv(g.grid * 2 * N * 4, 256) * 256


def ws_bytes(M):
    if M <= 0:
        return 256
    g = ls_geom(M)
    return part2_offset(g, MAX_N) + g.ngroups * 2 * MAX_N * 4 + 256


def supported(M, K, N):
    return M > 0 and N in (128, 256, 384) and BK <= K <= MAX_K and K % BK == 0


def tiles_of(g, b):
    return len(range(b, g.tiles, g.grid))


# M -> (grid, ngroups, CTAs in the last group, tiles of CTA 0)
SPLITS = {1: (1, 1, 1, 1), 127: (1, 1, 1, 1), 128: (1, 1, 1, 1),         # single CTA
          129: (2, 1, 2, 1), 2048: (16, 1, 16, 1),                          # one group
          2049: (17, 2, 1, 1),                                              # last group of 1
          18944: (148, 10, 4, 1), 18945: (148, 10, 4, 2),                   # 148 CTAs; CTA 0: 2 tiles
          37889: (148, 10, 4, 3),                                           # accumulator 0 reused
          75777: (148, 10, 4, 5),                                           # both buffers wrap
          230147: (148, 10, 4, 13)}                                         # ZINC scale: 12-13 tiles
LAST_ROWS = {1: 0, 32: 0, 33: 1, 80: 2, 97: 3, 127: 3}   # M % 128 -> warp quarter of the last row
KS = (32, 64, 96, 160, 192, 384, 4096)


def split_of(M):
    g = ls_geom(M)
    return g.grid, g.ngroups, g.grid - (g.ngroups - 1) * g.grp, tiles_of(g, 0)


def test_geometry_restatement_matches_workspace_size():
    """Ties the restatement to the C code without a device: the workspace size it implies equals
    pgh_linear_stats_ws_bytes over a sweep of M, the supported shapes agree, and every case of this
    file reaches the split its table names."""
    from pygho_b200 import _lib
    lib = _lib.load()
    Ms = list(range(-2, 1200)) + [m + e for m in (2048, 18944, 37888, 75776, 230144, 2 ** 24)
                                  for e in (-1, 0, 1, 127, 128, 129)] + [16777516, 10 ** 8]
    for M in Ms:
        assert ws_bytes(M) == int(lib.pgh_linear_stats_ws_bytes(M)), M
        if M > 0:
            g = ls_geom(M)
            assert g.ngroups <= 10 and g.grid <= g.grp * g.ngroups
            assert part2_offset(g, MAX_N) + g.ngroups * 2 * MAX_N * 4 <= ws_bytes(M)
    for M in (1, 127, 4096, 230147):
        for K in (0, 16, 31, 32, 48, 64, 4064, 4096, 4128, 8192):
            for N in (64, 128, 192, 256, 384, 512):
                assert supported(M, K, N) == bool(lib.pgh_linear_stats_supported(M, K, N)), (M, K, N)
    assert not lib.pgh_linear_stats_supported(0, 32, 128)
    for M, split in SPLITS.items():
        assert split_of(M) == split, (M, split_of(M))
    assert tiles_of(ls_geom(230147), 147) == 12
    for r, q in LAST_ROWS.items():
        assert (r - 1) // 32 == q
    for NT in (1, 2, 3):
        # K reaches kblocks below, equal to and above the ring's stage count; CTA 0 reuses every
        # accumulator buffer (3 tiles for two buffers, 2 for one) and wraps its phase (5 and 3)
        assert {(kb > STAGES[NT]) - (kb < STAGES[NT]) for kb in (K // BK for K in KS)} == {-1, 0, 1}
        assert tiles_of(ls_geom(37889), 0) >= ACC_BUFS[NT] + 1
        assert tiles_of(ls_geom(75777), 0) >= 2 * ACC_BUFS[NT] + 1


# ------------------------------------------------------------------------------ checks
def same_bits(a, b):
    if a is None or b is None:
        return a is None and b is None
    if a.dtype == torch.float32:
        a, b = a.view(torch.int32), b.view(torch.int32)
    return a.shape == b.shape and torch.equal(a, b)


def check_bound(family, got, want, bound, what):
    """|got - want| <= bound per element (NaN fails); records the worst ratio of the family."""
    err = (got.double() - want).abs()
    ok = err <= bound
    if not bool(ok.all()):
        bad = ~ok
        i = tuple(int(v) for v in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} outside the bound; first at "
                             f"{i}: got {float(got[i])!r} want {float(want[i])!r} bound {float(bound[i]):.3g}")
    pos = bound > 0
    if bool(pos.any()):
        RATIOS[family] = max(RATIOS.get(family, 0.0), float((err[pos] / bound[pos]).max()))


def ulps(a, b):
    """Distance in float32 ulps of two arrays of finite floats of one sign."""
    a = np.asarray(a, np.float32).view(np.int32).astype(np.int64)
    b = np.asarray(b, np.float32).view(np.int32).astype(np.int64)
    return np.abs(a - b)


PDL_DEFAULT = 0 if os.environ.get("PYGHO_B200_NO_PDL") else 1     # _lib.load() applies the variable


def set_pdl(on):
    """Key 8 off, or back to its default."""
    call("pgh_set_tuning", 8, PDL_DEFAULT if on else 0)


def gemm_ref(x, w, b, rows=None):
    """float64 y and mag over the first ``rows`` rows."""
    xd = (x if rows is None else x[:rows]).double()
    wd = w.double()
    y = xd @ wd.t()
    mag = xd.abs() @ wd.abs().t()
    if b is not None:
        y = y + b.double()
    return y, mag


def gemm_bound(K, mag, y64, bias_term=True):
    bound = (2.0 ** -9 + 2.0 ** -20 + 1.01 * K * 2.0 ** -23) * mag
    return bound + U * y64.abs() if bias_term else bound


Launch = namedtuple("Launch", "y mean rstd local part part2 rm rv nbt")


def direct(x, w, b, rows_dev=None, local=False, running=None, tickets=None, stream=None, sync=True):
    """One pgh_linear_stats_f32 call into a NaN-filled workspace (and a NaN-filled y with a guard
    row after it) with a ticket buffer of the test's own.  ``running`` = (rm, rv, nbt) to update."""
    M, K = x.shape
    N = w.shape[0]
    g = ls_geom(M)
    nws = ws_bytes(M)
    ws = torch.full((nws // 4,), NAN, device=DEV)
    own = tickets is None
    if own:
        tickets = torch.zeros(1 + g.ngroups + 31, dtype=torch.int32, device=DEV)
    ybuf = torch.full((M + 1, N), NAN, device=DEV)
    y = ybuf[:M]
    mean = rstd = lo = None
    if local:
        lo = torch.full((3, N), NAN, device=DEV)
    else:
        mean, rstd = torch.full((N,), NAN, device=DEV), torch.full((N,), NAN, device=DEV)
    rm, rv, nbt = running if running is not None else (None, None, None)
    call("pgh_linear_stats_f32", ptr(x), M, K, ptr(w), N, ptr(b), ptr(rows_dev), ptr(y), EPS, MOM,
         ptr(mean), ptr(rstd), ptr(rm), ptr(rv), ptr(lo), ptr(nbt), ptr(ws), nws, ptr(tickets),
         stream_of(stream))
    if not sync:
        return ws, tickets, ybuf, Launch(y, mean, rstd, lo, None, None, rm, rv, nbt)
    torch.cuda.synchronize()
    return check_workspace(ws, tickets, ybuf, g, N, Launch(y, mean, rstd, lo, None, None, rm, rv, nbt),
                           own)


def check_workspace(ws, tickets, ybuf, g, N, L, own=True):
    """Exactly ``grid`` partial rows, ``ngroups`` group rows when ngroups > 1 (none otherwise),
    nothing else written, tickets zero, the guard row of y untouched."""
    W = 2 * N
    assert bool((tickets == 0).all()), f"tickets not reset: {tickets.nonzero().flatten().tolist()}"
    assert bool(torch.isnan(ybuf[-1]).all()), "y written past row M"
    part = ws[:g.grid * W]
    assert not bool(torch.isnan(part).any()), "a CTA partial row not written"
    o2 = part2_offset(g, N) // 4
    assert bool(torch.isnan(ws[g.grid * W:o2]).all()), "written past the CTA partials"
    part2 = None
    end = o2
    if g.ngroups > 1:
        part2 = ws[o2:o2 + g.ngroups * W]
        assert not bool(torch.isnan(part2).any()), "a group row not written"
        part2 = part2.view(g.ngroups, W).cpu().numpy()
        end = o2 + g.ngroups * W
    assert bool(torch.isnan(ws[end:]).all()), "written past the group rows"
    return L._replace(part=part.view(g.grid, W).cpu().numpy(), part2=part2)


def three(fn, what):
    """fn() twice and once more without programmatic dependent launch: the same bits."""
    runs = [fn(), fn()]
    set_pdl(False)
    try:
        runs.append(fn())
    finally:
        set_pdl(True)
    for other in runs[1:]:
        for f in Launch._fields:
            a, c = getattr(runs[0], f), getattr(other, f)
            if isinstance(a, np.ndarray):
                assert np.array_equal(a.view(np.int32), c.view(np.int32)), f"{what}: {f} differs"
            elif f != "nbt":
                assert same_bits(a, c), f"{what}: {f} differs between launches"
    return runs[0]


def seq_sum(rows):
    acc = np.zeros(rows.shape[1], np.float64)
    for r in rows:
        acc = acc + r
    return acc


def restate_combine(L, g, N):
    """fin (float64) from the kernel's own CTA partials, in ticketed_combine's order; checks the
    group rows bit for bit."""
    p = L.part.astype(np.float64)
    if g.grid == 1:
        return p[0]
    if g.ngroups == 1:
        return seq_sum(p)
    p2 = np.stack([seq_sum(p[i * GRP:(i + 1) * GRP]) for i in range(g.ngroups)]).astype(np.float32)
    assert np.array_equal(p2.view(np.int32), L.part2.view(np.int32)), "group rows"
    return seq_sum(p2.astype(np.float64))


def check_finalize(L, g, N, b, n, what):
    """bn_finalize_stats restated from fin: mean (or the triple's mean) bit for bit, rstd / M2
    within 1 ulp, the count exact."""
    fin = restate_combine(L, g, N)
    S, Q = fin[:N], fin[N:]
    bb = b.double().cpu().numpy() if b is not None else 0.0
    if n > 0:
        ms = S / n
        m = ms + bb
    else:
        ms = m = np.zeros(N)
    m2 = np.maximum(Q - S * ms, 0.0)
    var = m2 / n if n > 0 else np.zeros(N)
    if L.local is not None:
        lo = L.local.cpu().numpy()
        assert np.array_equal(lo[0].view(np.int32), m.astype(np.float32).view(np.int32)), what + " triple mean"
        assert ulps(lo[1], m2.astype(np.float32)).max() <= 1, what + " triple M2"
        assert bool((lo[2] == np.float32(n)).all()), what + " triple count"
        return
    mean, rstd = L.mean.cpu().numpy(), L.rstd.cpu().numpy()
    assert np.array_equal(mean.view(np.int32), m.astype(np.float32).view(np.int32)), what + " mean"
    assert ulps(rstd, (1.0 / np.sqrt(var + EPS32)).astype(np.float32)).max() <= 1, what + " rstd"


class VRef:
    """float64 d = y - b over the first n rows (the kernel's own y) and its uncertainty du."""

    def __init__(self, y, b, n):
        yv = y[:n].double()
        if b is not None:
            self.d, self.du = yv - b.double(), U * yv.abs()
        else:
            self.d, self.du = yv, torch.zeros_like(yv)
        self.n = n
        self.a = self.d.abs() + self.du
        self.dq = 2.0 * self.d.abs() * self.du + self.du * self.du

    def by_cta(self, t, g):
        cta = (torch.arange(self.n, device=DEV) // BM) % g.grid
        return torch.zeros((g.grid, t.shape[1]), dtype=torch.float64, device=DEV).index_add_(0, cta, t)


def check_partials(L, v, g, N, what):
    part = torch.from_numpy(L.part).to(DEV)
    S, Q = part[:, :N], part[:, N:]
    d = v.d
    check_bound("CTA partials", S, v.by_cta(d, g), 1.01 * 9 * U * v.by_cta(v.a, g) + v.by_cta(v.du, g),
                what + " partial S")
    check_bound("CTA partials", Q, v.by_cta(d * d, g),
                1.01 * 10 * U * v.by_cta(v.a * v.a, g) + v.by_cta(v.dq, g), what + " partial Q")


def check_stats(L, Lloc, v, b, rm0, rv0, what, family="statistics"):
    n = v.n
    if n == 0:
        assert not bool(L.mean.any()), what + " mean"
        assert bool((L.rstd == float(np.float32(1.0 / math.sqrt(EPS32)))).all()), what + " rstd"
        assert same_bits(L.rm, rm0) and same_bits(L.rv, rv0), what + ": running statistics moved"
        assert not bool(Lloc.local.any()), what + " triple"
        return
    d = v.d
    S = d.sum(0)
    Sb = 1.01 * 10 * U * v.a.sum(0) + v.du.sum(0)
    Qb = 1.01 * 11 * U * (v.a * v.a).sum(0) + v.dq.sum(0)
    shift = b.double() if b is not None else 0.0
    m = S / n + shift
    var = ((d - S / n) ** 2).sum(0) / n
    bm = Sb / n + 1.01 * U * m.abs()
    dvar = (Qb + (2.0 * S.abs() / n + Sb / n) * Sb) / n
    check_bound(family, L.mean, m, bm, what + " mean")
    r = 1.0 / torch.sqrt(var + EPS32)
    rel = dvar / (var + EPS32)
    br = r * ((1.0 - rel).clamp(min=1e-300).rsqrt() - 1.0) + 2.01 * U * r
    check_bound(family, L.rstd, r, br, what + " rstd")
    check_bound(family, Lloc.local[0], m, bm, what + " triple mean")
    check_bound(family, Lloc.local[1], var * n, n * dvar + 1.01 * U * var * n, what + " triple M2")
    assert bool((Lloc.local[2] == float(n)).all()), what + " triple count"
    unb, dunb = (var * n / (n - 1), dvar * n / (n - 1)) if n > 1 else (var, dvar)
    keep = 1.0 - MOM32
    for got, old, xv, dx, name in ((L.rm, rm0, m, bm, "running_mean"),
                                   (L.rv, rv0, unb, dunb + 1.01 * U * unb, "running_var")):
        old = old.double()
        check_bound(family, got, keep * old + MOM32 * xv,
                    MOM32 * dx + 3.0 * U * ((keep * old).abs() + (MOM32 * xv).abs()), f"{what} {name}")


def running0(N, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn(N, device=DEV, generator=g), torch.rand(N, device=DEV, generator=g) + 0.5


def launch_checked(x, w, b, rows_dev, what):
    """Training call (running statistics, num_batches_tracked 41 -> 42) and SyncBN call, each three
    times; -> (L, Lloc, rm0, rv0)."""
    N = w.shape[0]
    rm0, rv0 = running0(N, x.shape[0] + N)

    def train():
        L = direct(x, w, b, rows_dev, running=(rm0.clone(), rv0.clone(),
                                              torch.tensor(41, dtype=torch.int64, device=DEV)))
        assert int(L.nbt) == 42, what + ": num_batches_tracked"
        return L

    def syncbn():
        nbt = torch.tensor(5, dtype=torch.int64, device=DEV)
        L = direct(x, w, b, rows_dev, local=True, running=(None, None, nbt))
        assert int(nbt) == 6, what + ": num_batches_tracked (triple)"
        return L

    L = three(train, what)
    Lloc = three(syncbn, what + " triple")
    assert np.array_equal(L.part.view(np.int32), Lloc.part.view(np.int32)), what + ": partials differ"
    return L, Lloc, rm0, rv0


def valid_rows(rows_dev, M):
    return M if rows_dev is None else min(max(int(rows_dev), 0), M)


def check_training(x, w, b, rows_dev, what, y_rows=None, exact_y=False, family="GEMM"):
    """Everything one training launch produces, against float64: y over the first ``y_rows`` rows
    (all by default), the CTA partials, the restated combine and finalize, the statistics, running
    statistics and the SyncBN triple."""
    M, K = x.shape
    N = w.shape[0]
    g = ls_geom(M)
    n = valid_rows(rows_dev, M)
    L, Lloc, rm0, rv0 = launch_checked(x, w, b, rows_dev, what)
    y_rows = M if y_rows is None else y_rows
    y64, mag = gemm_ref(x, w, b, y_rows)
    if exact_y:
        assert same_bits(L.y[:y_rows], y64.float()), f"{what}: y not exact " \
            f"({int((L.y[:y_rows].double() != y64).sum())} elements differ)"
    else:
        check_bound(family, L.y[:y_rows], y64, gemm_bound(K, mag, y64), what + " y")
    del y64, mag
    v = VRef(L.y, b, n)
    check_partials(L, v, g, N, what)
    check_finalize(L, g, N, b, n, what)
    check_finalize(Lloc, g, N, b, n, what + " triple")
    check_stats(L, Lloc, v, b, rm0, rv0, what)
    return L._replace(local=Lloc.local)


def check_exact_stats(x, w, b, rows_dev, what):
    """x, w in {-1, 0, 1}, K = 32, integer b: every fp32 partial is exact (checked), so the CTA
    partials are the integer sums and mean / rstd are within 1 ulp of float64 from them."""
    M, K = x.shape
    N = w.shape[0]
    g = ls_geom(M)
    n = valid_rows(rows_dev, M)
    L, Lloc, _rm0, _rv0 = launch_checked(x, w, b, rows_dev, what)
    v = (x[:n].double() @ w.double().t())                   # exact: integers below 2^53
    assert float(v.abs().sum(0).max()) < 2 ** 24 and float((v * v).sum(0).max()) < 2 ** 24
    y64 = v + (b.double() if b is not None else 0.0)
    assert same_bits(L.y[:n], y64.float()), what + ": y not exact"
    cta = (torch.arange(n, device=DEV) // BM) % g.grid
    want = torch.zeros((g.grid, 2 * N), dtype=torch.float64, device=DEV)
    want.index_add_(0, cta, torch.cat([v, v * v], 1))
    got = torch.from_numpy(L.part).to(DEV).double()
    assert torch.equal(got, want), f"{what}: CTA partials differ from the integer sums " \
        f"(largest difference {float((got - want).abs().max())})"
    check_finalize(L, g, N, b, n, what)
    if n:
        S, Q = want.sum(0)[:N].cpu().numpy(), want.sum(0)[N:].cpu().numpy()
        bb = b.double().cpu().numpy() if b is not None else 0.0
        m = S / n + bb
        var = (Q - S * S / n) / n
        assert ulps(L.mean.cpu().numpy(), m.astype(np.float32)).max() <= 1, what + " mean"
        assert ulps(L.rstd.cpu().numpy(), (1.0 / np.sqrt(var + EPS32)).astype(np.float32)).max() <= 1, \
            what + " rstd"
        assert ulps(Lloc.local[1].cpu().numpy(), (var * n).astype(np.float32)).max() <= 1, what + " M2"


# ------------------------------------------------------------------------------ data
def gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def random_operands(M, K, N, seed, bias=True):
    """x = N(0.3, 1.5^2); W rows scaled by 10^U(-2, 2), so small channels sit beside large ones."""
    g = gen(seed)
    x = torch.randn(M, K, device=DEV, generator=g) * 1.5 + 0.3
    scale = 10.0 ** (torch.rand(N, 1, device=DEV, generator=g) * 4 - 2)
    w = torch.randn(N, K, device=DEV, generator=g) / K ** 0.5 * scale
    b = torch.randn(N, device=DEV, generator=g) if bias else None
    return x, w, b


def int_operands(M, K, N, seed, lim):
    g = gen(seed)

    def ri(*shape):
        return torch.randint(-lim, lim + 1, shape, device=DEV, generator=g).float()
    return ri(M, K), ri(N, K), ri(N)


# ------------------------------------------------------------------------------ training: splits
SPLIT_CASES = [(N, M) for N in (128, 256, 384) for M in SPLITS]


@gpu
@pytest.mark.parametrize("N,M", SPLIT_CASES)
def test_linear_stats_split_vs_fp64(N, M):
    """Every grid / ticket split of the table at every width: random data with and without a bias
    (K = 96: below NT = 1's ring of 5 stages, equal to the 3 of NT = 2, 3), integers in [-4, 4]
    (y exact), and {-1, 0, 1} at K = 32 (statistics exact)."""
    assert split_of(M) == SPLITS[M]
    for bias in (True, False):
        x, w, b = random_operands(M, 96, N, M + N + bias, bias)
        check_training(x, w, b, None, f"N={N} M={M} bias={bias}")
    x, w, b = int_operands(M, 96, N, M * N, 4)
    check_training(x, w, b, None, f"N={N} M={M} int", exact_y=True)
    x, w, b = int_operands(M, 32, N, M + 7 * N, 1)
    check_exact_stats(x, w, b, None, f"N={N} M={M} exact statistics")


@gpu
@pytest.mark.parametrize("N", (128, 256, 384))
@pytest.mark.parametrize("K", KS)
def test_linear_stats_k_vs_fp64(N, K):
    """K = 32 .. 4096 (kblocks 1, 2, 3, 5, 6, 12, 128: below, equal to and above the ring's stage
    count of every width) at 148 CTAs with 2 tiles for CTA 0, so the ring also wraps across tiles;
    random data with a bias and integer data (y exact)."""
    M = 18945
    kb = K // BK
    assert split_of(M) == SPLITS[M] and kb in (1, 2, 3, 5, 6, 12, 128)
    x, w, b = random_operands(M, K, N, K + N)
    check_training(x, w, b, None, f"N={N} K={K}")
    x, w, b = int_operands(M, K, N, K * N, 4)
    assert 16 * K + 4 < 2 ** 24
    check_training(x, w, b, None, f"N={N} K={K} int", exact_y=True)


@gpu
@pytest.mark.parametrize("N", (128, 384))
@pytest.mark.parametrize("r", list(LAST_ROWS))
def test_linear_stats_last_tile(N, r):
    """A last tile that ends in each of the four epilogue warp quarters (r = M % 128), with grids of
    one group, two groups and 148 CTAs."""
    for tiles in (3, 20, 160):
        M = (tiles - 1) * BM + r
        assert ls_geom(M).tiles == tiles and (M - 1) % BM // 32 == LAST_ROWS[r]
        x, w, b = random_operands(M, 64, N, M + N)
        check_training(x, w, b, None, f"N={N} M={M}")
        x, w, b = int_operands(M, 64, N, M * N, 4)
        check_training(x, w, b, None, f"N={N} M={M} int", exact_y=True)


@gpu
@pytest.mark.parametrize("M,K,N", [(1, 32, 128), (127, 128, 128), (128, 128, 128), (129, 384, 128),
                                   (4097, 128, 128), (70001, 384, 128), (300000, 128, 128),
                                   (20000, 64, 128), (70001, 384, 384), (4097, 384, 384),
                                   (33333, 256, 256), (257, 128, 384), (9000, 256, 128)])
@pytest.mark.parametrize("has_bias", [True, False])
def test_linear_stats_matches_torch_and_its_own_output(ops, M, K, N, has_bias):
    """y against float64 torch and the statistics against the kernel's own y, within the bounds of
    the module docstring, at the shapes of the tuplewise MLP; the public op gives the bits of the
    direct launch."""
    x, w, b = random_operands(M, K, N, M + K + N, has_bias)
    L = check_training(x, w, b, None, f"M={M} K={K} N={N} bias={has_bias}")
    y, mean, rstd = ops.linear_stats(x, w, b, EPS, MOM, None, None, None, None, False)
    assert same_bits(y, L.y) and same_bits(mean, L.mean) and same_bits(rstd, L.rstd)


def chan_reference(g64):
    """Chan's merge of (mean, M2, count) triples in rank order, float64 (as bn_sync_finalize)."""
    n = torch.zeros_like(g64[0, 0])
    m, m2 = n.clone(), n.clone()
    for r in range(g64.shape[0]):
        nb, mb, m2b = g64[r, 2], g64[r, 0], g64[r, 1]
        tot = n + nb
        delta = mb - m
        m = m + delta * (nb / tot)
        m2 = m2 + m2b + delta * delta * (n * nb / tot)
        n = tot
    return n, m, m2


@gpu
def test_linear_stats_pad_rows_and_syncbn_triples(ops):
    """Junk (x 50) pad rows past rows_dev on a capacity-padded batch: y of every row, statistics of
    the valid rows against float64, and the valid rows equal the call on the unpadded batch bit for
    bit.  Rank-local triples of two row ranges, each against float64, merged by bn_sync_finalize
    within 2u of Chan's merge of those triples in float64."""
    M, cap, K, N = 5000, 5200, 384, 128
    x, w, b = random_operands(cap, K, N, 9)
    x[M:] *= 50.0
    rows_dev = torch.tensor([M], dtype=torch.int32, device=DEV)
    Lp = check_training(x, w, b, rows_dev, "pad rows")
    y = ops.linear_stats(x[:M].contiguous(), w, b, EPS, MOM, None, None, None, None, False)[0]
    assert same_bits(Lp.y[:M], y), "valid rows differ from the unpadded call"
    trip = []
    for lo, hi in ((0, 1700), (1700, M)):
        part = x[lo:hi].contiguous()
        L = check_training(part, w, b, None, f"rows {lo}..{hi}")
        _yy, local, _e = ops.linear_stats(part, w, b, EPS, MOM, None, None, None, None, True)
        assert local.shape == (3, N) and same_bits(local, L.local)
        trip.append(local)
    g = torch.stack(trip)
    mean, rstd, inv_n = ops.bn_sync_finalize(g, EPS, MOM, None, None)
    n, m, m2 = chan_reference(g.double())
    tiny = 1e-13 * g[:, 0].double().abs().max()
    check_bound("SyncBN merge", mean, m, 2 * U * m.abs() + tiny, "merged mean")
    r = 1.0 / torch.sqrt(m2 / n + EPS32)
    check_bound("SyncBN merge", rstd, r, 2 * U * r + r * 1e-13, "merged rstd")
    assert abs(float(inv_n) * M - 1.0) <= 2 * U


# ------------------------------------------------------------------------------ training: rows_dev
ROWS_DEV = {"in_quarter": (5000, lambda M: 5 * BM + 40), "tile_boundary": (5000, lambda M: 7 * BM),
            "below_128_at_148_ctas": (2 * 18944, lambda M: 100), "above_M": (3001, lambda M: M + 1000),
            "negative": (3001, lambda M: -5), "zero": (3001, lambda M: 0), "all": (3001, lambda M: M)}


@gpu
@pytest.mark.parametrize("N", (128, 384))
@pytest.mark.parametrize("case", list(ROWS_DEV))
def test_linear_stats_rows_dev(N, case):
    """Device row counts: n inside a warp quarter, on a tile boundary, below 128 while M spans all
    148 CTAs, above M (clamped), negative and 0 (no valid row).  The pad rows of x hold NaN and
    Inf: the statistics are finite and bit-identical to the same call with zeros there."""
    M, f = ROWS_DEV[case]
    nd = f(M)
    n = valid_rows(nd, M)
    rows_dev = torch.tensor([nd], dtype=torch.int32, device=DEV)
    x, w, b = random_operands(M, 128, N, M + N)
    x[n:] = 0.0
    Lz = check_training(x, w, b, rows_dev, f"N={N} {case} zero pads")
    xi, wi, bi = int_operands(M, 32, N, n + N, 1)
    check_exact_stats(xi, wi, bi, rows_dev, f"N={N} {case} exact statistics")
    if n < M:
        x[n:] = torch.where(torch.arange(x[n:].numel(), device=DEV).view(M - n, -1) % 3 == 0, NAN,
                            torch.where(torch.arange(M - n, device=DEV)[:, None] % 2 == 0, INF, -INF))
        Ln = check_training(x, w, b, rows_dev, f"N={N} {case} NaN pads", y_rows=n)
        for f_ in ("mean", "rstd", "rm", "rv"):
            got = getattr(Ln, f_)
            assert bool(torch.isfinite(got).all()), f"{case}: {f_} not finite"
            assert same_bits(got, getattr(Lz, f_)), f"{case}: {f_} depends on the pad rows"
        assert np.array_equal(Ln.part.view(np.int32), Lz.part.view(np.int32)), case + ": partials"


# ------------------------------------------------------------------------------ training: families
@gpu
@pytest.mark.parametrize("N,K", [(128, 384), (128, 256), (384, 384)])
def test_linear_stats_large_mean_vs_fp64(N, K):
    """Post-SiLU inputs (positive mean) and weights with a positive mean per channel at ZINC scale:
    |mean| / std of the channels is 10 to 30 while the bias (the kernel's only shift) is small, so
    the cancellation term of the variance bound carries the check."""
    M = 230147
    g = gen(N + K)
    x = torch.nn.functional.silu(torch.randn(M, K, device=DEV, generator=g) + 2.0)
    mu = torch.rand(N, 1, device=DEV, generator=g) + 0.4
    w = (torch.randn(N, K, device=DEV, generator=g) + mu) / K ** 0.5
    b = torch.randn(N, device=DEV, generator=g) * 0.1
    L = check_training(x, w, b, None, f"large mean N={N} K={K}")
    d = L.y.double() - b.double()
    ratio = d.mean(0).abs() / d.std(0)
    assert float(ratio.min()) >= 8 and float(ratio.max()) <= 35 and 10 <= float(ratio.median()) <= 30, \
        (float(ratio.min()), float(ratio.median()), float(ratio.max()))
    var = d.var(0, unbiased=False)
    assert float(((d * d).mean(0) / var).median()) > 100         # Q / n is 100 x var and more


@gpu
def test_linear_stats_64bit_row_offsets():
    """M N > 2^31 outputs (N = 128, K = 32, 2^24 + 300 rows, ~11 GB): x is zero except the first
    rows, the rows around the 2^31-element boundary, the last tile and 4096 scattered rows, all in
    {-1, 0, 1}, so every output and every statistic is exact."""
    M, K, N = 2 ** 24 + 300, 32, 128
    assert M * N > 2 ** 31 and split_of(M)[:2] == (148, 10)
    g = gen(31)
    nz = torch.cat([torch.arange(0, 256), torch.arange(2 ** 24 - 256, 2 ** 24 + 256),
                    torch.arange(M - 172, M), torch.randint(0, M, (4096,), generator=torch.Generator().manual_seed(3))])
    nz = torch.unique(nz).to(DEV)
    x = torch.zeros(M, K, device=DEV)
    x[nz] = torch.randint(-1, 2, (nz.numel(), K), device=DEV, generator=g).float()
    w = torch.randint(-1, 2, (N, K), device=DEV, generator=g).float()
    b = torch.randint(-4, 5, (N,), device=DEV, generator=g).float()
    L = direct(x, w, b)
    v = x[nz].double() @ w.double().t()
    assert float(v.abs().sum(0).max()) < 2 ** 24 and float((v * v).sum(0).max()) < 2 ** 24
    assert same_bits(L.y[nz], (v + b.double()).float()), "y at the non-zero rows"
    zero_row = torch.ones(M, dtype=torch.bool, device=DEV)
    zero_row[nz] = False
    step = 1 << 20
    for s in range(0, M, step):
        yc, zc = L.y[s:s + step], zero_row[s:s + step]
        assert bool((yc[zc] == b).all()), f"y rows {s}..: not the bias"
    cta = (nz // BM) % 148
    want = torch.zeros((148, 2 * N), dtype=torch.float64, device=DEV).index_add_(0, cta, torch.cat([v, v * v], 1))
    assert torch.equal(torch.from_numpy(L.part).to(DEV).double(), want), "CTA partials"
    geo = ls_geom(M)
    check_finalize(L, geo, N, b, M, "64-bit offsets")
    S, Q = want.sum(0)[:N].cpu().numpy(), want.sum(0)[N:].cpu().numpy()
    var = (Q - S * S / M) / M
    assert ulps(L.mean.cpu().numpy(), (S / M + b.double().cpu().numpy()).astype(np.float32)).max() <= 1
    assert ulps(L.rstd.cpu().numpy(), (1.0 / np.sqrt(var + EPS32)).astype(np.float32)).max() <= 1


# ------------------------------------------------------------------------------ ordering
@gpu
def test_two_streams_and_interleaved_tickets(ops):
    """Grid 148 on one stream and grid 17 on another at the same time (ticket slots of their own),
    each equal to its solo result; then launches with 10, 1, 2 and 10 groups interleaved on one
    ticket buffer, each equal to its solo result with the tickets zero after every launch."""
    shapes = [(230147, 384, 128), (2049, 384, 128), (129, 64, 256), (18945, 96, 384)]
    inputs = [random_operands(M, K, N, M) for M, K, N in shapes]
    solo = [ops.linear_stats(x, w, b, EPS, MOM, None, None, None, None, False) for x, w, b in inputs[:2]]
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    s1.wait_stream(torch.cuda.current_stream())
    s2.wait_stream(torch.cuda.current_stream())
    for _ in range(3):
        with torch.cuda.stream(s1):
            a = ops.linear_stats(*inputs[0], EPS, MOM, None, None, None, None, False)
        with torch.cuda.stream(s2):
            c = ops.linear_stats(*inputs[1], EPS, MOM, None, None, None, None, False)
        torch.cuda.synchronize()
        for got, want in zip((a, c), solo):
            for t, u_ in zip(got, want):
                assert same_bits(t, u_), "a launch beside another stream's differs from its solo run"
    alone = [direct(*xwb) for xwb in inputs]
    tickets = torch.zeros(64, dtype=torch.int32, device=DEV)
    for i in (0, 1, 2, 3, 0, 2, 1, 0):
        M, K, N = shapes[i]
        g = ls_geom(M)
        assert g.ngroups == (10, 2, 1, 10)[i]
        L = direct(*inputs[i], tickets=tickets)
        for f in ("y", "mean", "rstd"):
            assert same_bits(getattr(L, f), getattr(alone[i], f)), f"interleaved launch {i}: {f}"


@gpu
def test_graph_replay(ops):
    """A captured training call replayed 3 times: y, mean and rstd equal the eager calls bit for bit,
    and the running statistics after 3 replays equal those after 3 eager calls."""
    M, K, N = 75777, 384, 128
    x, w, b = random_operands(M, K, N, 5)
    rm0, rv0 = running0(N, 5)
    rm, rv, nbt = rm0.clone(), rv0.clone(), torch.zeros((), dtype=torch.int64, device=DEV)
    eager = [ops.linear_stats(x, w, b, EPS, MOM, rm, rv, None, nbt, False) for _ in range(3)]
    want_rm, want_rv = rm.clone(), rv.clone()
    grm, grv, gnbt = rm0.clone(), rv0.clone(), torch.zeros((), dtype=torch.int64, device=DEV)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.linear_stats(x, w, b, EPS, MOM, grm, grv, None, gnbt, False)     # warm-up
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = ops.linear_stats(x, w, b, EPS, MOM, grm, grv, None, gnbt, False)
    grm.copy_(rm0), grv.copy_(rv0), gnbt.zero_()
    for i in range(3):
        graph.replay()
        torch.cuda.synchronize()
        for t, e in zip(out, eager[i]):
            assert same_bits(t, e), f"replay {i}"
    assert same_bits(grm, want_rm) and same_bits(grv, want_rv) and int(gnbt) == 3


# ------------------------------------------------------------------------------ host rejections
def test_host_rejects_bad_arguments():
    """Both entry points refuse null, misaligned (x / w / residual 16 B, y / z 32 B), unsupported
    shapes, a short workspace and act outside 0..2 before any device call: fake addresses, no GPU.
    Every case but the last check of each entry point also carries a defect that a later check
    refuses (a zero workspace; a misaligned z), so no case can reach a launch even if an earlier
    check went missing; the workspace sizes come from the library's own query."""
    from pygho_b200 import _lib
    from pygho_b200._lib import KernelError
    lib = _lib.load()
    A = 1 << 24                              # fake addresses, 256-byte aligned, never dereferenced
    M, K, N = 5000, 384, 128

    def ws_of(m):
        return int(lib.pgh_linear_stats_ws_bytes(m))
    good = dict(x=A, M=M, K=K, w=2 * A, N=N, bias=3 * A, rows=None, y=4 * A, eps=EPS, mom=MOM,
                mean=5 * A, rstd=6 * A, rm=None, rv=None, local=None, nbt=None, ws=7 * A, nws=0,
                tickets=8 * A)
    bad = [({"x": None}, "null"), ({"w": None}, "null"), ({"y": None}, "null"), ({"ws": None}, "null"),
           ({"tickets": None}, "null"), ({"mean": None}, "null"), ({"rstd": None}, "null"),
           ({"N": 192}, "need N"), ({"N": 512}, "need N"), ({"N": 64}, "need N"),
           ({"K": 48}, "need N"), ({"K": 4128}, "need N"), ({"K": 0}, "need N"), ({"M": 0}, "need N"),
           ({"x": A + 8}, "16-byte"), ({"w": 2 * A + 4}, "16-byte"), ({"y": 4 * A + 16}, "32-byte"),
           ({"nws": ws_of(M) - 1}, "workspace"), ({"M": 230147, "nws": ws_of(2048)}, "workspace"),
           ({"N": 384, "nws": ws_of(M) - 4}, "workspace")]
    for change, msg in bad:
        a = {**good, **change}
        assert a["nws"] < ws_of(a["M"]), change                   # refused at the latest here
        with pytest.raises(KernelError, match=msg):
            _lib.call("pgh_linear_stats_f32", *a.values(), None)
    good = dict(x=A, M=M, K=K, w=2 * A, N=N, bias=None, gamma=None, beta=None, rm=3 * A, rv=4 * A,
                eps=EPS, act=1, res=5 * A, rows=None, z=6 * A + 16)
    bad = [({"x": None}, "null"), ({"w": None}, "null"), ({"rm": None}, "null"), ({"rv": None}, "null"),
           ({"z": None}, "null"), ({"N": 192}, "need N"), ({"K": 4128}, "need N"), ({"K": 100}, "need N"),
           ({"M": 0}, "need N"), ({"act": 3}, "act"), ({"act": -1}, "act"), ({"x": A + 4}, "16-byte"),
           ({"w": 2 * A + 8}, "16-byte"), ({"res": 5 * A + 8}, "16-byte"), ({}, "32-byte")]
    for change, msg in bad:
        a = {**good, **change}
        assert a["z"] is None or a["z"] % 32, change              # refused at the latest here
        with pytest.raises(KernelError, match=msg):
            _lib.call("pgh_linear_bn_eval_f32", *a.values(), None)


# ------------------------------------------------------------------------------ training dispatch
DISPATCH = [(4096, 256, 128, True, False, True), (4096, 384, 128, True, False, True),
            (230147, 384, 128, True, False, True), (4095, 384, 128, True, False, False),
            (4096, 128, 128, True, False, False), (4096, 384, 384, True, False, False),
            (4096, 384, 256, True, False, False), (4096, 384, 128, False, False, False),
            (4096, 128, 128, True, True, True), (4096, 384, 256, True, True, True),
            (4096, 384, 384, True, True, True), (4095, 128, 128, True, True, False),
            (4096, 384, 384, False, True, False), (4096, 96, 192, True, True, False)]


@gpu
@pytest.mark.parametrize("M,K,N,tf32,wide,fused", DISPATCH)
def test_training_dispatch(M, K, N, tf32, wide, fused, monkeypatch):
    """LinearBNAct calls pgh_linear_stats_f32 exactly where linear_stats_ok says: N = 128, K >= 256,
    M >= 4096 with TF32 on; with _FUSED_GEMM_WIDE also K = 128 and N = 256, 384.  Elsewhere cuBLAS
    and the statistics kernel."""
    from pygho_b200 import ops
    monkeypatch.setattr(ops, "_FUSED_GEMM", True)
    monkeypatch.setattr(ops, "_FUSED_GEMM_WIDE", wide)
    x, w, b = random_operands(M, K, N, 1)
    gamma, beta = torch.ones(N, device=DEV), torch.zeros(N, device=DEV)
    rm, rv = torch.zeros(N, device=DEV), torch.ones(N, device=DEV)
    names = []
    real = ops.call

    def spy(name, *args):
        names.append(name)
        return real(name, *args)
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = tf32
    try:
        assert ops.linear_stats_ok(x, w) == fused
        monkeypatch.setattr(ops, "call", spy)
        ops.LinearBNAct.apply(x, w, b, gamma, beta, rm, rv, MOM, EPS, 1)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    assert ("pgh_linear_stats_f32" in names) == fused and ("pgh_bn_stats_f32" in names) != fused, names


# ------------------------------------------------------------------------------ the MLP block
def close(a, b, rtol):
    a, b = a.detach().double().cpu().numpy(), b.detach().double().cpu().numpy()
    assert a.shape == b.shape, (a.shape, b.shape)
    scale = max(1.0, float(np.abs(b).max()) if b.size else 1.0)
    err = float(np.abs(a - b).max(initial=0.0))
    assert err <= rtol * scale, (err, scale)


@gpu
@pytest.mark.parametrize("rows,cin", [(6000, 128), (33333, 384), (20000, 256)])
def test_mlp_block_on_fused_gemm_equals_cublas_path(rows, cin):
    """MLP (Linear -> BN -> SiLU) x 2 with the fused GEMM + statistics against the same block on
    cuBLAS TF32 + separate statistics pass: outputs and all gradients within TF32 tolerance."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        _mlp_block(rows, cin)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


def _mlp_block(rows, cin):
    import copy

    from pygho_b200 import ops
    from pygho_b200.honn.utils import MLP
    torch.manual_seed(rows)
    mlp = MLP(cin, 128, 2, True, norm="bn", act="silu", normparam=0.3).to(DEV)
    # hidden block cin -> cin and output block cin -> 128: both on the fused GEMM
    ref = copy.deepcopy(mlp)
    x = torch.randn(rows, cin, device=DEV)
    w = torch.randn(rows, 128, device=DEV)
    xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    last = [m for m in mlp.modules() if isinstance(m, torch.nn.Linear)][-1]
    wide, ops._FUSED_GEMM_WIDE = ops._FUSED_GEMM_WIDE, True    # cover N = 256 / 384 and K = 128 too
    try:
        assert ops.linear_stats_ok(torch.empty(rows, last.in_features, device=DEV), last.weight)
        (mlp(xa) * w).sum().backward()
    finally:
        ops._FUSED_GEMM_WIDE = wide
    ops.set_fused_linear_stats(False)
    try:
        (ref(xb) * w).sum().backward()
    finally:
        ops.set_fused_linear_stats(True)
    close(xa.grad, xb.grad, 5e-3)
    for (k, p), (_, q) in zip(mlp.named_parameters(), ref.named_parameters()):
        if k.endswith("bias") and "norm" not in k:
            continue
        close(p.grad, q.grad, 5e-3)
    for (k, p), (_, q) in zip(mlp.named_buffers(), ref.named_buffers()):
        close(p.float(), q.float(), 2e-3)
