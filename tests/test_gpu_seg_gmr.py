"""seg_gmr (pygho_b200/csrc/seg_gmr.cu) against a float64 reference, at every work split its
kernels use.

    out[r] = aggr_{t in seg(r)} a[c_t] * s[c_t] * b[d_t]

The reference is computed on the CPU from the plan itself ``(rowptr, c, d, a_scale)``, never from
the kernels' own groupings:

* sum and mean in float64, compared per element with
  ``|got - ref| <= 1.01 * (len + 3) * 2^-24 * sum_{t in seg(r)} |a*s*b|``  (mean: divided by len)
  plus ``|acc_src|`` when the kernel adds into a preset output.  ``len`` is the row's own segment
  length: recursive float32 summation of ``len`` terms makes ``len - 1`` roundings, each term
  carries at most two more (``a*s``, ``*b``; in the mean backward the third is ``fl(1/len)``), and
  the mean division or the accumulate addition is one more, so ``len + 3`` roundings of relative
  size <= 2^-24 bound the error; 1.01 covers the second-order term (``len * 2^-24 <= 2^-7`` here).
  A row without entries has bound 0: it must be exactly 0 (or exactly the preset value).
* max and min over the float32 products rounded in the kernels' order ``fl(fl(a*s)*b)``, compared
  exactly; empty rows give 0.
* gradients of max and min follow torch's ``scatter_reduce`` rule: the gradient of a row is split
  evenly among the entries whose product equals the output, and an output of exactly 0 also
  counts the (zero) initial value as a tie.

Every launch asserts which kernel and work split it reaches (``geometry`` below) and runs twice
with equal bits.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda"
U = 2.0 ** -24
AGGRS = ("sum", "mean", "max", "min")
CODE = {"sum": 0, "mean": 1, "max": 2, "min": 3}
SENTINEL = 7.0


@pytest.fixture(scope="module")
def ops():
    import pygho_b200.ops  # noqa: F401  (registers torch.ops.pygho_b200)
    return torch.ops.pygho_b200


# ------------------------------------------------------------------------------ geometry
# Restates the launch rules of pygho_b200/csrc/seg_gmr.cu: geometry() (row-wise lpr / vec),
# launch_gmr() (which kernel), launch_lean() and launch_ring() (rows per warp).  kSMs and
# kThreads come from common.cuh / seg_gmr.cu.  Keep this in step with the C source.
K_SMS, K_THREADS, K_MAX_RW = 148, 256, 16
LEAN_ROWS_PER_RW = K_SMS * 4 * (K_THREADS // 32)       # launch_lean: rw <= n_rows / 4736
RING_ENTRIES_PER_WARP, RING_MAX_RW = 16, 31


def geometry(n_rows, n_entries, dense, lean, aligned=True):
    """(kernel, rw or lpr, vec) of one launch.  ``lean``: two operands or a fused epilogue."""
    vec = 4 if aligned and dense % 4 == 0 else 1
    if vec == 4 and dense % 128 == 0:
        have_avg = n_entries > 0 and n_rows > 0
        avg = max(n_entries / n_rows, 0.5) if have_avg else 0.0
        if lean:
            rw = K_MAX_RW
            if have_avg:
                rw = min(int(32.0 / avg), n_rows // LEAN_ROWS_PER_RW)
                rw = min(max(rw, 1), K_MAX_RW)
            return ("lean", rw, 4)
        rw = int(RING_ENTRIES_PER_WARP / avg) if have_avg else RING_ENTRIES_PER_WARP
        return ("ring", min(max(rw, 1), RING_MAX_RW), 4)
    units = dense // vec
    lpr = 1
    while lpr < 32 and lpr < units:
        lpr <<= 1
    return ("rowwise", lpr, vec)


# ------------------------------------------------------------------------------ plans
# Row lengths that put a warp's entry stream across a 32-entry chunk exactly at row boundaries
# (32 | 31 1 | 63 | 64 | 32 after empty rows) and inside rows (33, 63, 64, 65), with empty rows
# sitting on a chunk boundary.  Odd lengths make the ring's entry pairs straddle rows.
CHUNK_ROWS = [32, 31, 1, 33, 63, 0, 64, 65, 0, 0, 32, 1, 31]
HUB = 1 << 17


def edge_rows(rw):
    """Whole warps of ``rw`` rows: a warp whose first and last rows are empty, a warp of empty
    rows, then CHUNK_ROWS starting on a warp boundary (padded to a whole warp)."""
    rows = [0] + [3] * (rw - 2) + [0] if rw >= 2 else [0]
    rows += [0] * rw
    rows += CHUNK_ROWS
    rows += [2] * (-len(rows) % rw)
    return rows


class Plan:
    """A CSR plan built from explicit row lengths: edge warps for each rows-per-warp in
    ``rws`` (each section starts on a warp boundary of that geometry), Poisson(lam) filler,
    optionally one hub row between empty rows, and a last row that is empty.  ``c`` and ``d``
    are unsorted with repeats; rows of 60+ entries draw ``c`` from 8 rows only (many exact
    repeats inside one row).  ``identity``: c = None (operand A has one row per entry)."""

    def __init__(self, n_rows, lam, rws, seed, hub=False, identity=False, n_a=3000, n_b=2000):
        rng = np.random.default_rng(seed)
        lens = rng.poisson(lam, n_rows).astype(np.int64)
        pos = 0
        for rw in rws:
            pos = -(-pos // rw) * rw
            e = edge_rows(rw)
            lens[pos:pos + len(e)] = e
            pos += len(e)
        if hub:
            pos = -(-pos // 16) * 16 + 5            # inside a warp of 16 rows
            lens[pos - 2:pos + 3] = [0, 0, HUB, 0, 0]
        lens[-1] = 0
        self.n_rows, self.lens = n_rows, lens
        self.rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        self.T = T = int(self.rowptr[-1])
        self.row_of = np.repeat(np.arange(n_rows), lens)
        self.identity = identity
        self.n_a = T if identity else n_a
        self.n_b = n_b
        self.c = None if identity else rng.integers(0, n_a, T)
        if not identity:
            long_rows = np.repeat(lens >= 60, lens)
            self.c[long_rows] = rng.integers(0, 8, int(long_rows.sum()))
        self.d = rng.integers(0, n_b, T)
        self.ci = np.arange(T) if identity else self.c

    def dev(self):
        i32 = lambda x: None if x is None else torch.from_numpy(x.astype(np.int32)).to(DEV)  # noqa: E731
        return i32(self.rowptr), i32(self.c), i32(self.d)


# name -> (Plan arguments, dense, lean rw, ring rw).  n_rows is never a multiple of rw (the last
# warp is short); lean rw 2/4/8 come from the small-grid cap n_rows // 4736, rw 16 needs
# n_rows >= 75776 and avg <= 2, ring rw 31 needs avg <= 0.5, ring rw 1 needs avg > 8.
STREAM_PLANS = {
    "lean16_ring16": (dict(n_rows=75785, lam=0.95, rws=(16,), seed=1), 128, 16, 16),
    "lean16_ring31": (dict(n_rows=75785, lam=0.3, rws=(16, 31), seed=2), 128, 16, 31),
    "hub_lean16_ring8": (dict(n_rows=75785, lam=0.1, rws=(16, 8), seed=3, hub=True), 128, 16, 8),
    "lean8": (dict(n_rows=37893, lam=0.7, rws=(8, 22), seed=4), 256, 8, 22),
    "lean4_identity": (dict(n_rows=18947, lam=1.5, rws=(4, 10), seed=5, identity=True), 512, 4, 10),
    "lean2": (dict(n_rows=9473, lam=0.6, rws=(2, 23), seed=6), 1024, 2, 23),
    "lean1_ring1": (dict(n_rows=1000, lam=10.0, rws=(1,), seed=7), 1024, 1, 1),
    "ring2": (dict(n_rows=2001, lam=6.5, rws=(2,), seed=8), 384, 1, 2),
}

_PLANS = {}


def stream_plan(name):
    if name not in _PLANS:
        _PLANS.clear()                               # keep one plan's arrays alive at a time
        _PLANS[name] = Plan(**STREAM_PLANS[name][0])
    return _PLANS[name]


# ------------------------------------------------------------------------------ reference
def seg_reduce(how, row, n, x):
    """Reduce the entries ``x`` (numpy, one per ``row`` id) into ``n`` rows on the CPU: "sum",
    "amax" or "amin"; rows without entries are 0."""
    x, row = torch.from_numpy(np.ascontiguousarray(x)), torch.from_numpy(row)
    out = torch.zeros((n,) + tuple(x.shape[1:]), dtype=x.dtype)
    if how == "sum":
        return out.index_add_(0, row, x)
    return out.scatter_reduce_(0, row.view(-1, 1).expand_as(x), x, how, include_self=False)


class Reference:
    """float64 sums and magnitudes and float32 extrema of one operand form over a plan (CPU
    tensors)."""

    def __init__(self, plan, a, b, s):
        ci, row, n = plan.ci, plan.row_of, plan.n_rows
        p32 = a[ci]
        p64 = p32.astype(np.float64)
        if s is not None:
            p32 = p32 * s[ci, None]                  # fl(a*s)
            p64 = p64 * s[ci, None]
        if b is not None:
            p32 = p32 * b[plan.d]                    # fl(fl(a*s)*b)
            p64 = p64 * b[plan.d]
        self.lens = torch.from_numpy(plan.lens)
        self.sum = seg_reduce("sum", row, n, p64)
        self.mag = seg_reduce("sum", row, n, np.abs(p64))
        self.max = seg_reduce("amax", row, n, p32)
        self.min = seg_reduce("amin", row, n, p32)

    def want(self, aggr):
        """(value, magnitude or None for the exact aggregations)."""
        if aggr == "sum":
            return self.sum, self.mag
        if aggr == "mean":
            n = self.lens.clamp(min=1).double().unsqueeze(1)
            return self.sum / n, self.mag / n
        return getattr(self, aggr), None


def assert_sum_close(got, want, mag, lens, what):
    """Per-element bound of the module docstring; compared on ``got``'s device."""
    want, mag, lens = want.to(got.device), mag.to(got.device), lens.to(got.device)
    got = got.double()
    bound = mag * (1.01 * U * (lens.double() + 3)).unsqueeze(1)
    bad = ~((got - want).abs() <= bound)             # NaN counts as bad
    if bool(bad.any()):
        r, col = (int(i) for i in bad.nonzero()[0])
        raise AssertionError(
            f"{what}: {int(bad.sum())} elements outside the bound; first at row {r} "
            f"(len {int(lens[r])}) col {col}: got {float(got[r, col])!r} "
            f"want {float(want[r, col])!r} bound {float(bound[r, col]):.3g}")


def assert_exact(got, want, what):
    want = want.to(got.device)
    bad = got != want                                # +0 == -0: maxNum leaves the zero sign open
    if bool(bad.any()):
        r, col = (int(i) for i in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} elements differ; first at row {r} col {col}:"
                             f" got {float(got[r, col])!r} want {float(want[r, col])!r}")


def check(got, ref_val, ref_mag, lens, what):
    if ref_mag is None:
        assert_exact(got, ref_val, what)
    else:
        assert_sum_close(got, ref_val, ref_mag, lens, what)


def same_bits(x, y):
    return torch.equal(x.contiguous().view(torch.int32), y.contiguous().view(torch.int32))


# ------------------------------------------------------------------------------ launch helpers
def wide(x, rng):
    """``x`` as a 16-byte aligned column slice of a wider device buffer (leading dimension >
    dense) whose other columns hold noise."""
    rows, dense = x.shape
    ld = 4 + -(-dense // 4) * 4 + 4
    buf = rng.standard_normal((rows, ld), dtype=np.float32)
    buf[:, 4:4 + dense] = x
    return torch.from_numpy(buf).to(DEV)[:, 4:4 + dense]


def out_slice(n_rows, dense):
    ld = 4 + -(-dense // 4) * 4 + 4
    buf = torch.full((n_rows, ld), SENTINEL, device=DEV)
    return buf, buf[:, 4:4 + dense]


def assert_outside_untouched(buf, dense):
    assert bool((buf[:, :4] == SENTINEL).all()) and bool((buf[:, 4 + dense:] == SENTINEL).all()), \
        "seg_gmr wrote outside its output columns"


def run_forms(ops, plan, dense, a, b, s, expect, seed):
    """Every aggregation of the four operand forms (one operand / two operands, each with and
    without a_scale) through ``seg_gmr_out`` with strided operands and a strided output, twice
    (equal bits), then sum and mean once more accumulating into a preset output."""
    rng = np.random.default_rng(seed)
    rowptr, c, d = plan.dev()
    a_d, b_d, s_d = wide(a, rng), wide(b, rng), torch.from_numpy(s).to(DEV)
    for two in (False, True):
        geo = geometry(plan.n_rows, plan.T, dense, lean=two)
        assert geo == expect(two), (geo, expect(two))
        for scaled in (False, True):
            ref = Reference(plan, a, b if two else None, s if scaled else None)
            args = (a_d, c, s_d if scaled else None, b_d if two else None, d if two else None,
                    rowptr, plan.n_rows)
            for aggr in AGGRS:
                what = f"{geo} {aggr} two={two} scale={scaled}"
                buf1, o1 = out_slice(plan.n_rows, dense)
                buf2, o2 = out_slice(plan.n_rows, dense)
                ops.seg_gmr_out(*args, CODE[aggr], o1, False)
                ops.seg_gmr_out(*args, CODE[aggr], o2, False)
                assert same_bits(o1, o2), f"{what}: two runs differ"
                assert_outside_untouched(buf1, dense)
                val, mag = ref.want(aggr)
                check(o1, val, mag, ref.lens, what)
                if aggr in ("sum", "mean"):
                    preset = torch.from_numpy(
                        rng.standard_normal((plan.n_rows, dense), dtype=np.float32)).to(DEV)
                    o1.copy_(preset)
                    ops.seg_gmr_out(*args, CODE[aggr], o1, True)
                    assert_outside_untouched(buf1, dense)
                    preset = preset.double()
                    assert_sum_close(o1, preset + val.to(DEV), mag.to(DEV) + preset.abs(),
                                     ref.lens, what + " accumulate")
                del buf1, buf2, o1, o2


def operands(plan, dense, seed, kind="randn"):
    rng = np.random.default_rng(seed)
    if kind == "randn":
        a = rng.standard_normal((plan.n_a, dense), dtype=np.float32)
        b = rng.standard_normal((plan.n_b, dense), dtype=np.float32)
    elif kind == "ints":                             # exact ties and products of exactly 0
        a = rng.integers(-2, 3, (plan.n_a, dense)).astype(np.float32)
        b = rng.integers(-2, 3, (plan.n_b, dense)).astype(np.float32)
    else:                                            # "negative": every product is < 0
        a = -rng.integers(1, 4, (plan.n_a, dense)).astype(np.float32)
        b = rng.integers(1, 4, (plan.n_b, dense)).astype(np.float32)
    s = rng.uniform(0.25, 2.0, plan.n_a).astype(np.float32)
    return a, b, s


# ------------------------------------------------------------------------------ forward
@pytest.mark.parametrize("name", list(STREAM_PLANS))
def test_stream_kernels_vs_fp64(ops, name):
    """Lean (two operands) and ring (one operand) kernels at rows-per-warp 1..31 and widths
    128..1024: every aggregation, with and without a_scale, strided operands and output,
    accumulate, determinism."""
    _, dense, lean_rw, ring_rw = STREAM_PLANS[name]
    plan = stream_plan(name)
    for rw in (lean_rw, ring_rw):
        assert rw == 1 or plan.n_rows % rw, "the last warp must be short"
    a, b, s = operands(plan, dense, 11)
    expect = lambda two: ("lean", lean_rw, 4) if two else ("ring", ring_rw, 4)  # noqa: E731
    run_forms(ops, plan, dense, a, b, s, expect, 12)


# row-wise widths -> expected (lpr, vec); 24 is the one width with lpr 8 at vec 4
ROWWISE = {1: (1, 1), 3: (4, 1), 4: (1, 4), 8: (2, 4), 12: (4, 4), 24: (8, 4), 33: (32, 1),
           64: (16, 4), 124: (32, 4), 129: (32, 1), 132: (32, 4)}


def rowwise_plan(dense, seed):
    rows_per_warp = 32 // ROWWISE[dense][0]
    return Plan(n_rows=3001, lam=3.0, rws=(rows_per_warp,), seed=seed, hub=False, n_a=700, n_b=500)


@pytest.mark.parametrize("dense", list(ROWWISE))
def test_rowwise_kernel_vs_fp64(ops, dense):
    """The row-wise kernel at every lanes-per-row it uses, vec 4 and vec 1."""
    plan = rowwise_plan(dense, 100 + dense)
    a, b, s = operands(plan, dense, 13 + dense)
    lpr, vec = ROWWISE[dense]
    run_forms(ops, plan, dense, a, b, s, lambda two: ("rowwise", lpr, vec), 14 + dense)


def test_rowwise_vec1_at_dense_128(ops):
    """dense % 128 == 0 with an operand that is not 16-byte aligned: the row-wise kernel with
    scalar loads.  The ops copy such an operand first, so this calls the C ABI directly."""
    from pygho_b200 import _lib
    dense = 128
    plan = Plan(n_rows=2001, lam=5.0, rws=(1,), seed=15, n_a=700, n_b=500)
    a, b, s = operands(plan, dense, 16)
    rowptr, c, d = plan.dev()
    store = torch.zeros(plan.n_a * dense + 4, device=DEV)
    a_d = store[1:1 + plan.n_a * dense].view(plan.n_a, dense)     # one float past an aligned base
    a_d.copy_(torch.from_numpy(a))
    assert a_d.data_ptr() % 16 == 4
    b_d, s_d = torch.from_numpy(b).to(DEV), torch.from_numpy(s).to(DEV)
    assert geometry(plan.n_rows, plan.T, dense, lean=True, aligned=False) == ("rowwise", 32, 1)
    stream = _lib.stream_ptr(torch.device(DEV))
    for two in (False, True):
        for scaled in (False, True):
            ref = Reference(plan, a, b if two else None, s if scaled else None)
            for aggr in AGGRS:
                outs = []
                for _ in range(2):
                    out = torch.empty(plan.n_rows, dense, device=DEV)
                    _lib.call("pgh_seg_gmr_ld_f32", a_d.data_ptr(), dense, c.data_ptr(),
                              s_d.data_ptr() if scaled else None, b_d.data_ptr() if two else None,
                              dense, d.data_ptr() if two else None, rowptr.data_ptr(), plan.n_rows,
                              plan.T, dense, CODE[aggr], 0, out.data_ptr(), dense, stream)
                    outs.append(out)
                assert same_bits(outs[0], outs[1])
                val, mag = ref.want(aggr)
                check(outs[0], val, mag, ref.lens, f"vec1 {aggr} two={two} scale={scaled}")


# ------------------------------------------------------------------------------ gradients
def grad_reference(plan, a, b, w, aggr, out):
    """float64 gradients of sum_r w[r] * out[r]: [(g_a, mag_a, len_a)] and, with two operands,
    (g_b, mag_b, len_b); ``len`` is each operand row's number of entries.  ``out`` is the
    (already checked) float32 forward result, whose ties decide the max / min gradients."""
    ci, di, rows = plan.ci, plan.d, plan.row_of
    if aggr in ("sum", "mean"):
        coef = w[rows].astype(np.float64)
        if aggr == "mean":
            coef /= plan.lens[rows][:, None]
    else:
        p = a[ci] * b[di] if b is not None else a[ci]
        eq = p == out[rows]
        ties = seg_reduce("sum", rows, plan.n_rows, eq.astype(np.int64)).numpy() + (out == 0)
        coef = np.where(eq, w[rows].astype(np.float64) / ties[rows], 0.0)
    groups = [(ci, plan.n_a, coef if b is None else coef * b[di])]
    if b is not None:
        groups.append((di, plan.n_b, coef * a[ci]))
    return [(seg_reduce("sum", key, n, terms), seg_reduce("sum", key, n, np.abs(terms)),
             torch.from_numpy(np.bincount(key, minlength=n))) for key, n, terms in groups]


GRAD_CASES = {"hub_lean16_ring8": 128, "lean1_ring1": 1024, 3: 3, 33: 33, 132: 132}


@pytest.mark.parametrize("kind", ["randn", "ints", "negative"])
@pytest.mark.parametrize("case", list(GRAD_CASES))
def test_gradients_vs_fp64(case, kind):
    """Both operand gradients through ops.seg_gmr's autograd for every aggregation: the sum /
    mean backward is seg_gmr again over the plan grouped by c and by d (the single-operand mean
    backward is the ring kernel with a_scale); max / min run the tie-splitting kernels.  ``ints``
    gives exact ties and outputs of exactly 0, ``negative`` all-negative products."""
    from pygho_b200 import plans as P
    from pygho_b200.ops import seg_gmr
    dense = GRAD_CASES[case]
    plan = stream_plan(case) if isinstance(case, str) else rowwise_plan(dense, 200 + dense)
    a, b, _ = operands(plan, dense, 17, kind)
    w = np.random.default_rng(18).standard_normal((plan.n_rows, dense), dtype=np.float32)
    acd = torch.from_numpy(np.stack([plan.row_of, plan.ci, plan.d])).to(DEV)
    tplan = P.plan_from_acd(acd, plan.n_rows, plan.n_a, plan.n_b)
    assert torch.equal(tplan.group("a").rowptr.cpu(), torch.from_numpy(plan.rowptr.astype(np.int32)))
    w_d = torch.from_numpy(w).to(DEV)
    for two in (True, False):
        for aggr in AGGRS:
            what = f"{case} {kind} {aggr} two={two}"
            runs = []
            for _ in range(2):
                a_d = torch.from_numpy(a).to(DEV).requires_grad_(True)
                b_d = torch.from_numpy(b).to(DEV).requires_grad_(True) if two else None
                out = seg_gmr(a_d, b_d, tplan, aggr)
                grads = torch.autograd.grad(out, [a_d] + ([b_d] if two else []), w_d)
                runs.append((out.detach(), grads))
            assert same_bits(runs[0][0], runs[1][0]), what
            assert all(same_bits(x, y) for x, y in zip(runs[0][1], runs[1][1])), what
            out = runs[0][0].cpu()
            ref = Reference(plan, a, b if two else None, None)
            val, mag = ref.want(aggr)
            check(runs[0][0], val, mag, ref.lens, what + " forward")
            gref = grad_reference(plan, a, b if two else None, w, aggr, out.numpy())
            for i, (g, (gv, gm, gl)) in enumerate(zip(runs[0][1], gref)):
                assert_sum_close(g, gv, gm, gl, what + (" grad b" if i else " grad a"))


# ------------------------------------------------------------------------------ fused epilogue
LEAN_FUSED = ["lean16_ring16", "lean8", "lean4_identity", "lean2", "lean1_ring1"]


@pytest.mark.parametrize("name", LEAN_FUSED)
def test_fused_epilogue_bitwise(ops, name):
    """seg_gmr_fused at lean rows-per-warp 16, 8, 4, 2, 1, laid out like the SSWL concatenated
    buffer [untouched | out | copy_dst]: out == fl(fl(add_src + red) + add_src2) bit for bit,
    with ``red`` from the plain launch on the same plan (itself checked against float64),
    copy_dst == copy_src bit for bit, and no write outside out and copy_dst."""
    _, dense, lean_rw, _ = STREAM_PLANS[name]
    plan = stream_plan(name)
    n = plan.n_rows
    assert geometry(n, plan.T, dense, lean=True) == ("lean", lean_rw, 4)
    rng = np.random.default_rng(19)
    a, b, s = operands(plan, dense, 20)
    rowptr, c, d = plan.dev()
    a_d, b_d, s_d = wide(a, rng), wide(b, rng), torch.from_numpy(s).to(DEV)
    src = torch.from_numpy(rng.standard_normal((n, 3 * dense), dtype=np.float32)).to(DEV)
    src_bits = src.clone()
    add_src, add_src2, copy_src = src[:, :dense], src[:, dense:2 * dense], src[:, 2 * dense:]
    variants = [dict(add=True, add2=False, copy=False), dict(add=True, add2=True, copy=False),
                dict(add=False, add2=False, copy=True), dict(add=True, add2=True, copy=True),
                dict(add=False, add2=False, copy=False)]
    for scaled in (False, True):
        ref = Reference(plan, a, b, s if scaled else None)
        for aggr in ("sum", "mean"):
            args = (a_d, c, s_d if scaled else None, b_d, d, rowptr, n, CODE[aggr])
            red = ops.seg_gmr(*args)
            val, mag = ref.want(aggr)
            assert_sum_close(red, val, mag, ref.lens, f"{name} {aggr} plain")
            for v in variants:
                what = f"{name} {aggr} scale={scaled} {v}"
                cats = []
                for _ in range(2):
                    cat = torch.full((n, 3 * dense), SENTINEL, device=DEV)
                    ops.seg_gmr_fused(*args, add_src if v["add"] else None,
                                      copy_src if v["copy"] else None,
                                      cat[:, 2 * dense:] if v["copy"] else None,
                                      cat[:, dense:2 * dense], add_src2 if v["add2"] else None)
                    cats.append(cat)
                assert same_bits(cats[0], cats[1]), what + ": two runs differ"
                cat = cats[0]
                want = red
                if v["add"]:
                    want = add_src + want
                if v["add2"]:
                    want = want + add_src2
                assert same_bits(cat[:, dense:2 * dense], want), what
                assert bool((cat[:, :dense] == SENTINEL).all()), what + ": wrote left of out"
                if v["copy"]:
                    assert same_bits(cat[:, 2 * dense:], copy_src), what + ": copy"
                else:
                    assert bool((cat[:, 2 * dense:] == SENTINEL).all()), what + ": wrote copy_dst"
                del cats, cat
    assert same_bits(src, src_bits), "an input buffer was written"


def test_host_rejects_before_launch(ops):
    """Arguments the C ABI refuses before any launch leave the output untouched."""
    plan = Plan(n_rows=300, lam=2.0, rws=(16,), seed=21, n_a=50, n_b=40)
    a, b, s = operands(plan, 128, 22)
    rowptr, c, d = plan.dev()
    a_d, b_d = torch.from_numpy(a).to(DEV), torch.from_numpy(b).to(DEV)
    n = plan.n_rows
    out = torch.full((n, 128), SENTINEL, device=DEV)
    src = torch.randn(n, 128, device=DEV)
    for aggr in ("max", "min"):
        with pytest.raises(Exception, match="accumulate needs sum or mean"):
            ops.seg_gmr_out(a_d, c, None, b_d, d, rowptr, n, CODE[aggr], out, True)
        with pytest.raises(Exception, match="sum or mean only"):
            ops.seg_gmr_fused(a_d, c, None, b_d, d, rowptr, n, CODE[aggr], src, None, None, out)
    with pytest.raises(Exception, match="add_src2 needs add_src"):
        ops.seg_gmr_fused(a_d, c, None, b_d, d, rowptr, n, 0, None, None, None, out, src)
    with pytest.raises(Exception, match="copy pair"):
        ops.seg_gmr_fused(a_d, c, None, b_d, d, rowptr, n, 0, None, src, None, out)
    out64 = torch.full((n, 64), SENTINEL, device=DEV)
    with pytest.raises(Exception, match="dense % 128"):
        ops.seg_gmr_fused(a_d[:, :64].contiguous(), c, None, None, None, rowptr, n, 0, None, None,
                          None, out64)
    torch.cuda.synchronize()
    assert bool((out == SENTINEL).all()) and bool((out64 == SENTINEL).all())
