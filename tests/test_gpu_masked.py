"""The MaskedTensor kernels -- the 2-FWL contraction ``mamamm`` (algo 0 in
pygho_b200/csrc/masked.cu, algos 1 and 2 in mamamm_tc.cu, algo 4 in mamamm_smem.cu) and masked
pooling (masked.cu) -- against a float64 reference, at every work split they use.

    mamamm:  out[b,i,k,c] = M[b,i,k] * sum_{j < e_j} A'[b,i,j,c] B'[b,j,k,c]    (i < e_i, k < e_k)
    pool:    out[o,q,c]   = aggr_{r : m[o,r,q]} x[o,r,q,c]        over the view (outer, red, inner)

u = 2^-24.  References are built on the CPU in float64 from the inputs (batched ``bmm`` for the
contractions), never from a kernel's own groupings.  Bounds are per element and channel, never
scaled by a global maximum; ``mag`` is the float64 sum of the absolute terms:

* mamamm, algos 0 and 4 (exact fp32, one ``fmaf`` chain per output in ascending j):
  ``|got - ref| <= 1.01 e_j u mag`` with e_j the graph's contraction extent (e_j roundings of
  size <= u; 1.01 covers the second-order term).  Outside the mask and the extents the output is
  exactly 0.  Algo 4 equals algo 0 bit for bit.
* mamamm, algos 1 and 2 (tcgen05 TF32): ``(2^-9 + 2^-20 + 1.01 k_pad 2^-23) mag``: at most 2^-10
  of truncation per TF32 operand (2^-9 + 2^-20 per product), and one truncating fp32 addition per
  K position, k_pad = e_j rounded up to 8.  Algo 2 equals algo 1 bit for bit (same tiles, same
  MMAs).
* mamamm through autograd: the forward as above with e_j = n; a gradient is a contraction over
  the other index (n terms) of the masked upstream gradient, so the same bound with its own
  ``mag``; pads of the leaves get exactly 0 through the MaskedTensor constructor.
* pool sum: ``1.01 (cnt + 16) u mag`` (a row's chain has cnt - 1 roundings; the cluster split
  adds at most 14 more: 7 in the warp combine, 7 in the rank combine).
* pool mean: the sum bound divided by cnt, plus ``1.01 u |mean|`` for the division.
* pool max / min and ``out_mask``: exact.  A valid +inf (max) or -inf (min) makes the output 0
  (filterinf), as in the reference.
* pool backward, bit for bit against numpy float32: sum ``g`` at valid positions; mean
  ``fl(g / cnt)``; max / min ``fl(g / ties)`` at the valid positions equal to the output, and 0
  for the whole channel when a valid entry is +inf (max) or -inf (min): the reference's
  ``masked_fill`` of the infinite result passes no gradient; 0 everywhere else.

Every raw launch writes into a NaN-filled output inside a larger buffer with guard regions; all
positions must be written and the guards untouched.  Every launch runs twice with the same bits.
Each case asserts the split it reaches through restatements of the C launch rules below; the ring
restatement is tied to the device through the profiling hook ``pgh_debug_trace``.  Tuning key 7,
bit 16 (four channels per lane in the ring's consumers) changes only the work split: every algo-4
case gives the same bits with key 7 = 0 and 16.
"""
import itertools
import zlib

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu
DEV = "cuda"
U = 2.0 ** -24
NAN = float("nan")
INF = float("inf")
AGGRS = ("sum", "mean", "max", "min")
CODE = {"sum": 0, "mean": 1, "max": 2, "min": 3}
GUARD = 1024                       # guard elements before (when offset) and after every output
RATIOS = {}                        # kernel -> worst |error| / bound seen (printed after the module)


@pytest.fixture(autouse=True)
def _reset_knobs():
    """Key 7 and the trace buffer are process-global: reset them after every test."""
    try:
        yield
    finally:
        if torch.cuda.is_available():
            from pygho_b200 import _lib
            _lib.call("pgh_set_tuning", 7, 0)
            _lib.call("pgh_debug_trace", None, 0)


@pytest.fixture(scope="module", autouse=True)
def _report_ratios():
    yield
    if RATIOS:
        print("\nworst |error| / bound: " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(RATIOS.items())))


def call(name, *args):
    from pygho_b200 import _lib
    _lib.call(name, *args)


def ptr(t):
    return None if t is None else t.data_ptr()


def stream():
    from pygho_b200._lib import stream_ptr
    return stream_ptr(torch.device(DEV))


def same_bits(a, b, what=""):
    if a.dtype == torch.float32:
        a, b = a.view(torch.int32), b.view(torch.int32)
    assert torch.equal(a, b), what


class Poisoned:
    """``n`` output elements at ``offset`` inside a buffer with GUARD elements after them, all
    NaN (float) or 0xAB (bytes) before the launch."""

    def __init__(self, n, offset=0, dtype=torch.float32):
        self.fill = NAN if dtype == torch.float32 else 0xAB
        self.buf = torch.full((offset + n + GUARD,), self.fill, dtype=dtype, device=DEV)
        self.out = self.buf[offset:offset + n]
        self.offset, self.n = offset, n

    def check(self, shape):
        """Every position written, both guards untouched; returns a copy of the output."""
        before, after = self.buf[:self.offset], self.buf[self.offset + self.n:]
        if self.buf.dtype == torch.float32:
            assert bool(torch.isnan(before).all()) and bool(torch.isnan(after).all()), "guard overwritten"
            assert not bool(torch.isnan(self.out).any()), "output position not written"
        else:
            assert bool((before == 0xAB).all()) and bool((after == 0xAB).all()), "guard overwritten"
            assert bool((self.out <= 1).all()), "output mask position not written"
        return self.out.view(shape).clone()


def check_bound(kernel, got, want, bound, what=""):
    """``|got - want| <= bound`` per element (NaN fails); records the worst ratio."""
    got = got.detach().cpu().double()
    err = (got - want).abs()
    ok = err <= bound
    if not bool(ok.all()):
        bad = ~ok
        idx = tuple(int(i) for i in bad.nonzero()[0])
        raise AssertionError(f"{kernel} {what}: {int(bad.sum())} elements over the bound; first at "
                             f"{idx}: got {float(got[idx])} want {float(want[idx])} bound {float(bound[idx])}")
    pos = bound > 0
    if bool(pos.any()):
        RATIOS[kernel] = max(RATIOS.get(kernel, 0.0), float((err[pos] / bound[pos]).max()))


def cdiv(a, b):
    return -(-a // b)


# ====================================================================== mamamm: restatements
# mamamm_smem.cu: kMsCH, kMsRB, kMsConsumers / 8 (kMsMaxPairs), kMsMaxStages, kMsSmemCap,
# kMsZeroBytes, ms_rows_per_pass, ms_plan, the producer's unit walk and the consumers' choice of
# channels per lane.  Keep in step with the C source.
MS_CH, MS_RB, MS_CONSUMERS, MS_MAX_STAGES = 16, 8, 224, 8
MS_MAX_PAIRS = MS_CONSUMERS // 8
MS_ROOM = 113 * 1024 - 2048 - 128 - 4096
MS_GRID = 2 * 148


def ms_rows_per_pass(nkb):
    itp = MS_MAX_PAIRS // nkb if nkb > 0 else MS_MAX_PAIRS
    return 4 * max(itp, 1)


def ms_plan(n_i, n_j, n_k, dense, tb):
    """(JC, stages) of a launch the ring takes, or None (the launch runs on algo 0)."""
    if dense % MS_CH or min(n_i, n_j, n_k) <= 0:
        return None
    jc = 5 if tb else 4
    nkb_max = cdiv(n_k, MS_RB)
    if nkb_max > MS_MAX_PAIRS:
        return None
    ni4 = cdiv(n_i, 4) * 4
    boxes = max(cdiv(min(ms_rows_per_pass(nkb), ni4), MS_RB) + nkb for nkb in range(1, nkb_max + 1))
    st = MS_ROOM // (boxes * MS_RB * jc * 64)
    return None if st < 3 else (jc, min(st, MS_MAX_STAGES))


def ms_unit(ei, ej, ek, jc):
    """(rows of each pass, chunks per pass, channels per lane of each pass) of one unit."""
    nkb = cdiv(ek, MS_RB)
    rpp = ms_rows_per_pass(nkb)
    nch = max(cdiv(ej, jc), 1) if ek > 0 else 0
    rows = [min(ei - r0, rpp) for r0 in range(0, ei, rpp)] if nch else []
    lanes = [2 if cdiv(r, 4) * nkb * 16 <= MS_CONSUMERS else 4 for r in rows]
    return rows, nch, lanes


# mamamm_tc.cu: mamamm_tc_launch (argument checks, k_pad, n_pad, tile sizes, the pipeline's ring
# and its fallback, wide) and the per-graph ch_round of both kernels.  Keep in step with the C
# source.
def tc_path(n_i, n_j, n_k, dense, out_ptr, pipelined):
    """"error", "pipe_wide", "pipe_narrow" or "tc" (the one-CTA-per-item kernel)."""
    if dense % 8 or n_i > 128 or n_k > 64 or n_j > 128:
        return "error"
    k_pad, n_pad = cdiv(n_j, 8) * 8, cdiv(n_k, 16) * 16
    sbo = k_pad // 4 * 128
    ts_a, ts_b = cdiv(n_i, 8) * sbo + 16, cdiv(n_k, 8) * sbo + 16
    off_b = cdiv(8 * ts_a, 128) * 128
    total = max(off_b + 8 * ts_b, 7 * ts_a + 16 * sbo, off_b + 7 * ts_b + n_pad // 8 * sbo)
    total = cdiv(total, 128) * 128
    ring_off = total + 3 * cdiv(n_i * 8, 128) * 128
    ring_bytes = (227 * 1024 - 1024 - ring_off) & ~127
    max_item = cdiv((n_i + n_k) * (k_pad * 32 + 16), 128) * 128
    if pipelined and ring_bytes >= max_item:
        return "pipe_wide" if out_ptr % 32 == 0 else "pipe_narrow"
    if total + cdiv(n_i * n_k, 128) * 128 > 227 * 1024:
        return "error"
    return "tc"


def tc_ch_round(ek):
    return 8 if 8 * max(cdiv(ek, 16) * 16, 16) <= 256 else 4


# ====================================================================== mamamm: operands, reference
def band(e1, n1, e2, n2):
    """(b, n1, n2) bool: rows < e1[b] and columns < e2[b]."""
    return (torch.arange(n1)[None, :, None] < e1[:, None, None]) & (torch.arange(n2)[None, None, :] < e2[:, None, None])


class MmCase:
    """Operands of one raw launch, stored as the kernels read them: A (b, n_i, n_j, d) or its
    transpose, B' likewise; zero outside the per-graph extents unless ``dirty_j`` (nonzero
    entries at j >= e_j, which the extents must exclude); a mask with holes that also covers
    positions outside the extents."""

    def __init__(self, b, n_i, n_j, n_k, d, ta, tb, ext, seed, dirty_j=False, hole=0.8):
        gen = torch.Generator().manual_seed(seed)
        ei, ej, ek = ext[:, 0].long(), ext[:, 1].long(), ext[:, 2].long()
        a = torch.randn((b, n_i, n_j, d), generator=gen)
        bb = torch.randn((b, n_j, n_k, d), generator=gen)
        if dirty_j:
            a = a * band(ei, n_i, torch.full_like(ej, n_j), n_j).unsqueeze(-1)
            bb = bb * band(torch.full_like(ej, n_j), n_j, ek, n_k).unsqueeze(-1)
        else:
            a = a * band(ei, n_i, ej, n_j).unsqueeze(-1)
            bb = bb * band(ej, n_j, ek, n_k).unsqueeze(-1)
        self.a, self.bb = a, bb                                  # A' and B' (CPU, float32)
        self.mask = torch.rand((b, n_i, n_k), generator=gen) < hole
        self.ext = ext
        self.ta, self.tb = ta, tb
        self.shape = (b, n_i, n_j, n_k, d)
        self.A = (a.transpose(1, 2) if ta else a).contiguous().to(DEV)
        self.B = (bb.transpose(1, 2) if tb else bb).contiguous().to(DEV)
        self.mask_dev = self.mask.to(DEV)
        self.ext_dev = ext.to(torch.int32).contiguous().to(DEV)

    def reference(self):
        """float64 (value, mag, e_j per graph) on the CPU."""
        b, n_i, n_j, n_k, d = self.shape
        ei, ej, ek = (self.ext[:, q].long().clamp(0) for q in range(3))
        a = self.a.double() * (torch.arange(n_j)[None, :] < ej[:, None])[:, None, :, None]
        x = a.permute(0, 3, 1, 2).reshape(b * d, n_i, n_j)
        y = self.bb.double().permute(0, 3, 1, 2).reshape(b * d, n_j, n_k)
        keep = (self.mask & band(ei, n_i, ek, n_k)).unsqueeze(-1)

        def out(t):
            return t.reshape(b, d, n_i, n_k).permute(0, 2, 3, 1) * keep
        return out(torch.bmm(x, y)), out(torch.bmm(x.abs(), y.abs())), ej.clamp(max=n_j)

    def run(self, algo, ext=True, order=None, offset=0):
        """Two raw launches into poisoned, guarded outputs; equal bits; returns the output."""
        b, n_i, n_j, n_k, d = self.shape
        outs = []
        for _ in range(2):
            o = Poisoned(b * n_i * n_k * d, offset)
            call("pgh_mamamm_f32", ptr(self.A), int(self.ta), ptr(self.B), int(self.tb),
                 ptr(self.mask_dev.view(torch.uint8)), ptr(self.ext_dev) if ext else None, ptr(order),
                 b, n_i, n_j, n_k, d, algo, ptr(o.out), stream())
            outs.append(o.check((b, n_i, n_k, d)))
        same_bits(outs[0], outs[1], "two launches differ")
        return outs[0]

    def check_exact(self, got, kernel):
        want, mag, ej = self.reference()
        check_bound(kernel, got, want, 1.01 * U * ej.double().view(-1, 1, 1, 1) * mag)

    def check_tf32(self, got, kernel):
        want, mag, ej = self.reference()
        k_pad = (cdiv(ej, 8) * 8).double().view(-1, 1, 1, 1)
        check_bound(kernel, got, want, (2.0 ** -9 + 2.0 ** -20 + 1.01 * k_pad * 2.0 ** -23) * mag)


TRACE_HALF = 1 << 13


def ring_trace(fn):
    """Run ``fn`` with the profiling hook on; returns the (tag, clock) events of CTA 0's producer
    thread (region 0) of the last launch."""
    tr = torch.zeros(2 + 2 * TRACE_HALF, dtype=torch.int64, device=DEV)
    call("pgh_debug_trace", ptr(tr), tr.numel())
    try:
        r = fn()
        torch.cuda.synchronize()
    finally:
        call("pgh_debug_trace", None, 0)
    t = tr.cpu()
    n0, n1 = int(t[0]), int(t[1])
    ev = t[2:2 + TRACE_HALF].view(-1, 2)[:n0]
    return r, ev, n0 + n1


def exts(b, n_i, n_j, n_k, gen, full0=True):
    """Per-graph extents drawn independently in each dimension; graph 0 full."""
    e = torch.stack([torch.randint(0, n + 1, (b,), generator=gen) for n in (n_i, n_j, n_k)], 1)
    if full0:
        e[0] = torch.tensor([n_i, n_j, n_k])
    return e


# name -> (n_i, n_j, n_k, dense, tb: True / False, or None for both), and what the name promises
RING, RING_EXPECT = {}, {}
for _jc, _tb in ((4, False), (5, True)):
    for _nj in (1, _jc - 1, _jc, _jc + 1, 300):          # a partial last chunk; more chunks than stages
        RING[f"chunks_jc{_jc}_nj{_nj}"] = (13, _nj, 13, 16, _tb)
        RING_EXPECT[f"chunks_jc{_jc}_nj{_nj}"] = dict(ring=True, chunks=cdiv(_nj, _jc))
for _st, _nk in ((3, 104), (4, 72), (5, 56), (6, 48), (7, 40), (8, 8)):
    RING[f"stages{_st}"] = (9, 6, _nk, 16, False)
    RING_EXPECT[f"stages{_st}"] = dict(stages=_st)
RING.update({
    # row passes: one; several with a short last one; 13 passes of 8 rows
    "passes_23x23": (23, 23, 23, 16, None),
    "passes_113x8": (113, 9, 8, 16, None),
    "passes_100x100": (100, 7, 100, 16, None),
    # both sides of the 2-versus-4 channels per lane boundary
    "lanes_56x8": (56, 5, 8, 16, None),
    "lanes_57x8": (57, 5, 8, 16, None),
    "lanes_28x16": (28, 6, 16, 16, None),
    "lanes_29x16": (29, 6, 16, 16, None),
    # both sides of the supported region's edges
    "edge_nk128_jc4": (9, 6, 128, 16, False),
    "edge_nk129_jc4": (9, 6, 129, 16, False),
    "edge_nk104_jc5": (9, 6, 104, 16, True),
    "edge_nk105_jc5": (9, 6, 105, 16, True),
    "edge_ni104_jc5": (104, 6, 9, 16, True),
    "edge_ni105_jc5": (105, 6, 9, 16, True),
    # one slab; more slabs than rows for the pad fill
    "dense16": (23, 23, 23, 16, None),
    "dense512_ni9": (9, 11, 10, 512, None),
    # fall back to algo 0
    "fallback_dense8": (23, 23, 23, 8, None),
    "fallback_dense40": (23, 23, 23, 40, None),
})
RING_EXPECT.update({
    "passes_23x23": dict(rows=[23]), "passes_113x8": dict(rows=[112, 1]),
    "passes_100x100": dict(rows=[8] * 12 + [4]),
    "lanes_56x8": dict(lanes=[2]), "lanes_57x8": dict(lanes=[4]),
    "lanes_28x16": dict(lanes=[2]), "lanes_29x16": dict(lanes=[4]),
    "edge_nk128_jc4": dict(ring=True), "edge_nk129_jc4": dict(ring=False),
    "edge_nk104_jc5": dict(ring=True), "edge_nk105_jc5": dict(ring=False),
    "edge_ni104_jc5": dict(ring=True), "edge_ni105_jc5": dict(ring=False),
    "dense16": dict(ring=True), "dense512_ni9": dict(ring=True),
    "fallback_dense8": dict(ring=False), "fallback_dense40": dict(ring=False),
})
RING_FORMS = [(name, ta, tb) for name, c in RING.items() for ta in (False, True)
              for tb in ((c[4],) if c[4] is not None else (False, True))]


def test_ring_cases_reach_their_splits():
    """The restatement puts every named case where its name says (CPU only)."""
    stages = set()
    for name, (n_i, n_j, n_k, d, tb0) in RING.items():
        for tb in ((tb0,) if tb0 is not None else (False, True)):
            plan = ms_plan(n_i, n_j, n_k, d, tb)
            want = RING_EXPECT[name]
            if "ring" in want:
                assert (plan is not None) == want["ring"], (name, tb)
            if plan is None:
                continue
            rows, nch, lanes = ms_unit(n_i, n_j, n_k, plan[0])
            stages.add(plan[1])
            got = dict(ring=True, stages=plan[1], rows=rows, chunks=nch, lanes=lanes)
            for k, v in want.items():
                assert got[k] == v, (name, tb, k, got[k], v)
    assert stages == {3, 4, 5, 6, 7, 8}
    # the region: JC 4 takes n_k <= 128, JC 5 n_k <= 104 and never n_i >= 105
    assert ms_plan(1, 1, 128, 16, False) and not ms_plan(1, 1, 129, 16, False)
    assert ms_plan(1, 1, 104, 16, True) and not ms_plan(1, 1, 105, 16, True)
    assert all(ms_plan(105, 1, nk, 16, True) is None for nk in range(1, 200))
    # 2 channels per lane at n <= 16 (ZINC's small graphs), 4 at ZINC's median n = 23
    assert ms_unit(16, 16, 16, 4)[2] == [2] and ms_unit(23, 23, 23, 4)[2] == [4]


@gpu
@pytest.mark.parametrize("name,ta,tb", RING_FORMS)
def test_ring_split(name, ta, tb):
    """Algo 4 at one split: b = 2 units per slab (graph 0 full, so CTA 0 takes exactly its first
    unit), checked against the reference, against algo 0 bit for bit, with key 7 = 16 bit for bit,
    and through the trace: passes x chunks issue events, or none when the ring declines."""
    n_i, n_j, n_k, d, _ = RING[name]
    seed = zlib.crc32(name.encode()) % 10000 + 2 * ta + tb
    gen = torch.Generator().manual_seed(seed)
    c = MmCase(2, n_i, n_j, n_k, d, ta, tb, exts(2, n_i, n_j, n_k, gen), seed=seed)
    plan = ms_plan(n_i, n_j, n_k, d, tb)
    got, ev, nev = ring_trace(lambda: c.run(4))
    if plan is None:
        assert nev == 0, "the ring ran a shape it should decline"
    else:
        rows, nch, _ = ms_unit(n_i, n_j, n_k, plan[0])
        tags = (ev[:, 0] >> 56).tolist()
        assert tags.count(1) == len(rows) * nch, (tags.count(1), rows, nch)
        assert tags.count(7) == 1
    c.check_exact(got, "algo4" if plan else "algo0")
    same_bits(got, c.run(0), "algo 4 != algo 0")
    call("pgh_set_tuning", 7, 16)
    same_bits(got, c.run(4), "key 7 = 16 changed bits")


@gpu
@pytest.mark.parametrize("ta,tb", [(False, False), (True, True)])
def test_ring_misaligned_pointer_falls_back(ta, tb):
    """An output that is not 16-byte aligned: the ring declines (empty trace), algo 0 runs."""
    gen = torch.Generator().manual_seed(11)
    c = MmCase(3, 23, 23, 23, 16, ta, tb, exts(3, 23, 23, 23, gen), seed=12)
    got, _, nev = ring_trace(lambda: c.run(4, offset=1))
    assert nev == 0
    c.check_exact(got, "algo0")
    same_bits(got, c.run(0))


# ------------------------------------------------------------------------------ queue
def queue_case(seed, ta, tb, b=200, n=40, d=128):
    gen = torch.Generator().manual_seed(seed)
    e = exts(b, n, n, n, gen)
    e[1, 0] = 0                                 # an empty graph in each dimension
    e[2, 1] = 0
    e[3, 2] = 0
    return MmCase(b, n, n, n, d, ta, tb, e, seed=seed + 1)


@gpu
@pytest.mark.parametrize("ta,tb", [(False, False), (True, False), (False, True), (True, True)])
def test_ring_queue(ta, tb):
    """b = 200, dense = 128: 1600 units over 296 CTAs (dynamic queue, two-ahead reads), extents
    drawn per dimension with zeros, holes; order None, largest first and random: same bits."""
    c = queue_case(5 + 2 * ta + tb, ta, tb)
    assert c.shape[0] * c.shape[4] // MS_CH > MS_GRID
    ref0 = c.run(0)
    c.check_exact(ref0, "algo0")
    e = c.ext.long()
    lpt = torch.argsort(e[:, 0] * e[:, 1] * e[:, 2], descending=True, stable=True).to(torch.int32).to(DEV)
    perm = torch.randperm(c.shape[0], generator=torch.Generator().manual_seed(3)).to(torch.int32).to(DEV)
    for key7 in (0, 16):
        call("pgh_set_tuning", 7, key7)
        for order in (None, lpt, perm):
            same_bits(c.run(4, order=order), ref0, f"key7={key7}")


@gpu
def test_ring_two_streams_and_graph_replay():
    """Two launches of > 296 units each on two streams at once, and one CUDA graph holding two
    launches replayed three times: the same bits as serial launches."""
    import pygho_b200.ops  # noqa: F401
    mm = torch.ops.pygho_b200.mamamm
    c1, c2 = queue_case(21, False, True), queue_case(22, True, False)

    def launch(c):
        return mm(c.A, c.ta, c.B, c.tb, c.mask_dev, c.ext_dev, 4)
    r1, r2 = c1.run(0), c2.run(0)
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    s1.wait_stream(torch.cuda.current_stream())
    s2.wait_stream(torch.cuda.current_stream())
    for _ in range(2):
        with torch.cuda.stream(s1):
            o1 = launch(c1)
        with torch.cuda.stream(s2):
            o2 = launch(c2)
        torch.cuda.synchronize()
        same_bits(o1, r1)
        same_bits(o2, r2)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        o1 = launch(c1)
        o2 = launch(c2)
    for _ in range(3):
        o1.fill_(NAN)
        o2.fill_(NAN)
        g.replay()
        torch.cuda.synchronize()
        same_bits(o1, r1)
        same_bits(o2, r2)


# ------------------------------------------------------------------------------ algo 0
@gpu
@pytest.mark.parametrize("d", [1, 33, 40, 128])
@pytest.mark.parametrize("ta,tb", [(False, False), (True, False), (False, True), (True, True)])
def test_algo0(d, ta, tb):
    """Algo 0: 13 x 10 x 15 (no multiple of 4, 16 tiles > 8 warps), channel slabs with idle
    lanes, extents that limit j while the operands hold nonzero data beyond them."""
    gen = torch.Generator().manual_seed(d * 4 + 2 * ta + tb)
    b, n_i, n_j, n_k = 4, 13, 10, 15
    e = exts(b, n_i, n_j, n_k, gen)
    e[1] = torch.tensor([n_i, 3, n_k])
    c = MmCase(b, n_i, n_j, n_k, d, ta, tb, e, seed=d + 7, dirty_j=True)
    c.check_exact(c.run(0), "algo0")
    full = MmCase(b, n_i, n_j, n_k, d, ta, tb, torch.tensor([[n_i, n_j, n_k]] * b), seed=d + 8)
    full.check_exact(full.run(0, ext=False), "algo0")


# ------------------------------------------------------------------------------ algos 1 and 2
TC_SHAPES = []
for _q, (_ni, _nj) in enumerate(itertools.product((1, 33, 100, 128), (1, 7, 8, 9, 128))):
    TC_SHAPES.append((_ni, _nj, (32, 33, 64)[_q % 3], 16, [(False, False), (True, False), (False, True), (True, True)][_q % 4], _q % 2 * 4))
TC_SHAPES += [(40, 40, 40, 64, (False, False), 0),       # b x dense / 8 = 160 items > 148 SMs
              (40, 40, 40, 64, (True, True), 4),         # ... written 16-byte aligned only
              (48, 48, 48, 16, (False, True), 0)]        # does not fit the ring: algo 1's kernel
TC_LIMITS = [(129, 8, 8, 16), (8, 129, 8, 16), (8, 8, 65, 16), (8, 8, 8, 12), (33, 128, 32, 16)]


def test_tc_cases_reach_their_splits():
    paths = {tc_path(ni, nj, nk, d, off * 4, True) for ni, nj, nk, d, _, off in TC_SHAPES}
    assert paths == {"pipe_wide", "pipe_narrow", "tc", "error"}, paths
    rounds = {tc_ch_round(nk) for _, _, nk, _, _, _ in TC_SHAPES}
    assert rounds == {4, 8}
    assert any(ni * nk > 2048 for ni, _, nk, _, _, _ in TC_SHAPES)        # mask tile > 2048 B
    for shape in TC_LIMITS:
        assert tc_path(*shape, 0, True) == tc_path(*shape, 0, False) == "error", shape


@gpu
@pytest.mark.parametrize("n_i,n_j,n_k,d,tt,off", TC_SHAPES)
def test_tf32(n_i, n_j, n_k, d, tt, off):
    """Algos 1 and 2 against the TF32 bound; algo 2 equals algo 1 bit for bit; the trace shows
    whether the pipeline or its fallback ran."""
    ta, tb = tt
    b = 20 if d == 64 else 3
    gen = torch.Generator().manual_seed(n_i * 1000 + n_j * 10 + n_k + off)
    c = MmCase(b, n_i, n_j, n_k, d, ta, tb, exts(b, n_i, n_j, n_k, gen), seed=n_i + n_j + n_k)
    path = tc_path(n_i, n_j, n_k, d, off * 4, True)
    if path == "error":
        check_tc_limit(c)
        return
    one = c.run(1, offset=off)
    c.check_tf32(one, "algo1")
    # the pipeline's CTA 0 stamps the trace buffer, the one-CTA-per-item kernel never does
    tr = torch.zeros(512, dtype=torch.int64, device=DEV)
    call("pgh_debug_trace", ptr(tr), tr.numel())
    try:
        two = c.run(2, offset=off)
        torch.cuda.synchronize()
    finally:
        call("pgh_debug_trace", None, 0)
    assert bool((tr != 0).any()) == path.startswith("pipe"), path
    same_bits(two, one, "algo 2 != algo 1")
    c.check_tf32(two, "algo2")


def check_tc_limit(c):
    from pygho_b200 import _lib
    from pygho_b200.ops import mamamm_algo_for
    b, n_i, n_j, n_k, d = c.shape
    for algo in (1, 2):
        with pytest.raises(_lib.KernelError):
            c.run(algo)
        assert mamamm_algo_for(algo, n_i, n_j, n_k, d) == 0
    assert mamamm_algo_for(4, n_i, n_j, n_k, d) == 4


@gpu
@pytest.mark.parametrize("n_i,n_j,n_k,d", TC_LIMITS)
def test_tf32_limits(n_i, n_j, n_k, d):
    """Over the tensor-core limits (extents, dense % 8, tiles beyond shared memory) the raw op is
    an argument error and the library routes the call to algo 0."""
    check_tc_limit(MmCase(2, n_i, n_j, n_k, d, False, False, torch.tensor([[n_i, n_j, n_k]] * 2), seed=1))


# ------------------------------------------------------------------------------ autograd
def ref_mm_grads(a, bb, mA, mB, M, w, einsum):
    """float64 CPU autograd of sum(w * M o ((a o mA)' (bb o mB)')): value, grads."""
    x = a.double().requires_grad_(True)
    y = bb.double().requires_grad_(True)
    out = torch.einsum(einsum, x * mA.unsqueeze(-1), y * mB.unsqueeze(-1)) * M.unsqueeze(-1)
    (out * w.double()).sum().backward()
    return out.detach(), x.grad, y.grad


@gpu
@pytest.mark.parametrize("d", [16, 128])
@pytest.mark.parametrize("d1,d2", [(1, 1), (1, 2), (2, 1), (2, 2)])
def test_mamamm_autograd_default_algo(d, d1, d2):
    """``B.mamamm`` with the default algo: operand masks whose row extent differs from their
    column extent, an output mask reaching beyond the operands' extents; value and both leaf
    gradients against float64 autograd."""
    import pygho_b200.backend as B
    from pygho_b200.backend.Mamamm import default_algo
    assert default_algo() == 4
    b, n = 6, 23
    gen = torch.Generator().manual_seed(d + 10 * d1 + d2)
    r = lambda lo: torch.randint(lo, n + 1, (b,), generator=gen)  # noqa: E731
    rA, cA, rB, cB = r(2), r(2), r(2), r(2)
    rA[0], cA[0], rB[0], cB[0] = 9, 20, 17, 6              # rows != columns in both operands
    mA, mB = band(rA, n, cA, n), band(rB, n, cB, n)
    M = band(r(12), n, r(12), n) & (torch.rand((b, n, n), generator=gen) < 0.9)
    M[0] = True
    a = torch.randn((b, n, n, d), generator=gen)            # nonzero everywhere: the pads must be filled
    bb = torch.randn((b, n, n, d), generator=gen)
    w = torch.randn((b, n, n, d), generator=gen)
    sa = "bji" if d1 == 1 else "bij"
    sb = "bjk" if d2 == 1 else "bkj"
    es = f"{sa}d,{sb}d->bikd"
    want, ga, gb = ref_mm_grads(a, bb, mA, mB, M, w, es)
    mag, ma_, mb_ = ref_mm_grads(a.abs(), bb.abs(), mA, mB, M, w.abs(), es)
    ag, bg = a.to(DEV).requires_grad_(True), bb.to(DEV).requires_grad_(True)
    out = B.mamamm(B.MaskedTensor(ag, mA.to(DEV)), d1, B.MaskedTensor(bg, mB.to(DEV)), d2, M.to(DEV))
    (out.data * w.to(DEV)).sum().backward()
    bound = lambda m: 1.01 * n * U * m                     # noqa: E731
    check_bound("algo4", out.data, want, bound(mag), "forward")
    check_bound("algo4", ag.grad, ga, bound(ma_), "dA")
    check_bound("algo4", bg.grad, gb, bound(mb_), "dB")


@gpu
@pytest.mark.parametrize("d2", [1, 2])
def test_mamamm_autograd_3d_operand(d2):
    """A with three masked dims (b, n, n, n), contracted over its last; B (b, n, n)."""
    import pygho_b200.backend as B
    b, n, d = 3, 7, 16
    gen = torch.Generator().manual_seed(40 + d2)
    mA = torch.rand((b, n, n, n), generator=gen) < 0.7
    mB = band(torch.tensor([7, 4, 6]), n, torch.tensor([5, 7, 2]), n)
    M = torch.rand((b, n, n, n), generator=gen) < 0.8
    a = torch.randn((b, n, n, n, d), generator=gen)
    bb = torch.randn((b, n, n, d), generator=gen)
    w = torch.randn((b, n, n, n, d), generator=gen)
    es = "bxyjd,bjkd->bxykd" if d2 == 1 else "bxyjd,bkjd->bxykd"
    want, ga, gb = ref_mm_grads(a, bb, mA, mB, M, w, es)
    mag, ma_, mb_ = ref_mm_grads(a.abs(), bb.abs(), mA, mB, M, w.abs(), es)
    ag, bg = a.to(DEV).requires_grad_(True), bb.to(DEV).requires_grad_(True)
    out = B.mamamm(B.MaskedTensor(ag, mA.to(DEV)), 3, B.MaskedTensor(bg, mB.to(DEV)), d2, M.to(DEV))
    (out.data * w.to(DEV)).sum().backward()
    check_bound("algo4", out.data, want, 1.01 * n * U * mag, "forward")
    check_bound("algo4", ag.grad, ga, 1.01 * n * U * ma_, "dA")        # over k: n terms
    check_bound("algo4", bg.grad, gb, 1.01 * n * n * U * mb_, "dB")    # over (x, y): n^2


# ====================================================================== masked pooling
# masked.cu: pool_view and the dispatch of pgh_masked_pool_f32 / pgh_masked_pool_bwd_f32
# (warp_path = c4 % 32 == 0, split = red >= 128 && warps < 8 kSMs), kPoolCluster = 8 CTAs of 8
# warps, 32 positions per chunk.  Keep in step with the C source.
def pool_view(b, n1, n2, red_dims):
    return {1: (b, n1, n2), 2: (b * n1, n2, 1), 3: (b, n1 * n2, 1)}[red_dims]


def pool_kernel(b, n1, n2, dense, red_dims):
    outer, red, inner = pool_view(b, n1, n2, red_dims)
    c4 = dense // 4
    warps = outer * inner * (c4 // 32)
    if c4 % 32:
        return "thread"
    return "split" if red >= 128 and warps < 8 * 148 else "warp"


def pool_data(outer, red, inner, d, aggr, density, seed, infs=None):
    """(x, m) in the view's shape.  Small integers (ties) in most channels, Gaussians in every
    fourth group of 4; output rows: the second fully masked, the third with a single entry;
    max: channels 8..11 all negative, min: all positive; with ``infs``: valid +inf and -inf
    next to exact zeros (channels 0..7 of every row)."""
    rng = np.random.default_rng(seed)
    x = rng.integers(-3, 4, (outer, red, inner, d)).astype(np.float32)
    g4 = (np.arange(d) // 4) % 4 == 3
    x[..., g4] = rng.standard_normal((outer, red, inner, int(g4.sum()))).astype(np.float32)
    m = rng.random((outer, red, inner)) < density
    rows = [(o, q) for o in range(outer) for q in range(inner)]
    if len(rows) >= 3:
        o, q = rows[1]
        m[o, :, q] = False
        o, q = rows[2]
        m[o, :, q] = False
        m[o, rng.integers(red), q] = True
    if aggr in ("max", "min") and d >= 12:
        x[..., 8:12] = -np.abs(x[..., 8:12]) - 1 if aggr == "max" else np.abs(x[..., 8:12]) + 1
    if infs and d >= 8:
        x[..., 0:8] = 0.0
        pos = rng.integers(red, size=(outer, inner))
        for (o, q) in rows:
            r = pos[o, q]
            x[o, r, q, 0:2] = INF
            x[o, r, q, 2:4] = -INF
            x[o, (r + 1) % red, q, 4:6] = INF            # maybe masked out: then the zeros win
            x[o, :, q, 6] = -INF                         # channel 6: all -inf; 7: all +inf
            x[o, :, q, 7] = INF
    return x, m


def pool_reference(x, m, aggr, g):
    """float64 (value, bound) and the float32 gradient wanted, over axis 1 of the view."""
    x64 = x.astype(np.float64)
    mm = m[..., None]
    cnt = m.sum(1)[..., None].astype(np.float64)
    if aggr in ("sum", "mean"):
        s = np.where(mm, x64, 0).sum(1)
        mag = np.where(mm, np.abs(x64), 0).sum(1)
        bound = 1.01 * (cnt + 16) * U * mag
        gw = np.broadcast_to(g[:, None], x.shape)
        if aggr == "sum":
            return s, bound, np.where(mm, gw, np.float32(0))
        c1 = np.maximum(cnt, 1)
        mean = s / c1
        wgt = g / np.maximum(cnt, 1).astype(np.float32)
        return mean, bound / c1 + 1.01 * U * np.abs(mean), np.where(mm, wgt[:, None], np.float32(0))
    pole = INF if aggr == "max" else -INF
    red = np.where(mm, x64, -pole)
    ext = red.max(1) if aggr == "max" else red.min(1)
    ext = np.where(np.isinf(ext), 0.0, ext)
    tie = mm & (x64 == ext[:, None])
    ties = tie.sum(1)
    dead = (mm & (x64 == pole)).any(1)
    wgt = np.where((ties > 0) & ~dead, g / np.maximum(ties, 1).astype(np.float32), np.float32(0))
    return ext, np.zeros_like(ext), np.where(tie, wgt[:, None], np.float32(0)).astype(np.float32)


def pool_raw(x, m, b, n1, n2, red_dims, aggr):
    """Forward and backward through the C ABI, each twice, poisoned and guarded; returns the
    (output, out_mask, gradient, g) of the view."""
    d = x.shape[-1]
    outer, red, inner = pool_view(b, n1, n2, red_dims)
    xd = torch.from_numpy(x.reshape(b, n1, n2, d)).to(DEV)
    md = torch.from_numpy(m.reshape(b, n1, n2)).to(DEV).view(torch.uint8)
    keep = outer * inner
    res = []
    for _ in range(2):
        o = Poisoned(keep * d)
        om = Poisoned(keep, dtype=torch.uint8)
        call("pgh_masked_pool_f32", ptr(xd), ptr(md), b, n1, n2, d, red_dims, CODE[aggr], ptr(o.out),
             ptr(om.out), stream())
        res.append((o.check((outer, inner, d)), om.check((outer, inner))))
    same_bits(res[0][0], res[1][0], "forward: two launches differ")
    same_bits(res[0][1], res[1][1])
    out, omask = res[0]
    g = torch.from_numpy(np.random.default_rng(7).standard_normal((outer, inner, d)).astype(np.float32)).to(DEV)
    grads = []
    for _ in range(2):
        gd = Poisoned(x.size)
        call("pgh_masked_pool_bwd_f32", ptr(xd), ptr(md), ptr(out), ptr(g), b, n1, n2, d, red_dims,
             CODE[aggr], ptr(gd.out), stream())
        grads.append(gd.check((outer, red, inner, d)))
    same_bits(grads[0], grads[1], "backward: two launches differ")
    return out.cpu().numpy(), omask.cpu().numpy(), grads[0].cpu().numpy(), g.cpu().numpy()


def check_pool(x, m, b, n1, n2, red_dims, aggr, kernel):
    assert pool_kernel(b, n1, n2, x.shape[-1], red_dims) == kernel
    out, omask, grad, g = pool_raw(x, m, b, n1, n2, red_dims, aggr)
    want, bound, gwant = pool_reference(x, m, aggr, g)
    assert np.array_equal(omask.astype(bool), m.any(1)), "out_mask"
    check_bound(f"pool_{kernel}", torch.from_numpy(out), torch.from_numpy(want), torch.from_numpy(bound), aggr)
    assert np.array_equal(grad.view(np.int32), gwant.astype(np.float32).view(np.int32)), \
        f"{aggr} backward: {int((grad != gwant).sum())} positions differ"


def view_shape(outer, red, inner, red_dims):
    """(b, n1, n2) whose view is (outer, red, inner)."""
    if red_dims == 1:
        return outer, red, inner
    if red_dims == 2:
        assert inner == 1
        return outer, 1, red
    assert inner == 1
    return outer, red, 1


@gpu
@pytest.mark.parametrize("aggr", AGGRS)
@pytest.mark.parametrize("d", [4, 12, 124, 132])
@pytest.mark.parametrize("red", [1, 3, 4, 5, 7])
def test_pool_thread(aggr, d, red):
    """c4 % 32 != 0: the thread kernel's 4-row unroll and its tail."""
    x, m = pool_data(3, red, 5, d, aggr, 0.7, seed=d * 10 + red, infs=aggr in ("max", "min"))
    check_pool(x, m, 3, red, 5, 1, aggr, "thread")


@gpu
@pytest.mark.parametrize("aggr", AGGRS)
@pytest.mark.parametrize("d", [128, 256, 384])
@pytest.mark.parametrize("red", [1, 31, 32, 33, 127])
@pytest.mark.parametrize("density", [0.95, 0.2])
def test_pool_warp(aggr, d, red, density):
    """Warp kernel: partial and whole 32-position chunks; dense masks batch more than 8 loads per
    chunk, sparse masks few."""
    x, m = pool_data(2, red, 7, d, aggr, density, seed=d + red, infs=aggr in ("max", "min"))
    check_pool(x, m, 2, red, 7, 1, aggr, "warp")


@gpu
@pytest.mark.parametrize("aggr", AGGRS)
def test_pool_warp_past_split_limit(aggr):
    """red = 128 with 1184 = 8 x 148 warps: just past the split limit, the warp kernel."""
    x, m = pool_data(8, 128, 148, 128, aggr, 0.5, seed=3, infs=aggr in ("max", "min"))
    check_pool(x, m, 8, 128, 148, 1, aggr, "warp")


# (red, warps) -> (outer, inner, dense, red_dims)
SPLIT = {}
for _red in (128, 129, 1792, 1793, 2048, 2049, 4129):
    SPLIT[(_red, 1)] = (1, 1, 128, 2)
    SPLIT[(_red, 3)] = (1, 1, 384, 3) if _red % 2 else (3, 1, 128, 1)
SPLIT[(128, 1183)] = (7, 169, 128, 1)
SPLIT[(129, 1183)] = (1183, 1, 128, 2)


@gpu
@pytest.mark.parametrize("aggr", AGGRS)
@pytest.mark.parametrize("red,warps", list(SPLIT))
def test_pool_split(aggr, red, warps):
    """Cluster split (8 CTAs x 8 warps per output row, 2048 positions per pass): idle warps
    (128, 1792), a non-empty partial from CTA rank 7 (1793), second and third chunks per warp
    (2049, 4129)."""
    outer, inner, d, red_dims = SPLIT[(red, warps)]
    assert outer * inner * d // 128 == warps
    b, n1, n2 = view_shape(outer, red, inner, red_dims)
    x, m = pool_data(outer, red, inner, d, aggr, 0.6, seed=red + warps, infs=aggr in ("max", "min"))
    check_pool(x, m, b, n1, n2, red_dims, aggr, "split")


@gpu
@pytest.mark.parametrize("aggr", ["max", "min"])
@pytest.mark.parametrize("kernel", ["thread", "warp", "split"])
def test_pool_infinite_extreme_passes_no_gradient(aggr, kernel):
    """Data [inf, 0, 0] (max) or [-inf, 0, 0] (min), all valid: the output is 0 (filterinf) and,
    as in the reference, no entry gets a gradient -- not the zeros that equal the output."""
    d = {"thread": 4, "warp": 128, "split": 128}[kernel]
    red = 3 if kernel != "split" else 130
    x = np.zeros((1, red, 1, d), np.float32)
    x[0, 0, 0, :] = INF if aggr == "max" else -INF
    m = np.ones((1, red, 1), bool)
    check_pool(x, m, 1, red, 1, 1, aggr, kernel)
    _, _, grad, _ = pool_raw(x, m, 1, red, 1, 1, aggr)
    assert not grad.any()


@gpu
@pytest.mark.parametrize("red_dims", [2, 3])
@pytest.mark.parametrize("d", [12, 128])
def test_pool_red_dims(red_dims, d):
    """red_dims 2 (reduce n2) and 3 (reduce n1 x n2) through the raw op."""
    b, n1, n2 = 4, 9, 11
    outer, red, inner = pool_view(b, n1, n2, red_dims)
    for aggr in AGGRS:
        x, m = pool_data(outer, red, inner, d, aggr, 0.6, seed=red_dims + d, infs=aggr in ("max", "min"))
        check_pool(x, m, b, n1, n2, red_dims, aggr, pool_kernel(b, n1, n2, d, red_dims))


# ------------------------------------------------------------------------------ public API
def api_reference(x, m, dims, aggr, g):
    """Pool a (b, *masked, *dense) numpy tensor over masked ``dims``: value, bound and float32
    gradient wanted (the rules of the module docstring, over several axes)."""
    nd = x.ndim - m.ndim
    mm = m.reshape(m.shape + (1,) * nd)
    ax = tuple(dims)
    x64 = x.astype(np.float64)
    cnt = m.sum(ax).reshape(m.sum(ax).shape + (1,) * nd).astype(np.float64)

    def spread(v):
        return np.expand_dims(v, ax)
    if aggr in ("sum", "mean"):
        s = np.where(mm, x64, 0).sum(ax)
        bound = 1.01 * (cnt + 16) * U * np.where(mm, np.abs(x64), 0).sum(ax)
        if aggr == "sum":
            return s, bound, np.where(mm, spread(g), np.float32(0))
        c1 = np.maximum(cnt, 1)
        wgt = g / c1.astype(np.float32)
        return s / c1, bound / c1 + 1.01 * U * np.abs(s / c1), np.where(mm, spread(wgt), np.float32(0))
    pole = INF if aggr == "max" else -INF
    red = np.where(mm, x64, -pole)
    ext = red.max(ax) if aggr == "max" else red.min(ax)
    ext = np.where(np.isinf(ext), 0.0, ext)
    tie = mm & (x64 == spread(ext))
    ties = tie.sum(ax)
    dead = (mm & (x64 == pole)).any(ax)
    wgt = np.where((ties > 0) & ~dead, g / np.maximum(ties, 1).astype(np.float32), np.float32(0))
    return ext, np.zeros_like(ext), np.where(tie, spread(wgt), np.float32(0)).astype(np.float32)


API = [((5, 9, 9), 16, (0,)), ((5, 9, 9), 16, (1,)), ((5, 9, 9), 128, (2,)), ((5, 9, 9), 128, (1, 2)),
       ((5, 9, 9), 16, (0, 2)), ((3, 6, 6, 6), 128, (1, 3)), ((4, 7, 7), 1, (1,)), ((4, 7, 7), 3, (1, 2)),
       ((4, 7, 7), 130, (2,)), ((4, 7, 7), 130, (0, 2)),
       ((128, 38, 38), 128, (1, 2)), ((128, 38, 38), 128, (1,))]        # ZINC scale


@gpu
@pytest.mark.parametrize("aggr", AGGRS)
@pytest.mark.parametrize("mshape,d,dims", API)
def test_pool_public_api(aggr, mshape, d, dims):
    """MaskedTensor.sum / mean / max / min: dims 0, 1, 2, (1, 2), non-adjacent dims (permute),
    odd widths (pad to 4), ZINC scale; value, mask and the leaf gradient."""
    import pygho_b200.backend as B
    rng = np.random.default_rng(hash((mshape, d, dims)) % 1000)
    x = rng.integers(-3, 4, mshape + (d,)).astype(np.float32)
    x[..., ::3] = rng.standard_normal(x[..., ::3].shape).astype(np.float32)
    m = rng.random(mshape) < 0.6
    m[0] = False                                            # fully masked output rows
    if aggr in ("max", "min"):
        flat = x.reshape(-1, d)
        pick = rng.integers(flat.shape[0], size=flat.shape[0] // 20)
        flat[pick, 0] = INF if aggr == "max" else -INF
        flat[pick[::2], min(1, d - 1)] = -INF if aggr == "max" else INF
        flat[rng.integers(flat.shape[0], size=flat.shape[0] // 4), d - 1] = 0.0
    xd = torch.from_numpy(x).to(DEV).requires_grad_(True)
    r = getattr(B.MaskedTensor(xd, torch.from_numpy(m).to(DEV)), aggr)(list(dims))
    g = rng.standard_normal(tuple(r.data.shape)).astype(np.float32)
    (r.data * torch.from_numpy(g).to(DEV)).sum().backward()
    want, bound, gwant = api_reference(x, m, dims, aggr, g)
    assert np.array_equal(r.mask.cpu().numpy(), m.any(tuple(dims)))
    check_bound("pool_api", r.data, torch.from_numpy(want), torch.from_numpy(bound), f"{aggr} {dims}")
    got = xd.grad.cpu().numpy()
    assert np.array_equal(got.view(np.int32), gwant.view(np.int32)), \
        f"{aggr} backward: {int((got != gwant).sum())} positions differ"
