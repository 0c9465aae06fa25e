"""Device-side index plans (int32 CSR groupings) and the integer kernels that build them.

A *triple plan* is a list of T triples ``(a_t, c_t, d_t)`` meaning "row ``c_t`` of operand
A times row ``d_t`` of operand B contributes to output row ``a_t``".  The reference keeps
it as a ``(3, T)`` LongTensor (``acd``, backend/Spspmm.py:186-222) and scatters with
atomics; here it is regrouped once per batch into up to three CSR groupings

* by ``a`` -- the forward pass (segmented reduce into output rows),
* by ``c`` and by ``d`` -- the two operand gradients,

each built with a stable radix sort so every reduction order is deterministic.  An index
that is ``None`` is the identity (``t`` itself); a grouping whose ``rowptr`` is ``None``
has exactly one triple per row, in order.  Plans are cached on the index tensor they
were derived from (``tensor._pgh_cache``), which is how "precomputed once per batch in
hodata and cached on device" (BASELINE.json north_star) is realised without changing the
reference's ``datadict`` contract.
"""
from __future__ import annotations

import os
from typing import Dict, NamedTuple, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib
from ._lib import call, ptr, size_query, stream_ptr

_CHECK = os.environ.get("PYGHO_B200_CHECK", "0") == "1"


class Group(NamedTuple):
    rowptr: Optional[Tensor]
    first: Optional[Tensor]
    second: Optional[Tensor]


# ------------------------------------------------------------------ small raw wrappers
def _empty(n, dtype, device):
    return torch.empty((int(n),), dtype=dtype, device=device)


def _ws(nbytes: int, device) -> Tensor:
    return torch.empty((max(int(nbytes), 256),), dtype=torch.uint8, device=device)


def _launch(name, *args):
    call(name, *args)
    _lib.count_launch()


def _host_i32(vals: Sequence[int]):
    import ctypes as C
    return (C.c_int32 * len(vals))(*[int(v) for v in vals])


def _host_i64(vals: Sequence[int]):
    import ctypes as C
    return (C.c_int64 * len(vals))(*[int(v) for v in vals])


def to_i32(x: Tensor) -> Tensor:
    """int64 -> int32 on the device (values are row ids, < 2^31)."""
    if x.dtype == torch.int32:
        return x.contiguous()
    x = x.contiguous()
    _lib.require_cuda(x)
    out = _empty(x.numel(), torch.int32, x.device)
    _launch("pgh_i64_to_i32", ptr(x), x.numel(), ptr(out), None, stream_ptr(x.device))
    return out


def to_i64(x: Tensor) -> Tensor:
    x = x.contiguous()
    out = _empty(x.numel(), torch.int64, x.device)
    _launch("pgh_i32_to_i64", ptr(x), x.numel(), ptr(out), stream_ptr(x.device))
    return out


def gather_i32(src: Tensor, idx: Tensor) -> Tensor:
    out = _empty(idx.numel(), torch.int32, idx.device)
    _launch("pgh_gather_i32", ptr(src), ptr(idx), idx.numel(), ptr(out), stream_ptr(idx.device))
    return out


def sort_keys(key: Tensor, end_bit: int) -> Tuple[Tensor, Tensor]:
    """Stable sort of int64 keys on their low ``end_bit`` bits -> (sorted keys, perm int32)."""
    n = key.numel()
    dev = key.device
    ks, perm = _empty(n, torch.int64, dev), _empty(n, torch.int32, dev)
    if n:
        nb = size_query("pgh_sort_ws_bytes", n)
        ws = _ws(nb, dev)
        _launch("pgh_sort_keys_perm", ptr(key), n, int(end_bit), ptr(ks), ptr(perm), ptr(ws),
                ws.numel(), stream_ptr(dev))
    return ks, perm


def unique_sorted(ks: Tensor) -> Tuple[Tensor, Tensor, int]:
    """Run-length unique of sorted keys -> (unique keys, run id per element, count).
    Reads the count back (one host synchronisation)."""
    n = ks.numel()
    dev = ks.device
    ukey, seg = _empty(n, torch.int64, dev), _empty(n, torch.int32, dev)
    cnt = torch.zeros((1,), dtype=torch.int32, device=dev)
    if n:
        ws = _ws(size_query("pgh_unique_ws_bytes", n), dev)
        _launch("pgh_unique_sorted", ptr(ks), n, ptr(ukey), ptr(seg), ptr(cnt), ptr(ws),
                ws.numel(), stream_ptr(dev))
    count = int(cnt.item()) if n else 0
    return ukey[:count], seg, count


def rowptr_from_sorted(key32: Tensor, n_rows: int) -> Tensor:
    rp = _empty(n_rows + 1, torch.int32, key32.device)
    _launch("pgh_rowptr_from_sorted", ptr(key32), key32.numel(), int(n_rows), ptr(rp),
            stream_ptr(key32.device))
    return rp


def csr_of(key32: Tensor, n_rows: int, assume_sorted: bool = False
           ) -> Tuple[Tensor, Optional[Tensor]]:
    """(rowptr, perm) of an int32 key array; ``perm`` is None when the caller knows the
    keys are non-decreasing.  Sorting is stable, so a segment keeps the input order.
    A key equal to ``n_rows`` means "no row": such entries sort behind ``rowptr[n_rows]`` and
    are never visited (filler entries of capacity-padded plans, pygho_b200/static.py)."""
    if assume_sorted or key32.numel() == 0:
        return rowptr_from_sorted(key32, n_rows), None
    n, dev = key32.numel(), key32.device
    key32 = key32.contiguous()
    ks, perm = _empty(n, torch.int32, dev), _empty(n, torch.int32, dev)
    ws = _ws(size_query("pgh_sort_ws_bytes", n), dev)
    _launch("pgh_sort_i32_perm", ptr(key32), n, max(1, int(n_rows).bit_length()), ptr(ks), ptr(perm),
            ptr(ws), ws.numel(), stream_ptr(dev))
    return rowptr_from_sorted(ks, n_rows), perm


def _take(x: Optional[Tensor], perm: Optional[Tensor]) -> Optional[Tensor]:
    if perm is None:
        return x
    if x is None:
        return perm
    return gather_i32(x, perm)


class TriplePlan:
    """T triples (a, c, d) with lazily built, cached CSR groupings (all int32)."""

    def __init__(self, T: int, n_out: int, n_a: int, n_b: int, a: Optional[Tensor],
                 c: Optional[Tensor], d: Optional[Tensor], sorted_by: str = ""):
        self.T, self.n_out, self.n_a, self.n_b = int(T), int(n_out), int(n_a), int(n_b)
        self.idx = {"a": a, "c": c, "d": d}
        self.sorted_by = sorted_by  # which index arrays are known to be non-decreasing
        self._groups: Dict[str, Group] = {}
        self._inv: Optional[Tensor] = None
        self._swapped: Optional["TriplePlan"] = None

    _ORDER = {"a": ("c", "d", "n_out"), "c": ("a", "d", "n_a"), "d": ("a", "c", "n_b")}

    def group(self, which: str) -> Group:
        g = self._groups.get(which)
        if g is None:
            first, second, nrows = self._ORDER[which]
            key = self.idx[which]
            if key is None:  # identity: one triple per row, in order
                g = Group(None, self.idx[first], self.idx[second])
            else:
                rowptr, perm = csr_of(key, getattr(self, nrows), which in self.sorted_by)
                g = Group(rowptr, _take(self.idx[first], perm), _take(self.idx[second], perm))
            self._groups[which] = g
        return g

    def inv_count(self) -> Tensor:
        """1 / max(#triples of each output row, 1): the mean-backward scale."""
        if self._inv is None:
            g = self.group("a")
            if g.rowptr is None:
                self._inv = torch.ones((self.n_out,), dtype=torch.float32,
                                       device=self._device())
            else:
                self._inv = torch.ops.pygho_b200.inv_count(g.rowptr)
        return self._inv

    def _device(self):
        for v in self.idx.values():
            if v is not None:
                return v.device
        raise RuntimeError("plan without index arrays")

    def swapped(self) -> "TriplePlan":
        """Same triples with the roles of the two operands exchanged."""
        if self._swapped is None:
            s = TriplePlan(self.T, self.n_out, self.n_b, self.n_a, self.idx["a"], self.idx["d"],
                           self.idx["c"], self.sorted_by.replace("c", "#").replace("d", "c")
                           .replace("#", "d"))
            s._swapped = self
            rename = {"a": "a", "c": "d", "d": "c"}
            for k, g in self._groups.items():
                s._groups[rename[k]] = Group(g.rowptr, g.second, g.first) if k == "a" else g
            s._inv = self._inv
            self._swapped = s
        return self._swapped

    def transposed(self) -> "TriplePlan":
        """Exchange the roles of output rows and operand-A rows (pooling <-> un-pooling);
        shares the sorted groupings with ``self``."""
        t = getattr(self, "_transposed", None)
        if t is None:
            flip = {"a": "c", "c": "a", "d": "d"}
            t = TriplePlan(self.T, self.n_a, self.n_out, self.n_b, self.idx["c"], self.idx["a"],
                           self.idx["d"], "".join(flip[k] for k in self.sorted_by))
            t._groups = _TransposedGroups(self)
            t._transposed = self
            self._transposed = t
        return t

    def prefetch(self, backward: bool = True) -> "TriplePlan":
        self.group("a")
        if backward:
            self.group("c")
            self.group("d")
        return self


class _TransposedGroups(dict):
    """Group cache of a transposed plan: builds through the parent so both share sorts."""

    _FLIP = {"a": "c", "c": "a", "d": "d"}

    def __init__(self, parent: TriplePlan):
        super().__init__()
        self.parent = parent

    def get(self, which, default=None):
        if which in self:
            return self[which]
        g = self.parent.group(self._FLIP[which])
        if which == "d":  # parent order (a, c) -> ours (a', c') = (c, a)
            g = Group(g.rowptr, g.second, g.first)
        self[which] = g
        return g


def _cache(t: Tensor) -> dict:
    c = getattr(t, "_pgh_cache", None)
    if c is None:
        c = {}
        t._pgh_cache = c
    return c


def plan_from_acd(acd: Tensor, n_out: int, n_a: int, n_b: int, build_all: bool = False
                  ) -> TriplePlan:
    """Plan of a reference-format ``acd``/``bcd`` LongTensor (3, T); cached on ``acd``.
    ``acd[0]`` is not assumed sorted (a stable sort puts it in CSR order either way).
    ``build_all``: also build the three CSR groupings now, with ONE library call
    (``pgh_acd_regroup``) instead of ~30 small operations -- what a training step needs anyway
    (forward: by a, gradients: by c and by d); the batch feeders ask for it."""
    cache = _cache(acd)
    key = ("acd", int(n_out), int(n_a), int(n_b))
    plan = cache.get(key)
    if plan is None:
        if acd.ndim != 2 or acd.shape[0] != 3:
            raise ValueError("acd must have shape (3, T)")
        _lib.require_cuda(acd)
        acd = acd.contiguous()
        if _CHECK and acd.numel():
            lim = torch.tensor([[n_out], [n_a], [n_b]], device=acd.device)
            assert bool(((acd >= 0) & (acd < lim)).all()), "acd index out of range"
        if build_all and acd.dtype == torch.int64:
            plan = _regroup_all(acd, int(n_out), int(n_a), int(n_b))
        else:
            plan = TriplePlan(acd.shape[1], n_out, n_a, n_b, to_i32(acd[0]), to_i32(acd[1]),
                              to_i32(acd[2]))
        cache[key] = plan
    if build_all:
        plan.prefetch(True)
    return plan


def _regroup_all(acd: Tensor, n_out: int, n_a: int, n_b: int) -> TriplePlan:
    """TriplePlan of an int64 (3, T) plan with all three groupings, one C-ABI call."""
    T = acd.shape[1]
    dev = acd.device
    idx = torch.empty((3, T), dtype=torch.int32, device=dev)
    # one allocation for the nine outputs: [rowptr_a | rowptr_c | rowptr_d | 6 x T]
    sizes = (n_out + 1, n_a + 1, n_b + 1) + (T,) * 6
    buf = torch.empty((sum(sizes),), dtype=torch.int32, device=dev)
    parts, off = [], 0
    for sz in sizes:
        parts.append(buf[off:off + sz])
        off += sz
    rp_a, rp_c, rp_d, f_a, s_a, f_c, s_c, f_d, s_d = parts
    ws = _ws(size_query("pgh_acd_regroup_ws_bytes", T), dev)
    _launch("pgh_acd_regroup", ptr(acd), T, n_out, n_a, n_b, 7, ptr(idx), ptr(rp_a), ptr(f_a),
            ptr(s_a), ptr(rp_c), ptr(f_c), ptr(s_c), ptr(rp_d), ptr(f_d), ptr(s_d), ptr(ws),
            ws.numel(), stream_ptr(dev))
    plan = TriplePlan(T, n_out, n_a, n_b, idx[0], idx[1], idx[2])
    plan._groups = {"a": Group(rp_a, f_a, s_a), "c": Group(rp_c, f_c, s_c),
                    "d": Group(rp_d, f_d, s_d)}
    return plan


def merge_groups(g1: Group, g2: Group, n_rows: int, stride: int, off1: int, off2: int) -> Group:
    """Row-wise concatenation of two CSR groupings over the same ``n_rows`` rows: row r of the
    result holds the entries of ``g1``'s row r followed by those of ``g2``'s row r.  The first
    index of every entry is remapped to ``stride * first + off`` (the two groupings read
    different column slices of ONE row-major buffer viewed as (stride * rows, width / stride)).
    Fixed-shape torch ops only (no size read-back): capacity-padded plans keep their filler
    entries behind ``rowptr[n_rows]`` of the result."""
    if g1.rowptr is None or g2.rowptr is None:
        raise ValueError("merge_groups needs CSR groupings")
    if g1.rowptr.is_cuda and all(t.dtype == torch.int32 for t in (g1.rowptr, g1.first, g1.second,
                                                                  g2.rowptr, g2.first, g2.second)):
        # one rowptr kernel + one entry kernel (binary search of the row) instead of ~14 torch ops
        T1, T2 = g1.first.numel(), g2.first.numel()
        dev = g1.rowptr.device
        rp = _empty(n_rows + 1, torch.int32, dev)
        first, second = _empty(T1 + T2, torch.int32, dev), _empty(T1 + T2, torch.int32, dev)
        _launch("pgh_merge_groups_i32", ptr(g1.rowptr.contiguous()), ptr(g1.first.contiguous()),
                ptr(g1.second.contiguous()), T1, ptr(g2.rowptr.contiguous()), ptr(g2.first.contiguous()),
                ptr(g2.second.contiguous()), T2, int(n_rows), int(stride), int(off1), int(off2),
                ptr(rp), ptr(first), ptr(second), stream_ptr(dev))
        return Group(rp, first, second)
    rp1, rp2 = g1.rowptr.to(torch.int64), g2.rowptr.to(torch.int64)
    T1, T2 = g1.first.numel(), g2.first.numel()
    dev = rp1.device
    t1 = torch.arange(T1, device=dev)
    t2 = torch.arange(T2, device=dev)
    r1 = torch.searchsorted(rp1[1:].contiguous(), t1, right=True)        # row of entry t (n_rows: filler)
    r2 = torch.searchsorted(rp2[1:].contiguous(), t2, right=True)
    pos1 = t1 + rp2[r1]                                   # entries of g2 in earlier rows
    pos2 = t2 + rp1[torch.clamp(r2 + 1, max=n_rows)]     # entries of g1 in rows <= r
    first = torch.zeros((T1 + T2,), dtype=torch.int32, device=dev)
    second = torch.zeros((T1 + T2,), dtype=torch.int32, device=dev)
    first[pos1] = g1.first * stride + off1
    first[pos2] = g2.first * stride + off2
    second[pos1] = g1.second
    second[pos2] = g2.second
    return Group((rp1 + rp2).to(torch.int32), first, second)


def sswl_bwd_group(acd_xa: Tensor, acd_ax: Tensor, ax_name: str, nX: int, nA: int) -> Group:
    """The gradient of an SSWL layer's tuple features in ONE segmented reduction
    (``ops.SswlAggregate.backward``): for tuple r, the entries of ``X (x) A`` in which r is the
    first operand followed by the entries of ``A (x) X`` in which r is the second operand.  The
    first index addresses the gradient of the concatenation ``[X, X(x)A, A(x)X]`` viewed as
    (3 nX, d) rows: 3 a + 1 / 3 a + 2; the second index is the row of A.  Cached on ``acd_xa``
    (``ax_name`` = the datadict key of ``acd_ax``: static batches rebuild it by name)."""
    cache = _cache(acd_xa)
    key = ("sswl_bwd", ax_name, int(nX), int(nA))
    hit = cache.get(key)
    if hit is None:
        if 3 * int(nX) + 2 >= 2 ** 31:
            raise ValueError("sswl_bwd_group: too many tuples for int32 row ids")
        gc = plan_from_acd(acd_xa, nX, nX, nA).group("c")     # first = a, second = d (row of A)
        gd = plan_from_acd(acd_ax, nX, nA, nX).group("d")     # first = a, second = c (row of A)
        hit = merge_groups(gc, gd, int(nX), 3, 1, 2)
        cache[key] = hit
    return hit


def plan_from_key(key: Tensor, n_rows: int, assume_sorted: bool = False) -> TriplePlan:
    """Pooling plan: value row t goes to output row ``key[t]`` (a = key, c = identity);
    its transpose is the un-pooling gather.  Cached on ``key``."""
    cache = _cache(key)
    ck = ("key", int(n_rows), bool(assume_sorted))
    plan = cache.get(ck)
    if plan is None:
        _lib.require_cuda(key)
        if _CHECK and key.numel():
            assert int(key.min()) >= 0 and int(key.max()) < n_rows, "index out of range"
        n = key.numel()
        plan = TriplePlan(n, n_rows, n, 0, to_i32(key), None, None,
                          "a" if assume_sorted else "")
        cache[ck] = plan
    return plan


# ------------------------------------------------------------------------------ hashing
def hash_bits(sparse_dim: int) -> int:
    return 63 // sparse_dim


def pack_keys(ind: Tensor, rows: Optional[Sequence[int]] = None, check: bool = False) -> Tensor:
    """Packed lexicographic key of the selected rows of an (sd, nnz) LongTensor."""
    _lib.require_cuda(ind)
    if ind.dtype != torch.int64:
        raise TypeError("indices must be int64 (LongTensor)")
    if ind.stride(1) != 1 and ind.shape[1] > 1:
        ind = ind.contiguous()
    rows = list(range(ind.shape[0])) if rows is None else list(rows)
    nnz = ind.shape[1]
    key = _empty(nnz, torch.int64, ind.device)
    info = torch.zeros((2,), dtype=torch.int32, device=ind.device) if check else None
    bits = hash_bits(len(rows)) if len(rows) > 1 else 63
    if nnz:
        _launch("pgh_pack_keys", ptr(ind), ind.stride(0), _host_i32(rows), len(rows), bits, nnz,
                ptr(key), ptr(info), stream_ptr(ind.device))
    if check and nnz:
        neg, big = info.tolist()
        assert neg == 0, "indice cannot be negative"
        assert big == 0, "too large indice, hash is not injective"
    return key


def unpack_keys(key: Tensor, sparse_dim: int) -> Tensor:
    _lib.require_cuda(key)
    key = key.contiguous()
    n = key.numel()
    out = torch.empty((sparse_dim, n), dtype=torch.int64, device=key.device)
    if n:
        _launch("pgh_unpack_keys", ptr(key), n, int(sparse_dim),
                hash_bits(sparse_dim) if sparse_dim > 1 else 63, ptr(out), n,
                stream_ptr(key.device))
    return out


def pack_tight(ind: Tensor, dims: Sequence[int], rows: Optional[Sequence[int]] = None,
               check: bool = False) -> Tensor:
    _lib.require_cuda(ind)
    if ind.stride(1) != 1 and ind.shape[1] > 1:
        ind = ind.contiguous()
    rows = list(range(ind.shape[0])) if rows is None else list(rows)
    assert len(rows) == len(dims), "indice dim and dim size not match"
    nnz = ind.shape[1]
    key = _empty(nnz, torch.int64, ind.device)
    info = torch.zeros((2,), dtype=torch.int32, device=ind.device) if check else None
    if nnz:
        _launch("pgh_pack_tight", ptr(ind), ind.stride(0), _host_i32(rows), _host_i64(dims),
                len(rows), nnz, ptr(key), ptr(info), stream_ptr(ind.device))
    if check and nnz:
        assert info.tolist()[0] == 0, "indice exceeds dimsize"
    return key


def unpack_tight(key: Tensor, dims: Sequence[int]) -> Tensor:
    _lib.require_cuda(key)
    key = key.contiguous()
    n = key.numel()
    out = torch.empty((len(dims), n), dtype=torch.int64, device=key.device)
    if n:
        _launch("pgh_unpack_tight", ptr(key), n, _host_i64(dims), len(dims), ptr(out), n,
                stream_ptr(key.device))
    return out


def is_sorted(key: Tensor, strict: bool = False) -> bool:
    """Host-synchronising check (debug / assert paths only)."""
    info = torch.zeros((1,), dtype=torch.int32, device=key.device)
    key = key.contiguous()
    if key.numel() > 1:
        _launch("pgh_check_sorted_i64", ptr(key), key.numel(), int(strict), ptr(info),
                stream_ptr(key.device))
    return int(info.item()) == 0


def lookup_sorted(tkeys: Tensor, keys: Tensor) -> Tensor:
    """Position (int32) of each key in the sorted unique ``tkeys`` or -1."""
    pos = _empty(keys.numel(), torch.int32, keys.device)
    if keys.numel():
        _launch("pgh_lookup_sorted", ptr(tkeys), tkeys.numel(), ptr(keys), keys.numel(),
                ptr(pos), stream_ptr(keys.device))
    return pos


# --------------------------------------------------------------- contraction plans
def _expand_matches(ind1: Tensor, dim1: int, ind2: Tensor, dim2: int, k2_sorted: bool):
    """All (p, q) with ind1[dim1, p] == ind2[dim2, q], ordered by p then by position of q
    in the key-sorted ind2.  Returns (c int32, d int32, T0).  One host sync (T0)."""
    dev = _lib.require_cuda(ind1, ind2)
    nnz1 = ind1.shape[1]
    k1 = ind1[dim1].contiguous()
    k2 = ind2[dim2].contiguous()
    perm2 = None
    if not k2_sorted:
        # keys are node ids; sort on as many bits as the largest possible id needs
        k2, perm2 = sort_keys(k2, 63)
    lo = _empty(nnz1, torch.int32, dev)
    off = _empty(nnz1 + 1, torch.int64, dev)
    ws = _ws(size_query("pgh_match_ws_bytes", nnz1), dev)
    _launch("pgh_match_ranges", ptr(k2), k2.numel(), ptr(k1), nnz1, ptr(lo), ptr(off), ptr(ws),
            ws.numel(), stream_ptr(dev))
    total = int(off[-1].item())
    c, d = _empty(total, torch.int32, dev), _empty(total, torch.int32, dev)
    if total:
        _launch("pgh_expand_pairs", ptr(off), ptr(lo), ptr(perm2), nnz1, total, ptr(c), ptr(d),
                stream_ptr(dev))
    return c, d, total


def _pair_keys(ind1, dim1, ind2, dim2, c, d) -> Tensor:
    sd_out = ind1.shape[0] + ind2.shape[0] - 2
    if sd_out < 1:
        raise ValueError("contraction leaves no sparse dimension")
    ind1 = ind1 if ind1.stride(1) == 1 else ind1.contiguous()
    ind2 = ind2 if ind2.stride(1) == 1 else ind2.contiguous()
    key = _empty(c.numel(), torch.int64, c.device)
    if c.numel():
        _launch("pgh_pair_keys", ptr(ind1), ind1.stride(0), ind1.shape[0], int(dim1), ptr(ind2),
                ind2.stride(0), ind2.shape[0], int(dim2), ptr(c), ptr(d), c.numel(),
                hash_bits(sd_out) if sd_out > 1 else 63, ptr(key), None, stream_ptr(c.device))
    return key


def spspmm_ind_i32(ind1: Tensor, dim1: int, ind2: Tensor, dim2: int, k2_sorted: bool):
    """Device build of the contraction plan.  Returns (tarind int64 (sd_out, nnzP),
    b int32, c int32, d int32) with the triples sorted by (b, c, d-position)."""
    sd_out = ind1.shape[0] + ind2.shape[0] - 2
    c, d, total = _expand_matches(ind1, dim1, ind2, dim2, k2_sorted)
    key = _pair_keys(ind1, dim1, ind2, dim2, c, d)
    end_bit = hash_bits(sd_out) * sd_out if sd_out > 1 else 63
    ks, permT = sort_keys(key, end_bit)
    ukey, seg, _count = unique_sorted(ks)
    tarind = unpack_keys(ukey, sd_out)
    if total:
        c, d = gather_i32(c, permT), gather_i32(d, permT)
    return tarind, seg, c, d


def filter_triples(tar_ind: Tensor, ind: Tensor, b: Tensor, c: Tensor, d: Tensor, check: bool):
    """Hadamard filter of a plan onto the pattern ``tar_ind`` (filterind); keeps order."""
    dev = _lib.require_cuda(tar_ind, ind)
    tkey = pack_keys(tar_ind, check=check)
    if check:
        assert is_sorted(tkey, strict=True), "tar_ind should be sorted and coalesce"
    b2a = lookup_sorted(tkey, pack_keys(ind, check=check))
    n = b.numel()
    oa, oc, od = (_empty(n, torch.int32, dev) for _ in range(3))
    cnt = torch.zeros((1,), dtype=torch.int32, device=dev)
    if n:
        ws = _ws(size_query("pgh_compact_ws_bytes", n), dev)
        _launch("pgh_compact_triples", ptr(b), ptr(b2a), ptr(c), ptr(d), n, ptr(oa), ptr(oc),
                ptr(od), ptr(cnt), ptr(ws), ws.numel(), stream_ptr(dev))
    T = int(cnt.item()) if n else 0
    return oa[:T], oc[:T], od[:T]


def filtered_plan(tar_ind: Tensor, ind1: Tensor, dim1: int, ind2: Tensor, dim2: int,
                  k2_sorted: bool = False) -> Tuple[Tensor, TriplePlan]:
    """Fused ``filterind(tar_ind, *spspmm_ind(ind1, dim1, ind2, dim2))`` that never
    materialises the unfiltered product pattern: expand matches, look each output
    coordinate up in ``tar_ind`` directly, compact, sort by output row.
    Returns (acd int64 (3, T) in canonical order, its TriplePlan).  Two host syncs."""
    dev = _lib.require_cuda(tar_ind, ind1, ind2)
    c, d, total = _expand_matches(ind1, dim1, ind2, dim2, k2_sorted)
    key = _pair_keys(ind1, dim1, ind2, dim2, c, d)
    a = lookup_sorted(pack_keys(tar_ind), key)
    oa, oc, od = (_empty(total, torch.int32, dev) for _ in range(3))
    cnt = torch.zeros((1,), dtype=torch.int32, device=dev)
    if total:
        ws = _ws(size_query("pgh_compact_ws_bytes", total), dev)
        _launch("pgh_compact_triples", ptr(a), None, ptr(c), ptr(d), total, ptr(oa), ptr(oc),
                ptr(od), ptr(cnt), ptr(ws), ws.numel(), stream_ptr(dev))
    T = int(cnt.item()) if total else 0
    oa, oc, od = oa[:T].contiguous(), oc[:T].contiguous(), od[:T].contiguous()
    n_out = tar_ind.shape[1]
    rowptr, perm = csr_of(oa, n_out)
    if perm is not None:
        oa, oc, od = gather_i32(oa, perm), gather_i32(oc, perm), gather_i32(od, perm)
    plan = TriplePlan(T, n_out, ind1.shape[1], ind2.shape[1], oa, oc, od, sorted_by="a")
    plan._groups["a"] = Group(rowptr, oc, od)
    acd = torch.stack((to_i64(oa), to_i64(oc), to_i64(od))) if T else \
        torch.zeros((3, 0), dtype=torch.int64, device=dev)
    _cache(acd)[("acd", n_out, ind1.shape[1], ind2.shape[1])] = plan
    return acd, plan


# ------------------------------------------------------------------------- embedding tables
class EmbeddingPlan(NamedTuple):
    """Index structures of one ``nn.Embedding`` lookup (``idx`` -> rows of the table), built
    once per index tensor and cached on it:

    * ``idx32``: the indices as int32 (forward gather);
    * ``perm``: stable sort of the positions by index value;
    * ``levels``: row pointers of a reduction tree.  Level 0 cuts the sorted positions into
      chunks of at most ``chunk`` entries that never straddle two index values, every further
      level does the same with the partial sums of the level before, the last one has exactly
      ``num_embeddings`` rows.  All sizes are static (V + ceil(n / chunk) per level), so
      building the plan needs no host synchronisation.  The weight gradient is then a chain of
      segmented sums in a fixed order: deterministic, no atomics, no per-step sort."""
    idx32: Tensor
    perm: Tensor
    levels: Tuple[Tensor, ...]
    num_embeddings: int


def embedding_plan(idx: Tensor, num_embeddings: int, chunk: int = 64) -> EmbeddingPlan:
    cache = _cache(idx)
    ck = ("embedding", int(num_embeddings), int(chunk))
    hit = cache.get(ck)
    if hit is not None:
        return hit
    dev = _lib.require_cuda(idx)
    flat = idx.reshape(-1)
    n, V = flat.numel(), int(num_embeddings)
    if n and flat.dtype in (torch.int64, torch.int32) and V < (1 << 24):
        # one library call: a 32-bit radix sort + one small kernel per level of the tree
        flat = flat.contiguous()
        sizes, size = [], n
        while size > max(2 * V, 4 * chunk):
            size = V + (size + chunk - 1) // chunk
            sizes.append(size + 1)
        sizes.append(V + 1)
        idx32 = _empty(n, torch.int32, dev)
        perm = _empty(n, torch.int32, dev)
        lv = _empty(sum(sizes), torch.int32, dev)
        bws = _empty(2 * (V + 1), torch.int32, dev)
        ws = _ws(size_query("pgh_embedding_plan_ws_bytes", n), dev)
        _launch("pgh_embedding_plan", ptr(flat), int(flat.dtype == torch.int64), n, V, int(chunk),
                ptr(idx32), ptr(perm), ptr(lv), lv.numel(), ptr(bws), ptr(ws), ws.numel(),
                stream_ptr(dev))
        levels, off = [], 0
        for sz in sizes:
            levels.append(lv[off:off + sz])
            off += sz
        plan = EmbeddingPlan(idx32, perm, tuple(levels), V)
        cache[ck] = plan
        return plan
    idx32 = to_i32(flat)
    rowptr_id, perm = csr_of(idx32, V)                 # positions grouped by index value
    if perm is None:
        perm = torch.arange(n, dtype=torch.int32, device=dev)
    levels = []
    bounds, size = rowptr_id, n                        # id boundaries in units of the current level
    while size > max(2 * V, 4 * chunk):
        cuts = torch.arange(0, size, chunk, dtype=torch.int32, device=dev)
        starts = torch.sort(torch.cat([bounds[:V], cuts])).values
        rows = starts.numel()
        levels.append(torch.cat([starts, bounds[V:V + 1]]).contiguous())
        # chunk k belongs to the index value whose range contains its start
        bounds = torch.searchsorted(starts, bounds[:V], right=False).to(torch.int32)
        bounds = torch.cat([bounds, torch.full((1,), rows, dtype=torch.int32, device=dev)])
        size = rows
    levels.append(bounds.contiguous())
    plan = EmbeddingPlan(idx32, perm, tuple(levels), V)
    cache[ck] = plan
    return plan
