"""Host batch -> device ``datadict`` (the contract of reference ``hodata/SpData.py:80-112``
/ ``MaData.py:200-255`` + ``Wrapper.py:90-98``), PyG-free.

``sp_datadict`` wraps the concatenated index arrays into ``SparseTensor`` objects and
makes sure every requested ``<key>___acd`` plan exists: either the host batch already
carries it (the reference precomputes plans per graph on the CPU and ships them with
every batch) or it is built on the device by the fused plan kernels."""
from __future__ import annotations

import queue
import sys
import threading
from typing import Dict, Iterable, Optional

import numpy as np
import torch

from .. import plans as P
from ..backend.MaTensor import MaskedTensor
from ..backend.SpTensor import SparseTensor
from ..honn.SpOperator import KEYSEP
from .synthetic import HostBatch


def parse_key(key: str):
    """``op0___op1___dim1___op2___dim2`` (reference hodata/SpData.py:34-53)."""
    parts = key.split(KEYSEP)
    assert len(parts) == 5, "key format not match"
    op0, op1, dim1, op2, dim2 = parts
    for op in (op0, op1, op2):
        if not (op == "A" or op.startswith("X")):
            raise NotImplementedError(f"operator name {op} not implemented now")
    return op0, op1, int(dim1), op2, int(dim2)


def _h2d(arr: np.ndarray, device, pinned: Optional[Dict[int, tuple]] = None):
    """Asynchronous copy of a host array; ``pinned`` caches the page-locked staging copy per
    array OBJECT (the entry keeps the array alive, so a recycled id() can never alias it)."""
    t = torch.from_numpy(arr)
    if pinned is not None:
        hit = pinned.get(id(arr))
        if hit is None or hit[0] is not arr:
            hit = (arr, t.pin_memory())
            pinned[id(arr)] = hit
        t = hit[1]
    return t.to(device, non_blocking=True)


def pin_host_batch(hb: HostBatch, pinned: dict) -> None:
    """Page-lock every array of a host batch (incl. its plans) ahead of time."""
    arrs = [hb.x, hb.edge_index, hb.edge_attr, hb.tupleid, hb.tuplefeat, hb.batch, hb.y]
    arrs += list(hb.plans.values())
    if getattr(hb, "valid", None) is not None:
        arrs.append(hb.valid)
    for a in arrs:
        if id(a) not in pinned or pinned[id(a)][0] is not a:
            pinned[id(a)] = (a, torch.from_numpy(a).pin_memory())


def sp_datadict(hb: HostBatch, device, keys: Iterable[str] = (),
                pinned: Optional[dict] = None) -> dict:
    """Copy a host batch to ``device`` and assemble the sparse-mode ``datadict``."""
    N = hb.num_nodes
    ei = _h2d(hb.edge_index, device, pinned)
    tid = _h2d(hb.tupleid, device, pinned)
    ea = _h2d(hb.edge_attr, device, pinned)
    tf = _h2d(hb.tuplefeat, device, pinned)
    sd = tid.shape[0]
    dd = {
        "x": _h2d(hb.x, device, pinned),
        "A": SparseTensor(ei, ea, (N, N) + tuple(ea.shape[1:]), is_coalesced=True),
        "X": SparseTensor(tid, tf, (N,) * sd + tuple(tf.shape[1:]), is_coalesced=True),
        "batch": _h2d(hb.batch, device, pinned),
        "num_graphs": hb.num_graphs,
        "y": _h2d(hb.y, device, pinned),
    }
    if getattr(hb, "valid", None) is not None:     # capacity-padded batch (pygho_b200/static.py)
        dd["valid_rows"] = _h2d(hb.valid, device, pinned)
    for key in keys:
        name = key + KEYSEP + "acd"
        if key in hb.plans:
            dd[name] = _h2d(hb.plans[key], device, pinned)
            continue
        op0, op1, dim1, op2, dim2 = parse_key(key)
        pick = lambda op: ei if op == "A" else tid  # noqa: E731
        acd, _plan = P.filtered_plan(pick(op0), pick(op1), dim1, pick(op2), dim2,
                                     k2_sorted=(dim2 == 0))
        dd[name] = acd
    return dd


def prefetch_plans(datadict: dict, keys: Iterable[str], backward: bool = True,
                   embeddings: Optional[Dict[str, int]] = None) -> None:
    """Build (and cache on the ``acd`` tensors) the CSR groupings the kernels will ask for,
    so that the first layer of the model does not pay for them.  ``embeddings`` maps datadict
    entries holding integer labels ("x", "A", "X") to the size of the embedding table that
    encodes them: their :class:`pygho_b200.plans.EmbeddingPlan` is built here too."""
    for name, num in (embeddings or {}).items():
        t = datadict[name]
        t = t.values if isinstance(t, SparseTensor) else t
        if t is not None and t.is_cuda and t.dtype in (torch.int64, torch.int32) and t.numel():
            P.embedding_plan(t, int(num))
    nX, nA = datadict["X"].nnz, datadict["A"].nnz
    for key in keys:
        _op0, op1, _d1, op2, _d2 = parse_key(key)
        n1 = nA if op1 == "A" else nX
        n2 = nA if op2 == "A" else nX
        P.plan_from_acd(datadict[key + KEYSEP + "acd"], nX, n1, n2, build_all=backward).prefetch(backward)
    # the merged gradient plan of the SSWL layers (both products' entries per tuple)
    k_xa, k_ax = "X___X___1___A___0" + KEYSEP + "acd", "X___A___1___X___0" + KEYSEP + "acd"
    if backward and k_xa in datadict and k_ax in datadict and nX and nA:
        P.sswl_bwd_group(datadict[k_xa], datadict[k_ax], k_ax, nX, nA)


class DevicePrefetcher:
    """Double-buffered host -> device feeding (the role of the reference's
    ``IterWrapper``: ``.to(device)`` + batch transform, hodata/Wrapper.py:90-98).

    ``next()`` returns the datadict of the current batch and immediately issues, on a side
    stream, the pinned-memory copies, SparseTensor wrapping and CSR regrouping of the NEXT
    batch, so they overlap the training step that is about to be launched.

    The side stream never waits for the compute stream: everything it touches is allocated
    on it (its own allocator pool), and a batch's buffers only go back to that pool in
    ``advance()`` one step after the batch was consumed -- by which time the caller has
    synchronised with that step (see ``advance``).

    With ``threaded=True`` (default) the enqueueing itself (a few dozen small launches and
    their Python glue, ~4 ms of host time per batch) runs on a worker thread, like a
    DataLoader's pin-memory thread: the training step is launch-bound on the host
    (profiles/r1_graph_probe.json: 14.8 ms of host time per 16.4 ms step), so host work on
    the main thread would extend every step.  CUDA calls and the C-ABI kernels release the
    GIL while they run."""

    def __init__(self, host_batches, device, keys, pinned: Optional[dict] = None,
                 threaded: bool = True, embeddings: Optional[Dict[str, int]] = None):
        self.hbs, self.device, self.keys = list(host_batches), device, list(keys)
        self.embeddings = dict(embeddings or {})
        self.pinned = {} if pinned is None else pinned
        self.stream = torch.cuda.Stream(device)
        self.pos = 0
        self._ready = self._inflight = None
        self._error = None
        self._done = threading.Event()
        self._jobs: Optional[queue.Queue] = None
        if threaded:
            # The main thread releases the GIL around every kernel launch (ctypes, torch ops);
            # with CPython's default 5 ms switch interval each of those hand-overs can park it
            # behind the worker's Python code for milliseconds (convoy effect: e2e steps of
            # 26 ms instead of 14 ms were measured).  A 50 us interval keeps hand-overs short.
            if sys.getswitchinterval() > 1e-4:
                sys.setswitchinterval(5e-5)
            self._jobs = queue.Queue()
            self._worker = threading.Thread(target=self._run, name="pygho-prefetch", daemon=True)
            self._worker.start()
        self._submit()

    # -- the actual work: runs on the worker thread (or inline when not threaded)
    def _issue(self, hb):
        with torch.cuda.stream(self.stream):
            dd = sp_datadict(hb, self.device, self.keys, self.pinned)
            prefetch_plans(dd, self.keys, embeddings=self.embeddings)
        return dd

    def _run(self):
        torch.cuda.set_device(self.device)
        while True:
            hb = self._jobs.get()
            if hb is None:
                return
            try:
                self._ready = self._issue(hb)
            except BaseException as e:  # noqa: BLE001 - re-raised in get()
                self._error = e
            self._done.set()

    def _submit(self):
        hb = self.hbs[self.pos % len(self.hbs)]
        self.pos += 1
        self._done.clear()
        if self._jobs is not None:
            self._jobs.put(hb)
        else:
            self._ready = self._issue(hb)
            self._done.set()

    def get(self) -> dict:
        """Datadict of the current batch (waits, on the device, for its copies)."""
        self._done.wait()
        if self._error is not None:
            err, self._error = self._error, None
            raise err
        torch.cuda.current_stream(self.device).wait_stream(self.stream)
        return self._ready

    def advance(self) -> None:
        """Issue the next batch's copies and plan regrouping on the side stream.  Call it
        right after the training step has been launched: the host work overlaps the step's
        execution.  The caller must synchronise with the step BEFORE the one just launched
        (e.g. read its loss back) before calling this: the buffers of that older batch are
        released here and reused."""
        from ..static import release_datadict
        release_datadict(self._inflight)        # free the older batch now, not at the next GC
        self._inflight = self._ready
        self._submit()

    def next(self) -> dict:
        """``get()`` + ``advance()`` for simple loops.  Safe without any caller-side fence: it
        first waits (on the host) for everything queued on the compute stream so far -- i.e. for
        the step that consumed the batch whose buffers ``advance()`` is about to recycle."""
        torch.cuda.current_stream(self.device).synchronize()
        dd = self.get()
        self.advance()
        return dd

    def close(self) -> None:
        if self._jobs is not None:
            self._jobs.put(None)
            self._worker.join(timeout=5)
            self._jobs = None


class DeferredScalar:
    """Read a device scalar (the loss) ONE step late: ``push(t)`` copies ``t`` to pinned host
    memory behind an event and returns the value pushed the call before, waiting only for
    that older event -- the host never blocks on the step it has just launched.  The wait is
    also the fence :meth:`DevicePrefetcher.advance` asks for."""

    def __init__(self):
        self._buf = torch.zeros(2, dtype=torch.float32).pin_memory()
        self._evt = [torch.cuda.Event(), torch.cuda.Event()]
        self._n = 0
        self._unread: Optional[int] = None

    def _read(self, slot: Optional[int]) -> Optional[float]:
        if slot is None:
            return None
        self._evt[slot].synchronize()
        return float(self._buf[slot])

    def push(self, value: torch.Tensor) -> Optional[float]:
        slot = self._n & 1
        self._n += 1
        self._buf[slot:slot + 1].copy_(value.detach().reshape(1).float(), non_blocking=True)
        self._evt[slot].record()
        prev, self._unread = self._unread, slot
        return self._read(prev)

    def flush(self) -> Optional[float]:
        """Value of the last ``push`` (None if it has been returned already)."""
        prev, self._unread = self._unread, None
        return self._read(prev)


def attach_host_plans(hb: HostBatch, datadict: dict, keys: Iterable[str]) -> None:
    """Copy the device-built plans back into the host batch (done once per batch when a
    dataset is prepared), so later epochs ship them like the reference's loader does."""
    for key in keys:
        hb.plans[key] = datadict[key + KEYSEP + "acd"].cpu().numpy()


def ma_datadict(hb: HostBatch, device, max_dist: int = 5, tuples: str = "khop",
                pinned: Optional[dict] = None) -> dict:
    """Dense-mode ``datadict``: x (b, n, 1), A (b, n, n), X (b, n, n) masked tensors padded
    to the largest graph (reference hodata/MaData.py:109-255 ``to_dense_*`` / ``batch2dense``).

    The host batch is copied in its sparse form and padded ON THE DEVICE (pad / scatter
    kernels of ``hodata.cu``).  ``tuples="khop"``: X holds ``min(dist, max_dist) + 1`` on the
    sampled k-hop tuples and 0 elsewhere; ``tuples="spd"``: X is the shortest-path-distance
    matrix clamped to ``max_dist + 1``, computed on the device (``spdsampler``);
    ``tuples="rd"``: X is the float32 resistance-distance matrix (``rdsampler``)."""
    from .MaData import to_dense_adj, to_dense_x
    from .MaTupleSampler import rdsampler, spdsampler
    B = hb.num_graphs
    n = int(np.diff(hb.node_ptr).max())
    node_ptr = _h2d(hb.node_ptr, device, pinned)
    batch = _h2d(hb.batch, device, pinned)
    ei = _h2d(hb.edge_index, device, pinned)
    x = to_dense_x(_h2d(hb.x, device, pinned).unsqueeze(-1), node_ptr, n, B)
    A = to_dense_adj(ei, batch[ei[0]], _h2d(hb.edge_attr, device, pinned), n, B,
                     node_ptr=node_ptr)
    m2 = x.mask.unsqueeze(2) & x.mask.unsqueeze(1)
    if tuples == "spd":
        X = spdsampler(ei, hb.node_ptr, max_dist, n)
    elif tuples == "rd":
        X = rdsampler(ei, hb.node_ptr, n)
    else:
        tid = _h2d(hb.tupleid, device, pinned)
        feat = torch.clamp(_h2d(hb.tuplefeat, device, pinned), max=max_dist) + 1
        X = MaskedTensor(to_dense_adj(tid, batch[tid[0]], feat, n, B, node_ptr=node_ptr).data,
                         m2, 0, True)
    return {
        "x": x,
        "A": MaskedTensor(A.data, m2, 0, True),
        "X": X,
        "num_graphs": B,
        "y": _h2d(hb.y, device, pinned),
    }
