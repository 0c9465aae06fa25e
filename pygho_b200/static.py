"""Static-capacity batches: ONE captured CUDA graph trains on batches of different sizes.

A sparse-mode batch is a handful of index arrays whose lengths change from batch to batch
(nodes, edges, tuples, plan triples), so an eager training step re-launches ~400 kernels per
step and is bound by the host as soon as the per-GPU batch is small (128 graphs per GPU at the
8-GPU strong-scaling point: 1.7 ms of device work behind 10 ms of Python).  Here every array
is padded, at collate time, to a fixed *capacity* and the pads are built so that they are inert:

* pad nodes / edges / tuples sit at the END of their arrays; pad edges and tuples point at the
  last pad node, pad nodes belong to one extra "dummy" graph (``num_graphs = B + 1``);
* pad plan triples are (n_out, n_a, n_b): one past the last row of each array.  A CSR grouping
  built by a stable sort puts them after ``rowptr[n_rows]``, i.e. into NO row: the kernels
  never visit them (they only walk ``[rowptr[r], rowptr[r + 1])``), so a padded batch costs
  the segmented-reduce kernels exactly what the exact-size batch costs and no row gets long;
* the fused BatchNorm kernels take the number of VALID rows from device memory
  (``rows_dev``, csrc/fused_mlp.cu): pad rows are excluded from the statistics, get output 0
  and gradient 0, so no weight gradient ever sees them;
* the loss is taken over the first B graphs.

All shapes being equal, the device-side plan builders produce arrays of equal shapes for every
batch; ``StaticSlot.load`` rebuilds them on a side stream and copies them over the arrays the
captured graph reads.  Two slots alternate, so batch i+1 is loaded while the graph of batch i
runs; the host only enqueues copies, ~60 small integer kernels and one graph launch per step.

Scope: sparse mode with 2-D tuples (SSWL, NGNN, DSSGNN, PPGN-sparse) and MLPs whose blocks are
Linear -> BatchNorm -> SiLU/ReLU (the fused path); anything that needs a data-dependent output
size inside the step (3-D pooling to a sparse pattern) is rejected.
"""
from __future__ import annotations

import os
import threading
import time
from contextlib import contextmanager
from dataclasses import replace
from typing import Dict, Iterable, List, Optional, Sequence

import numpy as np
import torch

from . import plans as P
from .backend.SpTensor import SparseTensor
from .hodata.synthetic import HostBatch

KEYSEP = "___"
_ACTIVE: Optional[Dict[int, torch.Tensor]] = None


def rows_dev_for(n_rows: int) -> Optional[torch.Tensor]:
    """Device int32 scalar with the valid-row count of the ``n_rows``-row tensors of the active
    static batch, or None (not in static mode / not a padded row count)."""
    if _ACTIVE is None:
        return None
    return _ACTIVE.get(int(n_rows))


@contextmanager
def static_shapes(datadict: dict):
    """Make the BatchNorm blocks run inside see the valid-row counts of ``datadict`` (a padded
    batch made by :func:`pad_host_batch`); a no-op for ordinary batches."""
    global _ACTIVE
    prev = _ACTIVE
    reg = datadict.get("_rows_registry")
    _ACTIVE = reg if reg else prev
    try:
        yield
    finally:
        _ACTIVE = prev


# ------------------------------------------------------------------------- host side
def _parse(key: str):
    _o0, o1, d1, o2, d2 = key.split(KEYSEP)
    return o1, int(d1), o2, int(d2)


def capacities(host_batches: Iterable[HostBatch], keys: Sequence[str], margin: float = 0.0) -> dict:
    """Smallest capacities that fit every batch (+ ``margin``), each with at least one pad row."""
    hbs = list(host_batches)

    def cap(vals):
        m = int(np.ceil(max(vals) * (1.0 + margin))) + 1
        return (m + 7) // 8 * 8

    caps = {"N": cap([hb.num_nodes for hb in hbs]), "A": cap([hb.edge_index.shape[1] for hb in hbs]),
            "X": cap([hb.tupleid.shape[1] for hb in hbs]), "B": max(hb.num_graphs for hb in hbs)}
    for key in keys:
        caps[key] = cap([hb.plans[key].shape[1] for hb in hbs])
    sizes = sorted([caps["N"], caps["A"], caps["X"], caps["B"] + 1])
    while len(set(sizes)) != 4:      # row counts double as registry keys: keep them distinct
        caps["N"] += 8
        sizes = sorted([caps["N"], caps["A"], caps["X"], caps["B"] + 1])
    return caps


def pad_host_batch(hb: HostBatch, caps: dict, keys: Sequence[str],
                   fewer_graphs: bool = False) -> HostBatch:
    """Pad a collated batch (with its host plans) to ``caps``; see the module docstring.

    ``fewer_graphs``: accept a batch of ``B < caps["B"]`` graphs; graphs ``B .. caps["B"] - 1``
    are then empty and the dummy graph is ``caps["B"]``.  For evaluation only (the graph rows
    are read back as ``[:B]``): a training loss over ``num_valid_graphs`` would count the empty
    graphs."""
    if hb.tupleid.shape[0] != 2:
        raise NotImplementedError("static batches support 2-D tuples")
    N, nA, nX, B = hb.num_nodes, hb.edge_index.shape[1], hb.tupleid.shape[1], hb.num_graphs
    Nc, Ac, Xc, Bc = caps["N"], caps["A"], caps["X"], caps["B"]
    if not (B == Bc or (fewer_graphs and B < Bc)) or N >= Nc or nA >= Ac or nX >= Xc:
        raise ValueError("batch does not fit the capacities (every array needs >= 1 pad row)")

    def pad1(a, n, value):
        out = np.full((n,) + a.shape[1:], value, dtype=a.dtype)
        out[:a.shape[0]] = a
        return out

    def pad2(a, n, value):
        out = np.full((a.shape[0], n), value, dtype=a.dtype)
        out[:, :a.shape[1]] = a
        return out

    n_rows = {"A": (nA, Ac), "X": (nX, Xc)}
    plans = {}
    for key in keys:
        acd = hb.plans[key]
        T, Tc = acd.shape[1], caps[key]
        if T > Tc:
            raise ValueError(f"plan {key} has {T} triples, capacity {Tc}")
        o1, _d1, o2, _d2 = _parse(key)
        ops = ["A" if o == "A" else "X" for o in (o1, o2)]
        out = np.empty((3, Tc), np.int64)
        out[:, :T] = acd
        out[0, T:] = Xc                         # "no row" markers (see the module docstring)
        out[1, T:] = n_rows[ops[0]][1]
        out[2, T:] = n_rows[ops[1]][1]
        plans[key] = out
    padded = replace(
        hb, num_graphs=Bc + 1, num_nodes=Nc,
        x=pad1(hb.x, Nc, 0), edge_index=pad2(hb.edge_index, Ac, Nc - 1),
        edge_attr=pad1(hb.edge_attr, Ac, 0), tupleid=pad2(hb.tupleid, Xc, Nc - 1),
        tuplefeat=pad1(hb.tuplefeat, Xc, 0), batch=pad1(hb.batch, Nc, Bc), y=pad1(hb.y, Bc + 1, 0.0),
        plans=plans)
    padded.valid = np.array([nX, N, B], dtype=np.int32)
    return padded


def attach_registry(dd: dict, caps: dict) -> dict:
    """Row-capacity -> device valid-count scalar, stored in the datadict."""
    v = dd["valid_rows"]
    dd["_rows_registry"] = {caps["X"]: v[0:1], caps["N"]: v[1:2], caps["B"] + 1: v[2:3]}
    dd["num_valid_graphs"] = caps["B"]
    return dd


# ----------------------------------------------------------------- mirroring device state
def _owner_of(dd: dict, indices: torch.Tensor) -> SparseTensor:
    for v in dd.values():
        if isinstance(v, SparseTensor) and v.indices is indices:
            return v
    raise NotImplementedError("static batches: plan cached on an index tensor that no "
                              "SparseTensor of the datadict owns")


def _rebuild(dd: dict, t: torch.Tensor, key, template=None):
    """Build, on the new batch's tensor ``t``, the plan the template holds under ``key``."""
    kind = key[0] if isinstance(key, tuple) else key
    if kind == "acd":
        # a template that uses all three groupings (training) gets them from one library call
        every = isinstance(template, P.TriplePlan) and len(template._groups) == 3
        return P.plan_from_acd(t, *key[1:], build_all=every)
    if kind == "sswl_bwd":
        return P.sswl_bwd_group(t, dd[key[1]], key[1], key[2], key[3])
    if kind == "key":
        return P.plan_from_key(t, key[1], key[2])
    if kind == "embedding":
        return P.embedding_plan(t, key[1], key[2])
    if kind == "pool":
        return _owner_of(dd, t)._key_plan(key[1])
    if kind == "pairplan":
        return _owner_of(dd, t)._pair_plan()
    if kind == "spmm":
        from .backend.Spmm import _spmm_plan
        return _spmm_plan(_owner_of(dd, t), key[1])
    raise NotImplementedError(f"static batches: plan kind {key!r} has a data-dependent shape")


class _Mirror:
    """Pairs every device array reachable from a template datadict with the same array of a
    freshly built batch and copies new -> template."""

    def __init__(self):
        self.pairs: List = []
        self.seen = set()
        self.src_objs: List = []       # tensors / plans of the fresh batch (released after copy)

    def tensor(self, dst: torch.Tensor, src: torch.Tensor, dd_src: dict):
        if id(dst) in self.seen:
            return
        self.seen.add(id(dst))
        if dst.shape != src.shape or dst.dtype != src.dtype:
            raise RuntimeError(f"static batches: array shapes differ ({tuple(dst.shape)} vs "
                               f"{tuple(src.shape)})")
        self.pairs.append((dst, src))
        self.src_objs.append(src)
        cache = getattr(dst, "_pgh_cache", None)
        if cache:
            for key, dobj in cache.items():
                self.obj(dobj, _rebuild(dd_src, src, key, dobj), dd_src)

    def obj(self, d, s, dd_src):
        if d is None:
            return
        if isinstance(d, torch.Tensor):
            self.tensor(d, s, dd_src)
        elif isinstance(d, P.TriplePlan):
            self.plan(d, s, dd_src)
        elif isinstance(d, tuple):                   # Group / EmbeddingPlan / plain tuples
            for a, b in zip(d, s):
                if isinstance(a, (torch.Tensor, tuple, P.TriplePlan)):
                    self.obj(a, b, dd_src)
        else:
            raise NotImplementedError(f"static batches: cannot mirror {type(d).__name__}")

    def plan(self, d: P.TriplePlan, s: P.TriplePlan, dd_src):
        if id(d) in self.seen:
            return
        self.seen.add(id(d))
        self.src_objs.append(s)
        for k in ("a", "c", "d"):
            if d.idx[k] is not None:
                self.tensor(d.idx[k], s.idx[k], dd_src)
        for which in list(d._groups.keys()):
            self.obj(d._groups[which], s.group(which), dd_src)
        if d._inv is not None:
            self.tensor(d._inv, s.inv_count(), dd_src)
        if d._swapped is not None:
            self.plan(d._swapped, s.swapped(), dd_src)
        t = getattr(d, "_transposed", None)
        if t is not None:
            self.plan(t, s.transposed(), dd_src)


    def release(self):
        """Break the reference cycles of the fresh batch's plan objects (plan <-> swapped /
        transposed plan, tensor -> cache -> plan -> tensor): its device memory then goes back to
        the allocator as soon as the caller drops the datadict, instead of whenever the cyclic
        garbage collector next runs (which made the pool grow -- a cuMemMap stall of tens of
        milliseconds -- at unpredictable steps)."""
        for o in self.src_objs:
            if isinstance(o, torch.Tensor):
                c = getattr(o, "_pgh_cache", None)
                if c is not None:
                    c.clear()
            else:
                o._groups = {}
                o._swapped = None
                o._inv = None
                if hasattr(o, "_transposed"):
                    o._transposed = None
        self.src_objs = []
        self.pairs = []


def _copy_pairs(pairs) -> None:
    """dst <- src for every pair, stream-ordered: ONE launch of the library's batched copy for
    the arrays it takes (contiguous, sizes and addresses multiples of 4 bytes), ``copy_`` for
    the rest (e.g. byte masks of odd length)."""
    import ctypes as C
    from . import _lib
    srcs, dsts, sizes = [], [], []
    dev = None
    for dst, src in pairs:
        nb = dst.numel() * dst.element_size()
        if (dst.is_cuda and src.is_cuda and dst.device == src.device and dst.is_contiguous()
                and src.is_contiguous() and nb % 4 == 0 and dst.data_ptr() % 4 == 0
                and src.data_ptr() % 4 == 0 and (dev is None or dev == dst.device)):
            dev = dst.device
            if nb:
                srcs.append(src.data_ptr())
                dsts.append(dst.data_ptr())
                sizes.append(nb)
        else:
            dst.copy_(src, non_blocking=True)
    if srcs:
        n = len(srcs)
        _lib.call("pgh_multi_copy", (C.c_void_p * n)(*srcs), (C.c_void_p * n)(*dsts),
                  (C.c_int64 * n)(*sizes), n, _lib.stream_ptr(dev))
        _lib.count_launch()


def mirror_into(template: dict, fresh: dict) -> int:
    """Copy every device array of ``fresh`` (datadict of a batch padded to the same capacities,
    incl. all cached plans the template has built) over the template's arrays; returns the
    number of arrays copied.  Stream-ordered on the current stream."""
    m = _Mirror()
    for name, d in template.items():
        if name.startswith("_") or not isinstance(d, (SparseTensor, torch.Tensor)):
            continue
        s = fresh[name]
        if isinstance(d, SparseTensor):
            m.tensor(d.indices, s.indices, fresh)
            if d.values is not None:
                m.tensor(d.values, s.values, fresh)
        elif isinstance(d, torch.Tensor):
            m.tensor(d, s, fresh)
    _copy_pairs(m.pairs)
    n = len(m.pairs)
    m.release()
    return n


def release_datadict(dd: Optional[dict]) -> None:
    """Drop every cached plan reachable from a datadict that is no longer needed and break the
    plan objects' reference cycles, so its device memory is freed by reference counting at once
    (see :meth:`_Mirror.release`)."""
    if not dd:
        return
    seen = set()

    def visit(o):
        if o is None or id(o) in seen:
            return
        seen.add(id(o))
        if isinstance(o, torch.Tensor):
            c = getattr(o, "_pgh_cache", None)
            if c:
                vals = list(c.values())
                c.clear()
                for v in vals:
                    visit(v)
        elif isinstance(o, P.TriplePlan):
            subs = list(o.idx.values()) + list(dict.values(o._groups)) + [o._swapped, o._inv,
                                                                       getattr(o, "_transposed", None)]
            o._groups, o._swapped, o._inv = {}, None, None
            if hasattr(o, "_transposed"):
                o._transposed = None
            for v in subs:
                visit(v)
        elif isinstance(o, SparseTensor):
            visit(o.indices)
            visit(o.values)
        elif isinstance(o, (tuple, list)):
            for v in o:
                visit(v)

    for v in list(dd.values()):
        visit(v)


# ------------------------------------------------------------------------------ feeding
class StaticFeeder:
    """Host-fed training with graph replay: two static slots, each with its own captured graph
    of ``step_fn(datadict)``; ``step()`` replays the slot that holds the current batch while a
    worker thread loads the next host batch into the other slot on a side stream.

    ``host_batches``: padded :class:`HostBatch` objects (:func:`pad_host_batch`), cycled.
    ``step_fn(dd)`` must be capturable (see pygho_b200/graph.py) and return the step's output
    tensor (e.g. the loss)."""

    def __init__(self, host_batches, caps, device, keys, step_fn, pinned: Optional[dict] = None,
                 threaded: bool = True):
        from .graph import StepGraph
        from .hodata.device import sp_datadict
        self.hbs, self.caps, self.device, self.keys = list(host_batches), caps, device, list(keys)
        self.pinned = {} if pinned is None else pinned
        self._sp_datadict = sp_datadict
        self.side = torch.cuda.Stream(device)
        self.slots, self.graphs = [], []
        self.loaded = [torch.cuda.Event(), torch.cuda.Event()]    # slot content is ready
        self.consumed = [torch.cuda.Event(), torch.cuda.Event()]  # slot's replay has finished
        self.pos = 0
        for s in range(2):
            dd = attach_registry(sp_datadict(self.hbs[s % len(self.hbs)], device, self.keys, self.pinned), caps)
            with static_shapes(dd):
                g = StepGraph(lambda dd=dd: step_fn(dd), warmup=2)
            self.slots.append(dd)
            self.graphs.append(g)
        torch.cuda.synchronize(device)
        for s in range(2):
            self.loaded[s].record()
            self.consumed[s].record()
        self.pos = 0              # index of the batch the next step() consumes
        self._jobs = self._worker = None
        self._done = [threading.Event(), threading.Event()]
        self._error = None
        self.copies = 0
        self.load_ms: List[float] = []     # host time of every load (enqueue only)
        if threaded:
            import queue
            self._jobs = queue.Queue()
            self._worker = threading.Thread(target=self._run, name="pygho-static-feed", daemon=True)
            self._worker.start()
        # slot 0 holds batch 0 and slot 1 batch 1 already (they were captured on them)
        self._done[0].set()
        self._done[1].set()

    @property
    def launches(self) -> int:
        return self.graphs[0].launches

    def _load(self, index: int):
        slot = index & 1
        hb = self.hbs[index % len(self.hbs)]
        t0 = time.perf_counter()
        with torch.cuda.stream(self.side):
            self.side.wait_event(self.consumed[slot])      # the slot's last replay is over
            if os.environ.get("PYGHO_B200_FEEDER_NOLOAD"):  # profiling: replay without feeding
                self.loaded[slot].record(self.side)
                return
            fresh = self._sp_datadict(hb, self.device, self.keys, self.pinned)
            self.copies = mirror_into(self.slots[slot], fresh)
            self.loaded[slot].record(self.side)
            del fresh
        self.load_ms.append(1e3 * (time.perf_counter() - t0))

    def _run(self):
        torch.cuda.set_device(self.device)
        while True:
            index = self._jobs.get()
            if index is None:
                return
            try:
                self._load(index)
            except BaseException as e:  # noqa: BLE001 - re-raised in step()
                self._error = e
            self._done[index & 1].set()

    def _submit(self, index: int):
        self._done[index & 1].clear()
        if self._jobs is not None:
            self._jobs.put(index)
        else:
            self._load(index)
            self._done[index & 1].set()

    def step(self) -> torch.Tensor:
        """Replay the step on the current batch; returns the (static) output tensor of the
        slot -- read it (or copy it) before the same slot is replayed two steps later."""
        slot = self.pos & 1
        self._done[slot].wait()
        if self._error is not None:
            err, self._error = self._error, None
            raise err
        cur = torch.cuda.current_stream(self.device)
        cur.wait_event(self.loaded[slot])
        loss = self.graphs[slot].replay()
        self.consumed[slot].record(cur)
        self.pos += 1
        self._submit(self.pos + 1)         # refill the slot that was consumed one step ago
        return loss

    def close(self):
        if self._jobs is not None:
            self._jobs.put(None)
            self._worker.join(timeout=10)
            self._jobs = None
        self.graphs = []


class StaticPredictor:
    """Graph-replayed evaluation of a fixed held-out set: ``predictor()`` returns the model's
    predictions for every graph of ``host_batches``, in order, as one ``(sum B_i, out)`` device
    tensor.  Built on :class:`StaticFeeder` (same scope: sparse mode, 2-D tuples).

    ``host_batches``: UNPADDED :class:`HostBatch` objects with their host plans; they are padded
    here to ``caps`` (:func:`capacities` over these batches), and may hold fewer graphs than
    ``caps["B"]``.  ``model(dd)`` is captured on the two slots in ``eval()`` mode under
    ``torch.no_grad()`` -- the BatchNorm blocks take the one-pass inference path
    (ops.linear_bn_eval) and nothing writes the running statistics -- and the model's training
    flag is restored afterwards.  ``no_grad`` rather than ``inference_mode``: the plans are cached
    on the datadicts' index tensors, and inference tensors could not be used by a later training
    step on the same data.

    Lifetime: the graphs read the parameters and running statistics in place, so they follow
    optimizer steps and ``load_state_dict``; anything that reallocates them (``.to()``,
    replacing a module or a parameter) needs a new predictor."""

    def __init__(self, host_batches, caps, device, keys, model, pinned: Optional[dict] = None,
                 threaded: bool = True):
        hbs = list(host_batches)
        self.counts = [hb.num_graphs for hb in hbs]
        padded = [pad_host_batch(hb, caps, keys, fewer_graphs=True) for hb in hbs]
        was_training = model.training
        model.eval()
        try:
            with torch.no_grad():
                self.feeder = StaticFeeder(padded, caps, device, keys, model, pinned, threaded)
        finally:
            model.train(was_training)

    def __call__(self) -> torch.Tensor:
        """Replay every batch once; rows ``[:B_i]`` of each replay's output (the dummy pad graph
        and any empty graphs dropped), concatenated in batch order.  Stream-ordered."""
        out, off = None, 0
        for b in self.counts:
            pred = self.feeder.step()
            if out is None:
                out = pred.new_empty((sum(self.counts),) + tuple(pred.shape[1:]))
            out[off:off + b].copy_(pred[:b])
            off += b
        return out

    def close(self):
        self.feeder.close()
