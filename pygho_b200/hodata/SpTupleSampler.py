"""Tuple samplers on the device for whole batches (reference ``hodata/SpTupleSampler.py``).

The reference samples one graph at a time on the CPU: ``KhopSampler`` (:91-126) calls
``k_hop_subgraph`` (:12-88) once per node in a Python loop and collates the per-node
subgraphs with PyG.  Here one kernel computes the hop-distance matrix of every graph of a
block-diagonal batch (one CTA per graph, bit-set BFS in shared memory) and a second one
compacts the rows into the ``(i, j)``-sorted tuple list, so sampling a 1024-graph batch is
two launches plus a prefix sum.  ``rd_tuplefeat`` gives tuples their resistance-distance
features, gathered from the per-graph matrices of ``resistance_distances``.  Indices are
GLOBAL node ids (the collate offsets of ``SpHoData.__inc__``, ``hodata/SpData.py:60-77``, are
already applied).
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple, Union

import torch
from torch import LongTensor, Tensor

from .. import _lib
from .._lib import call, ptr, stream_ptr
from ..backend.SpTensor import SparseTensor

PtrLike = Union[Tensor, Sequence[int]]


def _as_ptr(node_ptr: PtrLike, device) -> Tuple[LongTensor, int, int]:
    """(device int64 ptr, number of nodes, largest graph) -- the sizes are read on the host
    when the pointer array is still there (the usual case: the loader knows its graph sizes)."""
    if isinstance(node_ptr, Tensor) and node_ptr.is_cuda:
        sizes = torch.diff(node_ptr)
        return node_ptr.to(torch.int64), int(node_ptr[-1]), int(sizes.max()) if sizes.numel() else 0
    host = torch.as_tensor(node_ptr, dtype=torch.int64)
    sizes = torch.diff(host)
    return (host.to(device, non_blocking=True), int(host[-1]),
            int(sizes.max()) if sizes.numel() else 0)


def node2graph(node_ptr: LongTensor, num_nodes: int) -> LongTensor:
    """batch vector: graph id of every node (``ptr2batch``, reference backend/Spspmm.py:9-31)."""
    B = node_ptr.numel() - 1
    return torch.repeat_interleave(torch.arange(B, device=node_ptr.device), torch.diff(node_ptr),
                                   output_size=num_nodes)


def _batch_layout(edge_index: LongTensor, node_ptr: PtrLike, grouped: bool):
    """Per-graph layout of a batch that the one-CTA-per-graph kernels read:
    ``(src, dst, node_ptr, edge_ptr, sq_ptr, node_graph, max_nodes)``.  ``src`` / ``dst`` are
    grouped by graph (sorted first unless ``grouped``), ``edge_ptr`` delimits each graph's
    edges and ``sq_ptr[g] = sum_{h<g} n_h^2`` its flat ``n_g x n_g`` matrix."""
    dev = _lib.require_cuda(edge_index)
    node_ptr, N, nmax = _as_ptr(node_ptr, dev)
    B = node_ptr.numel() - 1
    node_graph = node2graph(node_ptr, N)
    src, dst = edge_index[0].contiguous(), edge_index[1].contiguous()
    edge_graph = node_graph[src] if src.numel() else src
    if not grouped and src.numel():
        edge_graph, order = torch.sort(edge_graph, stable=True)
        src, dst = src[order], dst[order]
    edge_ptr = torch.searchsorted(edge_graph, torch.arange(B + 1, device=dev))
    sizes = torch.diff(node_ptr)
    sq_ptr = torch.zeros((B + 1,), dtype=torch.int64, device=dev)
    torch.cumsum(sizes * sizes, 0, out=sq_ptr[1:])
    return src, dst, node_ptr, edge_ptr, sq_ptr, node_graph, nmax


def graph_distances(edge_index: LongTensor, node_ptr: PtrLike, cutoff: int,
                    grouped: bool = True):
    """Hop distances of all graphs of a batch.

    ``edge_index``: (2, E) int64 global ids; ``grouped`` = the edges of a graph are contiguous
    and graphs appear in order (any PyG-style collate); otherwise they are sorted by graph
    first.  Returns ``(D, sq_ptr, cnt, node_ptr, node_graph, max_nodes)``:
    ``D[sq_ptr[g] + i * n_g + j]`` = dist (uint8, 255 beyond ``cutoff``), ``cnt[v]`` = number
    of nodes within ``cutoff`` hops of node v (int32)."""
    src, dst, node_ptr, edge_ptr, sq_ptr, node_graph, nmax = _batch_layout(edge_index, node_ptr,
                                                                            grouped)
    dev, B, N = node_ptr.device, node_ptr.numel() - 1, node_graph.numel()
    # sum of n_g^2 <= N * nmax: allocate the bound instead of reading the exact size back
    D = torch.empty((max(1, N * nmax),), dtype=torch.uint8, device=dev)
    cnt = torch.zeros((N,), dtype=torch.int32, device=dev)
    if B and N:
        call("pgh_graph_dist_u8", ptr(src), ptr(dst), ptr(node_ptr), ptr(edge_ptr), ptr(sq_ptr),
             B, max(1, nmax), int(cutoff), ptr(D), ptr(cnt), stream_ptr(dev))
        _lib.count_launch()
    return D, sq_ptr, cnt, node_ptr, node_graph, nmax


def resistance_distances(edge_index: LongTensor, node_ptr: PtrLike, grouped: bool = True):
    """Resistance distances of all graphs of a batch (``edge_index`` and ``grouped`` as in
    :func:`graph_distances`).  Returns ``(R, sq_ptr, node_ptr, node_graph, max_nodes)`` with
    ``R[sq_ptr[g] + i * n_g + j] = L+[i, i] + L+[j, j] - 2 L+[i, j]`` (float32), ``L+`` the
    pseudo-inverse of the Laplacian of graph g as a simple undirected graph.  Graphs of up to
    128 nodes."""
    src, dst, node_ptr, edge_ptr, sq_ptr, node_graph, nmax = _batch_layout(edge_index, node_ptr,
                                                                            grouped)
    dev, B, N = node_ptr.device, node_ptr.numel() - 1, node_graph.numel()
    R = torch.empty((max(1, N * nmax),), dtype=torch.float32, device=dev)
    if B and N:
        call("pgh_resistance_f32", ptr(src), ptr(dst), ptr(node_ptr), ptr(edge_ptr), ptr(sq_ptr),
             B, max(1, nmax), ptr(R), stream_ptr(dev))
        _lib.count_launch()
    return R, sq_ptr, node_ptr, node_graph, nmax


def rd_tuplefeat(tupleid: LongTensor, edge_index: LongTensor, node_ptr: PtrLike,
                 grouped: bool = True) -> Tensor:
    """Resistance distance of every 2-D tuple ``(i, j)`` of a batch (e.g. ``KhopSampler``'s
    ``X.indices``): ``(T,)`` float32, the values :func:`MaTupleSampler.rdsampler` holds at those
    positions.  Both nodes of a tuple must belong to the same graph."""
    R, sq_ptr, node_ptr, node_graph, _nmax = resistance_distances(edge_index, node_ptr, grouped)
    N = node_graph.numel()
    if tupleid.shape[1] == 0:
        return torch.empty((0,), dtype=torch.float32, device=R.device)
    msg = "rd_tuplefeat: every tuple must pair two nodes of one graph"
    if N == 0:
        raise ValueError(msg)
    i, j = tupleid[0].clamp(0, N - 1), tupleid[1].clamp(0, N - 1)
    g = node_graph[i]
    if not bool(((tupleid >= 0).all(0) & (tupleid < N).all(0) & (node_graph[j] == g)).all()):
        raise ValueError(msg)
    n0 = node_ptr[g]
    n = node_ptr[g + 1] - n0
    return R[sq_ptr[g] + (i - n0) * n + (j - n0)]


def KhopSampler(edge_index: LongTensor, node_ptr: PtrLike, hop: int = 2,
                grouped: bool = True) -> SparseTensor:
    """k-hop subgraph tuples of every node of a batch: ``X[i, j] = dist(i, j)`` for
    ``dist <= hop`` (the root itself included with distance 0), coalesced, sorted by (i, j).

    Batch-level counterpart of the reference ``KhopSampler(data, hop)``
    (SpTupleSampler.py:91-126) applied to every graph and collated."""
    dev = _lib.require_cuda(edge_index)
    D, sq_ptr, cnt, node_ptr, node_graph, _nmax = graph_distances(edge_index, node_ptr, hop,
                                                                  grouped)
    N = node_graph.numel()
    rowptr = torch.zeros((N + 1,), dtype=torch.int64, device=dev)
    torch.cumsum(cnt, 0, out=rowptr[1:])
    T = int(rowptr[-1]) if N else 0                       # the one size read-back of the sampler
    tupleid = torch.empty((2, T), dtype=torch.int64, device=dev)
    feat = torch.empty((T,), dtype=torch.int64, device=dev)
    if T:
        call("pgh_khop_emit", ptr(D), ptr(node_ptr), ptr(sq_ptr), ptr(node_graph), ptr(rowptr), N,
             T, ptr(tupleid), ptr(feat), stream_ptr(dev))
        _lib.count_launch()
    return SparseTensor(tupleid, feat, (N, N), is_coalesced=True)


def I2Sampler(edge_index: LongTensor, node_ptr: PtrLike, hop: int = 3,
              grouped: bool = True) -> SparseTensor:
    """I2-GNN tuples of a batch: for every directed edge ``(i, j)`` the nodes ``k`` within
    ``hop`` of ``i`` or of ``j``; ``X[i, j, k] = (dist(i, k), dist(j, k))`` clamped to
    ``hop + 1``.  Tuples follow the edge order, then ``k``: coalesced when ``edge_index`` is
    sorted by (row, col) (any coalesced batch).  Batch-level counterpart of the reference
    ``I2Sampler(data, hop)`` (SpTupleSampler.py:129-174) for undirected graphs."""
    dev = _lib.require_cuda(edge_index)
    D, sq_ptr, _cnt, node_ptr, node_graph, _nmax = graph_distances(edge_index, node_ptr, hop + 1,
                                                                   grouped)
    N, E = node_graph.numel(), edge_index.shape[1]
    src, dst = edge_index[0].contiguous(), edge_index[1].contiguous()
    cnt = torch.zeros((E,), dtype=torch.int32, device=dev)
    if E:
        call("pgh_i2_count", ptr(D), ptr(src), ptr(dst), ptr(node_ptr), ptr(sq_ptr),
             ptr(node_graph), E, int(hop), ptr(cnt), stream_ptr(dev))
        _lib.count_launch()
    rowptr = torch.zeros((E + 1,), dtype=torch.int64, device=dev)
    torch.cumsum(cnt, 0, out=rowptr[1:])
    T = int(rowptr[-1]) if E else 0
    tupleid = torch.empty((3, T), dtype=torch.int64, device=dev)
    feat = torch.empty((T, 2), dtype=torch.int64, device=dev)
    if T:
        call("pgh_i2_emit", ptr(D), ptr(src), ptr(dst), ptr(node_ptr), ptr(sq_ptr),
             ptr(node_graph), ptr(rowptr), E, T, int(hop), ptr(tupleid), ptr(feat), stream_ptr(dev))
        _lib.count_launch()
    return SparseTensor(tupleid, feat, (N, N, N, 2), is_coalesced=True)
