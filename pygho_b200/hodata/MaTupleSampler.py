"""Dense tuple samplers on the device (reference ``hodata/MaTupleSampler.py``).

``spdsampler`` (:11-31) runs scipy's ``shortest_path`` per graph on the CPU and the loader
pads the per-graph ``n x n`` matrices with ``to_dense_tuplefeat`` (``hodata/MaData.py:152-212``).
Here the bit-set BFS kernel produces all distance matrices of the batch and one more pass
writes the padded ``(B, nmax, nmax)`` MaskedTensor directly.  ``rdsampler`` (:34-57) takes the
pseudo-inverse of every graph's Laplacian with numpy; here one kernel inverts all of them in
fp64 in shared memory and the same kind of padding pass follows."""
from __future__ import annotations

import torch
from torch import LongTensor

from .. import _lib
from .._lib import call, ptr, stream_ptr
from ..backend.MaTensor import MaskedTensor
from .SpTupleSampler import PtrLike, graph_distances, resistance_distances


def spdsampler(edge_index: LongTensor, node_ptr: PtrLike, hop: int = 2,
               max_num_nodes: int = None, grouped: bool = True) -> MaskedTensor:
    """Shortest-path-distance tuple features of a whole batch, clamped to ``hop + 1``
    (unreachable pairs included), as a ``(B, nmax, nmax)`` int64 MaskedTensor with pads 0."""
    dev = _lib.require_cuda(edge_index)
    D, sq_ptr, _cnt, node_ptr, _ng, nmax = graph_distances(edge_index, node_ptr, hop, grouped)
    B = node_ptr.numel() - 1
    if max_num_nodes is not None:
        assert max_num_nodes >= nmax, "max_num_nodes is smaller than the largest graph"
        nmax = int(max_num_nodes)
    out = torch.empty((B, nmax, nmax), dtype=torch.int64, device=dev)
    mask = torch.empty((B, nmax, nmax), dtype=torch.bool, device=dev)
    if out.numel():
        call("pgh_spd_dense_i64", ptr(D), ptr(node_ptr), ptr(sq_ptr), B, nmax, int(hop) + 1, 0,
             ptr(out), ptr(mask), stream_ptr(dev))
        _lib.count_launch()
    return MaskedTensor(out, mask, 0, True)


def rdsampler(edge_index: LongTensor, node_ptr: PtrLike, max_num_nodes: int = None,
              grouped: bool = True) -> MaskedTensor:
    """Resistance-distance tuple features of a whole batch, ``R[i, j] = L+[i, i] + L+[j, j]
    - 2 L+[i, j]`` with ``L+`` the pseudo-inverse of the Laplacian of each graph as a simple
    undirected graph (pairs in different components keep what the pseudo-inverse gives), as
    a ``(B, nmax, nmax)`` float32 MaskedTensor with pads 0.  Graphs of up to 128 nodes.

    With ``node_ptr`` on the host there is no device read-back, so the call can be captured in
    a CUDA graph; torch then needs ``node_ptr`` as a pinned CPU tensor, kept alive with the
    graph (each replay copies it to the device again)."""
    dev = _lib.require_cuda(edge_index)
    R, sq_ptr, node_ptr, _ng, nmax = resistance_distances(edge_index, node_ptr, grouped)
    B = node_ptr.numel() - 1
    if max_num_nodes is not None:
        assert max_num_nodes >= nmax, "max_num_nodes is smaller than the largest graph"
        nmax = int(max_num_nodes)
    out = torch.empty((B, nmax, nmax), dtype=torch.float32, device=dev)
    mask = torch.empty((B, nmax, nmax), dtype=torch.bool, device=dev)
    if out.numel():
        call("pgh_rd_dense_f32", ptr(R), ptr(node_ptr), ptr(sq_ptr), B, nmax, 0.0, ptr(out),
             ptr(mask), stream_ptr(dev))
        _lib.count_launch()
    return MaskedTensor(out, mask, 0, True)
