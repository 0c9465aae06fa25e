"""``torch.library`` operators ``pygho_b200::*`` -- thin shims over the C ABI.

Each operator allocates its output with torch (device memory is torch's job), passes raw
device pointers plus the current CUDA stream to ``libpygho_b200.so`` and returns.  They are
registered for the CUDA dispatch key only: calling them with CPU tensors raises (there is
no CPU implementation of this package).  ``register_fake`` gives shape propagation so the
ops trace under ``torch.compile`` (the reference compiles its models, example/zinc.py:407).

Autograd lives one level up in :class:`SegGmr`, :class:`MaMaMM` and :class:`MaskedPool`,
which call only these operators in both directions.
"""
from __future__ import annotations

import os
from typing import Optional

import torch
from torch import Tensor

from . import _lib
from ._lib import AGGR_CODE, call, ptr, stream_ptr

_LIB = torch.library.Library("pygho_b200", "DEF")


def _f32c(t: Optional[Tensor]) -> Optional[Tensor]:
    if t is None:
        return None
    if t.dtype != torch.float32:
        raise TypeError(f"pygho_b200 kernels are float32; got {t.dtype}")
    return t if t.is_contiguous() else t.contiguous()


def _i32c(t: Optional[Tensor]) -> Optional[Tensor]:
    if t is None:
        return None
    if t.dtype != torch.int32:
        raise TypeError(f"plan indices must be int32; got {t.dtype}")
    return t if t.is_contiguous() else t.contiguous()


# ------------------------------------------------------------------------- seg_gmr
_LIB.define("seg_gmr(Tensor a_val, Tensor? c, Tensor? a_scale, Tensor? b_val, Tensor? d, "
            "Tensor? rowptr, int n_rows, int aggr) -> Tensor")


def _rows2d(t: Optional[Tensor]) -> Optional[Tensor]:
    """float32 (rows, dense) whose rows are contiguous; the row stride may exceed dense
    (column slice of a wider buffer).  Anything else is copied."""
    if t is None:
        return None
    if t.dtype != torch.float32:
        raise TypeError(f"pygho_b200 kernels are float32; got {t.dtype}")
    if t.ndim == 2 and t.stride(1) == 1 and t.stride(0) >= t.shape[1] and t.stride(0) % 4 == 0 \
            and t.data_ptr() % 16 == 0:
        return t
    return t.contiguous()


def _seg_gmr_into(a_val, c, a_scale, b_val, d, rowptr, n_rows, aggr, out, accumulate=False):
    a_val, b_val, a_scale = _rows2d(a_val), _rows2d(b_val), _f32c(a_scale)
    c, d, rowptr = _i32c(c), _i32c(d), _i32c(rowptr)
    dense = a_val.shape[1]
    if a_val.shape[0] == 0 or (b_val is not None and b_val.shape[0] == 0):
        if not accumulate:
            out.zero_()
        return out
    if n_rows and dense:
        n_entries = 0
        for idx in (c, d):
            if idx is not None:
                n_entries = idx.shape[0]
        if n_entries == 0 and rowptr is not None:
            n_entries = a_val.shape[0]          # identity index: one entry per operand row
        call("pgh_seg_gmr_ld_f32", ptr(a_val), a_val.stride(0), ptr(c), ptr(a_scale), ptr(b_val),
             b_val.stride(0) if b_val is not None else dense, ptr(d), ptr(rowptr), n_rows,
             n_entries, dense, aggr, int(accumulate), ptr(out), out.stride(0),
             stream_ptr(a_val.device))
        _lib.count_launch()
    return out


def _seg_gmr_cuda(a_val, c, a_scale, b_val, d, rowptr, n_rows, aggr):
    out = torch.empty((n_rows, a_val.shape[1]), dtype=torch.float32, device=a_val.device)
    return _seg_gmr_into(a_val, c, a_scale, b_val, d, rowptr, n_rows, aggr, out)


_LIB.impl("seg_gmr", _seg_gmr_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::seg_gmr")
def _seg_gmr_fake(a_val, c, a_scale, b_val, d, rowptr, n_rows, aggr):
    return a_val.new_empty((n_rows, a_val.shape[1]))


_LIB.define("seg_gmr_out(Tensor a_val, Tensor? c, Tensor? a_scale, Tensor? b_val, Tensor? d, "
            "Tensor? rowptr, int n_rows, int aggr, Tensor(a!) out, bool accumulate) -> ()")


def _seg_gmr_out_cuda(a_val, c, a_scale, b_val, d, rowptr, n_rows, aggr, out, accumulate):
    if out.dtype != torch.float32 or out.ndim != 2 or out.stride(1) != 1 or out.stride(0) % 4 \
            or out.data_ptr() % 16 or tuple(out.shape) != (n_rows, a_val.shape[1]):
        raise ValueError("seg_gmr_out: out must be a float32 (n_rows, dense) row-contiguous view")
    _seg_gmr_into(a_val, c, a_scale, b_val, d, rowptr, n_rows, aggr, out, accumulate)


_LIB.impl("seg_gmr_out", _seg_gmr_out_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::seg_gmr_out")
def _seg_gmr_out_fake(a_val, c, a_scale, b_val, d, rowptr, n_rows, aggr, out, accumulate):
    return None


_LIB.define("seg_gmr_fused(Tensor a_val, Tensor? c, Tensor? a_scale, Tensor? b_val, Tensor? d, "
            "Tensor? rowptr, int n_rows, int aggr, Tensor? add_src, Tensor? copy_src, "
            "Tensor(a!)? copy_dst, Tensor(b!) out, Tensor? add_src2=None) -> ()")


def _row_view_ok(t: Optional[Tensor], n_rows: int, dense: int) -> bool:
    return t is None or (t.dtype == torch.float32 and t.ndim == 2 and t.stride(1) == 1
                         and t.stride(0) >= dense and t.stride(0) % 4 == 0
                         and t.data_ptr() % 16 == 0 and tuple(t.shape) == (n_rows, dense))


def fused_epilogue_ok(dense: int, *views) -> bool:
    """The fused row epilogue (``seg_gmr_fused``) needs dense % 128 == 0 and 16-byte rows."""
    return dense % 128 == 0 and all(
        v is None or (v.dtype == torch.float32 and v.ndim == 2 and v.stride(1) == 1
                      and v.stride(0) % 4 == 0 and v.data_ptr() % 16 == 0) for v in views)


def _seg_gmr_fused_cuda(a_val, c, a_scale, b_val, d, rowptr, n_rows, aggr, add_src, copy_src,
                        copy_dst, out, add_src2=None):
    a_val, b_val, a_scale = _rows2d(a_val), _rows2d(b_val), _f32c(a_scale)
    c, d, rowptr = _i32c(c), _i32c(d), _i32c(rowptr)
    dense = a_val.shape[1]
    for name, t in (("out", out), ("add_src", add_src), ("copy_src", copy_src), ("copy_dst", copy_dst),
                    ("add_src2", add_src2)):
        if not _row_view_ok(t, n_rows, dense):
            raise ValueError(f"seg_gmr_fused: {name} must be a float32 (n_rows, dense) row-contiguous view")
    if n_rows == 0:
        return
    n_entries = 0
    for idx in (c, d):
        if idx is not None:
            n_entries = idx.shape[0]
    if n_entries == 0 and rowptr is not None:
        n_entries = a_val.shape[0]
    call("pgh_seg_gmr_fused_f32", ptr(a_val), a_val.stride(0), ptr(c), ptr(a_scale), ptr(b_val),
         b_val.stride(0) if b_val is not None else dense, ptr(d), ptr(rowptr), n_rows, n_entries,
         dense, aggr, ptr(add_src), add_src.stride(0) if add_src is not None else 0,
         ptr(add_src2), add_src2.stride(0) if add_src2 is not None else 0, ptr(copy_src), copy_src.stride(0) if copy_src is not None else 0, ptr(copy_dst),
         copy_dst.stride(0) if copy_dst is not None else 0, ptr(out), out.stride(0),
         stream_ptr(a_val.device))
    _lib.count_launch()


_LIB.impl("seg_gmr_fused", _seg_gmr_fused_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::seg_gmr_fused")
def _seg_gmr_fused_fake(a_val, c, a_scale, b_val, d, rowptr, n_rows, aggr, add_src, copy_src,
                        copy_dst, out, add_src2=None):
    return None


_LIB.define("seg_tie_scale(Tensor a_val, Tensor? c, Tensor? b_val, Tensor? d, Tensor? rowptr, "
            "Tensor out, Tensor grad) -> Tensor")


def _seg_tie_scale_cuda(a_val, c, b_val, d, rowptr, out, grad):
    a_val, b_val, out, grad = _f32c(a_val), _f32c(b_val), _f32c(out), _f32c(grad)
    n_rows, dense = out.shape
    gs = torch.empty_like(out)
    if out.numel():
        call("pgh_seg_tie_scale_f32", ptr(a_val), ptr(_i32c(c)), ptr(b_val), ptr(_i32c(d)),
             ptr(_i32c(rowptr)), n_rows, dense, ptr(out), ptr(grad), ptr(gs),
             stream_ptr(out.device))
        _lib.count_launch()
    return gs


_LIB.impl("seg_tie_scale", _seg_tie_scale_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::seg_tie_scale")
def _seg_tie_scale_fake(a_val, c, b_val, d, rowptr, out, grad):
    return torch.empty_like(out)


_LIB.define("seg_select_bwd(Tensor self_val, Tensor? other_val, Tensor? other_idx, "
            "Tensor? row_idx, Tensor? rowptr, Tensor out, Tensor gscaled) -> Tensor")


def _seg_select_bwd_cuda(self_val, other_val, other_idx, row_idx, rowptr, out, gscaled):
    self_val, other_val = _f32c(self_val), _f32c(other_val)
    out, gscaled = _f32c(out), _f32c(gscaled)
    n_rows, dense = self_val.shape
    g = torch.empty_like(self_val)
    if g.numel():
        call("pgh_seg_select_bwd_f32", ptr(self_val), ptr(other_val), ptr(_i32c(other_idx)),
             ptr(_i32c(row_idx)), ptr(_i32c(rowptr)), n_rows, dense, ptr(out), ptr(gscaled),
             ptr(g), stream_ptr(g.device))
        _lib.count_launch()
    return g


_LIB.impl("seg_select_bwd", _seg_select_bwd_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::seg_select_bwd")
def _seg_select_bwd_fake(self_val, other_val, other_idx, row_idx, rowptr, out, gscaled):
    return torch.empty_like(self_val)


_LIB.define("inv_count(Tensor rowptr) -> Tensor")


def _inv_count_cuda(rowptr):
    rowptr = _i32c(rowptr)
    n = rowptr.shape[0] - 1
    inv = torch.empty((n,), dtype=torch.float32, device=rowptr.device)
    if n > 0:
        call("pgh_inv_count_f32", ptr(rowptr), n, ptr(inv), stream_ptr(rowptr.device))
        _lib.count_launch()
    return inv


_LIB.impl("inv_count", _inv_count_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::inv_count")
def _inv_count_fake(rowptr):
    return rowptr.new_empty((rowptr.shape[0] - 1,), dtype=torch.float32)


# -------------------------------------------------------------------------- masked
_LIB.define("mamamm(Tensor A, bool trans_a, Tensor B, bool trans_b, Tensor mask, Tensor? ext, "
            "int algo, Tensor? order=None) -> Tensor")


def _mamamm_cuda(A, trans_a, B, trans_b, mask, ext, algo, order=None):
    A, B = _f32c(A), _f32c(B)
    mask = mask.contiguous()
    b = A.shape[0]
    n_i, n_j = (A.shape[2], A.shape[1]) if trans_a else (A.shape[1], A.shape[2])
    n_j2, n_k = (B.shape[2], B.shape[1]) if trans_b else (B.shape[1], B.shape[2])
    if n_j != n_j2 or A.shape[3] != B.shape[3] or B.shape[0] != b:
        raise ValueError(f"mamamm: incompatible shapes {tuple(A.shape)} x {tuple(B.shape)}")
    if tuple(mask.shape) != (b, n_i, n_k):
        raise ValueError(f"mamamm: mask shape {tuple(mask.shape)} != {(b, n_i, n_k)}")
    if ext is not None and (ext.dtype != torch.int32 or tuple(ext.shape) != (b, 3)):
        raise ValueError("mamamm: ext must be an int32 tensor of shape (batch, 3)")
    if order is not None and (order.dtype != torch.int32 or tuple(order.shape) != (b,)):
        raise ValueError("mamamm: order must be an int32 permutation of shape (batch,)")
    dense = A.shape[3]
    out = torch.empty((b, n_i, n_k, dense), dtype=torch.float32, device=A.device)
    if out.numel():
        call("pgh_mamamm_f32", ptr(A), int(trans_a), ptr(B), int(trans_b),
             ptr(mask.view(torch.uint8)), ptr(ext.contiguous() if ext is not None else None),
             ptr(order.contiguous() if order is not None else None),
             b, n_i, n_j, n_k, dense, algo, ptr(out), stream_ptr(A.device))
        _lib.count_launch()
    return out


_LIB.impl("mamamm", _mamamm_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::mamamm")
def _mamamm_fake(A, trans_a, B, trans_b, mask, ext, algo, order=None):
    n_i = A.shape[2] if trans_a else A.shape[1]
    n_k = B.shape[1] if trans_b else B.shape[2]
    return A.new_empty((A.shape[0], n_i, n_k, A.shape[3]))


_LIB.define("mask_extents(Tensor mask) -> Tensor")


def _mask_extents_cuda(mask):
    mask = mask.contiguous()
    b, n1, n2 = mask.shape
    ext = torch.empty((b, 2), dtype=torch.int32, device=mask.device)
    if b:
        call("pgh_mask_extents", ptr(mask.view(torch.uint8)), b, n1, n2, ptr(ext),
             stream_ptr(mask.device))
        _lib.count_launch()
    return ext


_LIB.impl("mask_extents", _mask_extents_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::mask_extents")
def _mask_extents_fake(mask):
    return mask.new_empty((mask.shape[0], 2), dtype=torch.int32)


_LIB.define("masked_pool(Tensor data, Tensor mask, int red_dims, int aggr) -> (Tensor, Tensor)")


def _pool_shape(b, n1, n2, red):
    return (b, n2) if red == 1 else (b, n1) if red == 2 else (b,)


def _masked_pool_cuda(data, mask, red_dims, aggr):
    data = _f32c(data)
    mask = mask.contiguous()
    b, n1, n2, dense = data.shape
    keep = _pool_shape(b, n1, n2, red_dims)
    out = torch.empty(keep + (dense,), dtype=torch.float32, device=data.device)
    omask = torch.empty(keep, dtype=torch.bool, device=data.device)
    if out.numel():
        call("pgh_masked_pool_f32", ptr(data), ptr(mask.view(torch.uint8)), b, n1, n2, dense,
             red_dims, aggr, ptr(out), ptr(omask.view(torch.uint8)), stream_ptr(data.device))
        _lib.count_launch()
    return out, omask


_LIB.impl("masked_pool", _masked_pool_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::masked_pool")
def _masked_pool_fake(data, mask, red_dims, aggr):
    b, n1, n2, dense = data.shape
    keep = _pool_shape(b, n1, n2, red_dims)
    return data.new_empty(keep + (dense,)), mask.new_empty(keep)


_LIB.define("masked_pool_bwd(Tensor data, Tensor mask, Tensor out, Tensor g_out, int red_dims, "
            "int aggr) -> Tensor")


def _masked_pool_bwd_cuda(data, mask, out, g_out, red_dims, aggr):
    data, out, g_out = _f32c(data), _f32c(out), _f32c(g_out)
    mask = mask.contiguous()
    b, n1, n2, dense = data.shape
    g = torch.empty_like(data)
    if g.numel():
        call("pgh_masked_pool_bwd_f32", ptr(data), ptr(mask.view(torch.uint8)), ptr(out),
             ptr(g_out), b, n1, n2, dense, red_dims, aggr, ptr(g), stream_ptr(data.device))
        _lib.count_launch()
    return g


_LIB.impl("masked_pool_bwd", _masked_pool_bwd_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::masked_pool_bwd")
def _masked_pool_bwd_fake(data, mask, out, g_out, red_dims, aggr):
    return torch.empty_like(data)


_LIB.define("masked_fill_rows(Tensor data, Tensor mask, float value) -> Tensor")


def _masked_fill_cuda(data, mask, value):
    data = _f32c(data)
    mask = mask.contiguous()
    rows = mask.numel()
    dense = data.numel() // max(rows, 1)
    out = torch.empty_like(data)
    if out.numel():
        call("pgh_masked_fill_f32", ptr(data), ptr(mask.view(torch.uint8)), rows, dense,
             float(value), ptr(out), stream_ptr(data.device))
        _lib.count_launch()
    return out


_LIB.impl("masked_fill_rows", _masked_fill_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::masked_fill_rows")
def _masked_fill_fake(data, mask, value):
    return torch.empty_like(data)


# ---------------------------------------------------------------- fused BatchNorm + act
def _bn_ws(rows, C, device):
    n = int(_lib.load().pgh_bn_ws_bytes(int(rows), int(C)))
    return torch.empty((n,), dtype=torch.uint8, device=device)


_TICKETS = {}


def _tickets(device) -> int:
    """Device address of 64 zeroed int32 ticket words for one launch of a ticketed reduction
    (csrc/fused_mlp.cu).  The kernels leave them zero; 64 slots are handed out round-robin so
    that launches in flight on different streams never share a slot."""
    ent = _TICKETS.get(device)
    if ent is None:
        ent = [torch.zeros((64 * 64,), dtype=torch.int32, device=device), 0]
        _TICKETS[device] = ent
    ent[1] = (ent[1] + 1) & 63
    return ent[0].data_ptr() + ent[1] * 64 * 4


def _rows_dev(t: Optional[Tensor]) -> Optional[Tensor]:
    if t is not None and (t.dtype != torch.int32 or t.numel() != 1 or not t.is_cuda):
        raise TypeError("rows_dev must be a one-element int32 CUDA tensor")
    return t


def _nbt(t: Optional[Tensor]) -> Optional[Tensor]:
    if t is not None and (t.dtype != torch.int64 or t.numel() != 1 or not t.is_cuda):
        raise TypeError("num_batches_tracked must be a one-element int64 CUDA tensor")
    return t


_LIB.define("bn_stats(Tensor y, float eps, float momentum, Tensor(a!)? running_mean, "
            "Tensor(b!)? running_var, Tensor? rows_dev=None, Tensor(c!)? num_batches_tracked=None) "
            "-> (Tensor, Tensor)")


def _bn_stats_cuda(y, eps, momentum, running_mean, running_var, rows_dev=None,
                   num_batches_tracked=None):
    y = _f32c(y)
    rows, C = y.shape
    mean = torch.empty((C,), dtype=torch.float32, device=y.device)
    rstd = torch.empty_like(mean)
    ws = _bn_ws(rows, C, y.device)
    call("pgh_bn_stats_f32", ptr(y), rows, C, ptr(_rows_dev(rows_dev)), float(eps), float(momentum),
         ptr(mean), ptr(rstd), ptr(running_mean), ptr(running_var), None,
         ptr(_nbt(num_batches_tracked)), ptr(ws), ws.numel(), _tickets(y.device),
         stream_ptr(y.device))
    _lib.count_launch()
    return mean, rstd


_LIB.impl("bn_stats", _bn_stats_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::bn_stats")
def _bn_stats_fake(y, eps, momentum, running_mean, running_var, rows_dev=None,
                   num_batches_tracked=None):
    return y.new_empty((y.shape[1],)), y.new_empty((y.shape[1],))


_LIB.define("linear_stats(Tensor x, Tensor weight, Tensor? bias, float eps, float momentum, "
            "Tensor(a!)? running_mean, Tensor(b!)? running_var, Tensor? rows_dev, "
            "Tensor(c!)? num_batches_tracked, bool local) -> (Tensor, Tensor, Tensor)")


def linear_stats_ok(x: Tensor, weight: Tensor) -> bool:
    """The TMA / tcgen05 GEMM with the BatchNorm statistics in its epilogue (csrc/linear_stats.cu)
    computes in TF32: it replaces cuBLAS only where cuBLAS would use TF32 too (the reference sets
    float32_matmul_precision('high'), example/zinc.py:30) and for the shapes it supports."""
    # below a few thousand rows the pipeline set-up and the ticketed tail outweigh the saved pass.
    # N = 256 / 384 are correct but re-read W (N x K) from L2 once per 128-row tile: at ~54 GB/s
    # of L2->SM traffic per SM that costs more than the statistics pass saves (384 -> 384 at
    # 230 k rows: 308 us against cuBLAS 140 us + 68 us, profiles/r2_linear_stats.md) -- they
    # stay opt-in (PYGHO_B200_FUSED_GEMM_WIDE=1) until the tile is shared by a CTA pair
    if weight.shape[0] != 128 and not _FUSED_GEMM_WIDE:
        return False
    # K = 128: the epilogue (TMEM load, statistics, stores: ~5.8 us per 128-row tile) is longer than
    # the loads, 70.9 us against cuBLAS 61.7 us + statistics at 230 k rows (profiles/r2_op_rooflines.md)
    if weight.shape[1] < 256 and not _FUSED_GEMM_WIDE:
        return False
    return (torch.backends.cuda.matmul.allow_tf32 and x.dtype == torch.float32 and x.ndim == 2
            and x.is_cuda and weight.dtype == torch.float32 and x.shape[0] >= _FUSED_GEMM_MIN_ROWS
            and bool(_lib.load().pgh_linear_stats_supported(x.shape[0], x.shape[1], weight.shape[0])))


def _linear_stats_cuda(x, weight, bias, eps, momentum, running_mean, running_var, rows_dev,
                       num_batches_tracked, local):
    """-> (y, mean, rstd), or (y, local (3, C), empty) with ``local`` (SyncBN)."""
    x, weight, bias = _f32c(x), _f32c(weight), _f32c(bias)
    M, K = x.shape
    N = weight.shape[0]
    y = torch.empty((M, N), dtype=torch.float32, device=x.device)
    if local:
        a = torch.empty((3, N), dtype=torch.float32, device=x.device)
        b = a.new_empty((0,))
        mean = rstd = None
    else:
        a = torch.empty((N,), dtype=torch.float32, device=x.device)
        b = torch.empty_like(a)
        mean, rstd = a, b
    nws = int(_lib.load().pgh_linear_stats_ws_bytes(int(M)))
    ws = torch.empty((nws,), dtype=torch.uint8, device=x.device)
    call("pgh_linear_stats_f32", ptr(x), M, K, ptr(weight), N, ptr(bias), ptr(_rows_dev(rows_dev)),
         ptr(y), float(eps), float(momentum), ptr(mean), ptr(rstd), ptr(running_mean),
         ptr(running_var), ptr(a) if local else None, ptr(_nbt(num_batches_tracked)), ptr(ws),
         ws.numel(), _tickets(x.device), stream_ptr(x.device))
    _lib.count_launch()
    return y, a, b


_LIB.impl("linear_stats", _linear_stats_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::linear_stats")
def _linear_stats_fake(x, weight, bias, eps, momentum, running_mean, running_var, rows_dev,
                       num_batches_tracked, local):
    N = weight.shape[0]
    y = x.new_empty((x.shape[0], N))
    if local:
        return y, x.new_empty((3, N)), x.new_empty((0,))
    return y, x.new_empty((N,)), x.new_empty((N,))


_LIB.define("linear_bn_eval(Tensor x, Tensor weight, Tensor? bias, Tensor? gamma, Tensor? beta, "
            "Tensor running_mean, Tensor running_var, float eps, int act, Tensor? residual=None, "
            "Tensor? rows_dev=None) -> Tensor")


def _linear_bn_eval_cuda(x, weight, bias, gamma, beta, running_mean, running_var, eps, act,
                         residual=None, rows_dev=None):
    """z = act(BatchNorm_eval(x @ W^T + b)) (+ residual) in one pass (csrc/linear_stats.cu)."""
    x, weight, bias, residual = _f32c(x), _f32c(weight), _f32c(bias), _f32c(residual)
    if x.ndim != 2 or weight.ndim != 2 or weight.shape[1] != x.shape[1]:
        raise ValueError("linear_bn_eval: need x (M, K) and weight (N, K)")
    M, K = x.shape
    N = weight.shape[0]
    for name, v in (("bias", bias), ("gamma", gamma), ("beta", beta),
                    ("running_mean", running_mean), ("running_var", running_var)):
        if v is not None and v.numel() != N:
            raise ValueError(f"linear_bn_eval: {name} must have {N} elements")
    if residual is not None and residual.shape != (M, N):
        raise ValueError("linear_bn_eval: residual must have the shape of the output")
    z = torch.empty((M, N), dtype=torch.float32, device=x.device)
    call("pgh_linear_bn_eval_f32", ptr(x), M, K, ptr(weight), N, ptr(bias), ptr(_f32c(gamma)),
         ptr(_f32c(beta)), ptr(_f32c(running_mean)), ptr(_f32c(running_var)), float(eps), int(act),
         ptr(residual), ptr(_rows_dev(rows_dev)), ptr(z), stream_ptr(x.device))
    _lib.count_launch()
    return z


_LIB.impl("linear_bn_eval", _linear_bn_eval_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::linear_bn_eval")
def _linear_bn_eval_fake(x, weight, bias, gamma, beta, running_mean, running_var, eps, act,
                         residual=None, rows_dev=None):
    return x.new_empty((x.shape[0], weight.shape[0]))


_LIB.define("bn_stats_local(Tensor y, Tensor? rows_dev=None, "
            "Tensor(a!)? num_batches_tracked=None) -> Tensor")


def _bn_stats_local_cuda(y, rows_dev=None, num_batches_tracked=None):
    """Rank-local (mean, M2, count) rows (3, C) for cross-rank statistics (SyncBN)."""
    y = _f32c(y)
    rows, C = y.shape
    local = torch.empty((3, C), dtype=torch.float32, device=y.device)
    ws = _bn_ws(rows, C, y.device)
    call("pgh_bn_stats_f32", ptr(y), rows, C, ptr(_rows_dev(rows_dev)), 0.0, 0.0, None, None, None,
         None, ptr(local), ptr(_nbt(num_batches_tracked)), ptr(ws), ws.numel(), _tickets(y.device),
         stream_ptr(y.device))
    _lib.count_launch()
    return local


_LIB.impl("bn_stats_local", _bn_stats_local_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::bn_stats_local")
def _bn_stats_local_fake(y, rows_dev=None, num_batches_tracked=None):
    return y.new_empty((3, y.shape[1]))


_LIB.define("bn_sync_finalize(Tensor gathered, float eps, float momentum, Tensor? running_mean, "
            "Tensor? running_var) -> (Tensor, Tensor, Tensor)")


def _bn_sync_finalize_cuda(gathered, eps, momentum, running_mean, running_var):
    gathered = _f32c(gathered)
    world, three, C = gathered.shape
    if three != 3:
        raise ValueError("bn_sync_finalize: gathered must be (world, 3, C)")
    mean = torch.empty((C,), dtype=torch.float32, device=gathered.device)
    rstd = torch.empty_like(mean)
    inv_n = torch.empty((1,), dtype=torch.float32, device=gathered.device)
    call("pgh_bn_sync_finalize_f32", ptr(gathered), world, C, float(eps), float(momentum), ptr(mean),
         ptr(rstd), ptr(running_mean), ptr(running_var), ptr(inv_n), stream_ptr(gathered.device))
    _lib.count_launch()
    return mean, rstd, inv_n


_LIB.impl("bn_sync_finalize", _bn_sync_finalize_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::bn_sync_finalize")
def _bn_sync_finalize_fake(gathered, eps, momentum, running_mean, running_var):
    C = gathered.shape[2]
    return gathered.new_empty((C,)), gathered.new_empty((C,)), gathered.new_empty((1,))


_LIB.define("bn_act_fwd(Tensor y, Tensor mean, Tensor rstd, Tensor? gamma, Tensor? beta, int act, "
            "Tensor? residual=None, Tensor? rows_dev=None) -> Tensor")


def _bn_act_fwd_cuda(y, mean, rstd, gamma, beta, act, residual=None, rows_dev=None):
    y, residual = _f32c(y), _f32c(residual)
    rows, C = y.shape
    if residual is not None and residual.shape != y.shape:
        raise ValueError("bn_act_fwd: residual must have the shape of y")
    z = torch.empty_like(y)
    call("pgh_bn_act_res_fwd_f32", ptr(y), ptr(mean), ptr(rstd), ptr(_f32c(gamma)),
         ptr(_f32c(beta)), rows, C, ptr(_rows_dev(rows_dev)), act, ptr(residual), ptr(z),
         stream_ptr(y.device))
    _lib.count_launch()
    return z


_LIB.impl("bn_act_fwd", _bn_act_fwd_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::bn_act_fwd")
def _bn_act_fwd_fake(y, mean, rstd, gamma, beta, act, residual=None, rows_dev=None):
    return torch.empty_like(y)


_LIB.define("bn_act_bwd_reduce(Tensor dz, Tensor y, Tensor mean, Tensor rstd, Tensor? gamma, "
            "Tensor? beta, int act, Tensor? rows_dev, Tensor(a!)? dgamma_acc, "
            "Tensor(b!)? dbeta_acc) -> (Tensor, Tensor, Tensor)")


def _grad_target(t: Optional[Tensor], C: int, name: str) -> Optional[Tensor]:
    if t is not None and (t.dtype != torch.float32 or not t.is_contiguous() or t.numel() != C):
        raise ValueError(f"{name}: gradient buffer must be a contiguous float32 tensor of {C} elements")
    return t


def _bn_act_bwd_reduce_cuda(dz, y, mean, rstd, gamma, beta, act, rows_dev, dgamma_acc, dbeta_acc):
    """-> (sums (2, C), dgamma, dbeta).  With ``dgamma_acc`` / ``dbeta_acc`` the kernel ADDS into
    those buffers (a parameter's ``.grad`` view of the flat bucket) and the returned tensors are
    empty placeholders."""
    dz, y = _f32c(dz), _f32c(y)
    rows, C = y.shape
    sums = torch.empty((2, C), dtype=torch.float32, device=y.device)
    acc = dgamma_acc is not None or dbeta_acc is not None
    if acc:
        dgamma, dbeta = _grad_target(dgamma_acc, C, "dgamma"), _grad_target(dbeta_acc, C, "dbeta")
    else:
        dgamma = torch.empty((C,), dtype=torch.float32, device=y.device)
        dbeta = torch.empty_like(dgamma)
    ws = _bn_ws(rows, C, y.device)
    call("pgh_bn_act_bwd_reduce_f32", ptr(dz), ptr(y), ptr(mean), ptr(rstd), ptr(_f32c(gamma)),
         ptr(_f32c(beta)), rows, C, ptr(_rows_dev(rows_dev)), act, ptr(sums), ptr(dgamma),
         ptr(dbeta), int(acc), ptr(ws), ws.numel(), _tickets(y.device), stream_ptr(y.device))
    _lib.count_launch()
    if acc:
        e = sums.new_empty((0,))
        return sums, e, e
    return sums, dgamma, dbeta


_LIB.impl("bn_act_bwd_reduce", _bn_act_bwd_reduce_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::bn_act_bwd_reduce")
def _bn_act_bwd_reduce_fake(dz, y, mean, rstd, gamma, beta, act, rows_dev, dgamma_acc, dbeta_acc):
    C = y.shape[1]
    n = 0 if (dgamma_acc is not None or dbeta_acc is not None) else C
    return y.new_empty((2, C)), y.new_empty((n,)), y.new_empty((n,))


_LIB.define("bn_act_bwd_apply(Tensor dz, Tensor y, Tensor mean, Tensor rstd, Tensor? gamma, "
            "Tensor? beta, Tensor sums, Tensor? inv_n, int act, Tensor? rows_dev, bool want_bias, "
            "Tensor(a!)? dbias_acc) -> (Tensor, Tensor)")


def _bn_act_bwd_apply_cuda(dz, y, mean, rstd, gamma, beta, sums, inv_n, act, rows_dev, want_bias,
                           dbias_acc):
    dz, y, sums = _f32c(dz), _f32c(y), _f32c(sums)
    rows, C = y.shape
    dy = torch.empty_like(y)
    acc = dbias_acc is not None
    dbias = _grad_target(dbias_acc, C, "dbias") if acc else (
        torch.empty((C,), dtype=torch.float32, device=y.device) if want_bias else None)
    ws = _bn_ws(rows, C, y.device)
    call("pgh_bn_act_bwd_apply_f32", ptr(dz), ptr(y), ptr(mean), ptr(rstd), ptr(_f32c(gamma)),
         ptr(_f32c(beta)), ptr(sums), ptr(_f32c(inv_n)), rows, C, ptr(_rows_dev(rows_dev)), act,
         ptr(dy), ptr(dbias), int(acc), ptr(ws), ws.numel(), _tickets(y.device),
         stream_ptr(y.device))
    _lib.count_launch()
    return dy, (dbias if (want_bias and not acc) else dy.new_empty((0,)))


_LIB.impl("bn_act_bwd_apply", _bn_act_bwd_apply_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::bn_act_bwd_apply")
def _bn_act_bwd_apply_fake(dz, y, mean, rstd, gamma, beta, sums, inv_n, act, rows_dev, want_bias,
                           dbias_acc):
    C = y.shape[1]
    return torch.empty_like(y), y.new_empty((C if (want_bias and dbias_acc is None) else 0,))


_LIB.define("sum_slabs(Tensor part, Tensor(a!) out, bool accumulate) -> ()")


def _sum_slabs_cuda(part, out, accumulate):
    """out (+)= part.sum(0) for a contiguous float32 (slabs, ...) tensor, fixed order."""
    part = _f32c(part)
    n = part[0].numel()
    if out.dtype != torch.float32 or not out.is_contiguous() or out.numel() != n:
        raise ValueError("sum_slabs: out must be a contiguous float32 tensor of part[0]'s size")
    call("pgh_sum_slabs_f32", ptr(part), part.shape[0], n, ptr(out), int(accumulate),
         stream_ptr(part.device))
    _lib.count_launch()


_LIB.impl("sum_slabs", _sum_slabs_cuda, "CUDA")


@torch.library.register_fake("pygho_b200::sum_slabs")
def _sum_slabs_fake(part, out, accumulate):
    return None


_ops = torch.ops.pygho_b200


# ------------------------------------------------------------------------- autograd
def _gmr(plan, which: str, first_val: Tensor, scale: Optional[Tensor], second_val: Optional[Tensor],
         n_rows: int, aggr: int) -> Tensor:
    """One segmented reduce over grouping ``which`` of ``plan``."""
    g = plan.group(which)
    return _ops.seg_gmr(first_val, g.first, scale, second_val,
                        g.second if second_val is not None else None, g.rowptr, n_rows, aggr)


class SegGmr(torch.autograd.Function):
    """out[r] = aggr_{t in seg(r)} A[c_t] * B[d_t] with the three CSR groupings of a
    :class:`pygho_b200.plans.TriplePlan`.  Gradients flow to the value operands only
    (SURVEY.md 8b "Autograd"); max/min split the gradient evenly among ties like
    torch's ``scatter_reduce_`` backward."""

    @staticmethod
    def forward(ctx, a_val: Tensor, b_val: Optional[Tensor], plan, aggr: int):
        out = _gmr(plan, "a", a_val, None, b_val, plan.n_out, aggr)
        ctx.plan, ctx.aggr = plan, aggr
        ctx.has_b = b_val is not None
        if aggr >= 2:
            ctx.save_for_backward(a_val, b_val, out)
        else:
            ctx.save_for_backward(a_val if ctx.has_b else None, b_val)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g: Tensor):
        plan, aggr = ctx.plan, ctx.aggr
        need_a, need_b = ctx.needs_input_grad[0], ctx.has_b and ctx.needs_input_grad[1]
        g_a = g_b = None
        if aggr >= 2:
            g = g.contiguous()
            a_val, b_val, out = ctx.saved_tensors
            ga = plan.group("a")
            gs = _ops.seg_tie_scale(a_val, ga.first, b_val,
                                    ga.second if ctx.has_b else None, ga.rowptr, out, g)
            if need_a:
                gc = plan.group("c")
                g_a = _ops.seg_select_bwd(a_val, b_val, gc.second if ctx.has_b else None,
                                          gc.first, gc.rowptr, out, gs)
            if need_b:
                gd = plan.group("d")
                g_b = _ops.seg_select_bwd(b_val, a_val, gd.second, gd.first, gd.rowptr, out, gs)
            return g_a, g_b, None, None
        a_val, b_val = ctx.saved_tensors
        scale = plan.inv_count() if aggr == 1 else None
        if need_a:
            g_a = _gmr(plan, "c", g, scale, b_val if ctx.has_b else None, plan.n_a, 0)
        if need_b:
            g_b = _gmr(plan, "d", g, scale, a_val, plan.n_b, 0)
        return g_a, g_b, None, None


def seg_gmr(a_val: Optional[Tensor], b_val: Optional[Tensor], plan, aggr: str) -> Tensor:
    """Differentiable gather-multiply-segment-reduce over ``plan``; a ``None`` operand
    counts as 1 (backend/Spspmm.py:309-314).  Operands are (rows, dense) float32."""
    code = AGGR_CODE[aggr]
    if a_val is None and b_val is None:
        raise ValueError("at least one operand needs values")
    if a_val is None:
        return SegGmr.apply(b_val, None, plan.swapped(), code)
    return SegGmr.apply(a_val, b_val, plan, code)


def mask_extents(mask: Optional[Tensor]) -> Optional[Tensor]:
    """(b, 2) int32 = 1 + last valid row / column of every graph of a (b, n1, n2) mask;
    cached on the mask tensor (masks are shared by all layers of a model)."""
    if mask is None:
        return None
    cache = getattr(mask, "_pgh_cache", None)
    if cache is None:
        cache = {}
        mask._pgh_cache = cache
    e = cache.get("ext2")
    if e is None:
        e = _ops.mask_extents(mask)
        cache["ext2"] = e
    return e


_EXT3_CACHE = {}


def _ext3(eX: Optional[Tensor], tx: bool, eY: Optional[Tensor], ty: bool, eM: Optional[Tensor],
          shape) -> Optional[Tensor]:
    """Per-graph (n_i, n_j, n_k) of X' @ Y' masked by M from the (rows, cols) extents of the
    stored operands, and the graphs in descending order of their work (the queue order of the
    algo-4 kernel); ``None`` extents mean "full" -> (None, None)."""
    if eX is None and eY is None and eM is None:
        return None, None
    key = (id(eX), tx, id(eY), ty, id(eM), shape)
    hit = _EXT3_CACHE.get(key)
    if hit is not None:
        return hit[0]
    b, n_i, n_j, n_k = shape
    ref = eX if eX is not None else eY if eY is not None else eM

    def oriented(e, trans, rows, cols):
        if e is None:
            return ref.new_full((b,), rows), ref.new_full((b,), cols)
        return (e[:, 1], e[:, 0]) if trans else (e[:, 0], e[:, 1])

    rX, cX = oriented(eX, tx, n_i, n_j)
    rY, cY = oriented(eY, ty, n_j, n_k)
    rM, cM = oriented(eM, False, n_i, n_k)
    ext = torch.stack((torch.minimum(rX, rM), torch.minimum(cX, rY), torch.minimum(cY, cM)),
                      dim=1).contiguous()
    work = ext[:, 0].to(torch.int64) * ext[:, 1] * ext[:, 2]
    order = torch.argsort(work, descending=True, stable=True).to(torch.int32)
    if len(_EXT3_CACHE) > 64:
        _EXT3_CACHE.clear()
    _EXT3_CACHE[key] = ((ext, order), eX, eY, eM)      # keep the keyed tensors alive
    return ext, order


def mamamm_algo_for(algo: int, n_i: int, n_j: int, n_k: int, dense: int) -> int:
    """The tensor-core kernels (algo 1 / 2) hold one (n_i x n_j) and one (n_j x n_k) tile per
    channel: n_i, n_j <= 128, n_k <= 64, dense % 8 == 0.  Anything else runs on the exact-fp32 kernel
    (algo 0).  Decided per CALL: the gradient contractions of a forward that fits may
    not fit themselves (their (n_i, n_j, n_k) roles are permuted).  algo 4 (exact fp32 from a
    TMA-fed shared-memory ring, csrc/mamamm_smem.cu) takes any shape: the library itself runs the
    shapes its ring cannot hold on algo 0."""
    if algo in (1, 2) and (dense % 8 != 0 or n_i > 128 or n_k > 64 or n_j > 128):
        return 0
    return algo


def _mm(X, tx, eX, Y, ty, eY, mask, eM, algo):
    b = X.shape[0]
    n_i, n_j = (X.shape[2], X.shape[1]) if tx else (X.shape[1], X.shape[2])
    n_k = Y.shape[1] if ty else Y.shape[2]
    algo = mamamm_algo_for(algo, n_i, n_j, n_k, X.shape[3])
    ext, order = _ext3(eX, tx, eY, ty, eM, (b, n_i, n_j, n_k))
    return _ops.mamamm(X, tx, Y, ty, mask, ext, algo, order)


class MaMaMM(torch.autograd.Function):
    """out = mask * (A' @ B') per channel; A' / B' optionally transposed in dims (1, 2).
    ``mA`` / ``mB`` are the operands' own masks (or None): their per-graph extents bound
    what the kernels read and multiply -- exact, because operand pads are zero."""

    @staticmethod
    def forward(ctx, A, trans_a, mA, B, trans_b, mB, mask, algo):
        eA, eB, eM = mask_extents(mA), mask_extents(mB), mask_extents(mask)
        ctx.save_for_backward(A, B, mask)
        ctx.cfg = (trans_a, trans_b, algo, eA, eB, eM)
        return _mm(A, trans_a, eA, B, trans_b, eB, mask, eM, algo)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        A, B, mask = ctx.saved_tensors
        trans_a, trans_b, algo, eA, eB, eM = ctx.cfg
        # out is masked in the epilogue -> its gradient only exists where mask is True
        g = _ops.masked_fill_rows(g.contiguous(), mask, 0.0)
        g_a = g_b = None
        if ctx.needs_input_grad[0]:
            # dA'[i,j] = sum_k g[i,k] B'[j,k]  -> g @ B'^T ; stored transposed if trans_a
            if not trans_a:
                g_a = _mm(g, False, eM, B, not trans_b, eB, _ones_mask(A), None, algo)
            else:
                g_a = _mm(B, trans_b, eB, g, True, eM, _ones_mask(A), None, algo)
        if ctx.needs_input_grad[3]:
            # dB'[j,k] = sum_i A'[i,j] g[i,k] -> A'^T @ g ; stored transposed if trans_b
            if not trans_b:
                g_b = _mm(A, not trans_a, eA, g, False, eM, _ones_mask(B), None, algo)
            else:
                g_b = _mm(g, True, eM, A, trans_a, eA, _ones_mask(B), None, algo)
        return g_a, None, None, g_b, None, None, None, None


_ONES_CACHE = {}


def _ones_mask(t: Tensor) -> Tensor:
    key = (t.device, tuple(t.shape[:3]))
    m = _ONES_CACHE.get(key)
    if m is None:
        if len(_ONES_CACHE) > 16:
            _ONES_CACHE.clear()
        m = torch.ones(t.shape[:3], dtype=torch.bool, device=t.device)
        _ONES_CACHE[key] = m
    return m


class MaskedPool(torch.autograd.Function):
    @staticmethod
    def forward(ctx, data, mask, red_dims, aggr):
        out, omask = _ops.masked_pool(data, mask, red_dims, aggr)
        ctx.save_for_backward(data, mask, out)
        ctx.cfg = (red_dims, aggr)
        ctx.mark_non_differentiable(omask)
        return out, omask

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g, _gm):
        data, mask, out = ctx.saved_tensors
        red_dims, aggr = ctx.cfg
        return _ops.masked_pool_bwd(data, mask, out, g.contiguous(), red_dims, aggr), None, None, None


class MaskedFill(torch.autograd.Function):
    @staticmethod
    def forward(ctx, data, mask, value):
        ctx.save_for_backward(mask)
        return _ops.masked_fill_rows(data, mask, value)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        (mask,) = ctx.saved_tensors
        return _ops.masked_fill_rows(g.contiguous(), mask, 0.0), None, None


_FORK = os.environ.get("PYGHO_B200_FORK", "1") != "0"
_FORK_STREAMS = {}


class _Fork:
    """Run a few independent kernel launches on a second stream (fork / join with stream waits;
    inside a CUDA-graph capture this becomes a parallel branch of the graph).  At the 8-GPU
    strong-scaling point (128 graphs per GPU) single kernels no longer fill the 148 SMs, and the
    tails of independent launches -- the two halves of an SSWL aggregation, dX and dA, the dx and
    dW GEMMs of a Linear -- overlap instead of queueing.  Rules: every tensor the branch WRITES
    that is used afterwards is allocated before the fork (on the main stream); temporaries
    allocated inside the branch are only ever touched by the branch."""

    def __init__(self, device):
        self.on = _FORK and device.type == "cuda"
        if self.on:
            self.main = torch.cuda.current_stream(device)
            side = _FORK_STREAMS.get(device)
            if side is None:
                side = torch.cuda.Stream(device)
                _FORK_STREAMS[device] = side
            self.side = side
            if self.side == self.main:
                self.on = False

    def __enter__(self):
        if self.on:
            self.side.wait_stream(self.main)
            self.ctx = torch.cuda.stream(self.side)
            self.ctx.__enter__()
        return self

    def __exit__(self, *exc):
        if self.on:
            self.ctx.__exit__(*exc)
        return False

    def join(self):
        if self.on:
            self.main.wait_stream(self.side)


class SswlAggregate(torch.autograd.Function):
    """``cat([X, X (x) A, A (x) X], -1)`` of one SSWL layer (reference Conv.py:97-103) built in
    ONE buffer: the two spspmm launches write their column slice directly, and the three
    gradient contributions to X (two to A) are accumulated by the kernels themselves instead of
    materialising temporaries and adding them.  sum / mean aggregation.

    With ``tap_residual`` the function also returns ``Xv`` itself as a second output: feeding
    THAT tensor to the residual connection (``X + conv(X)``, example/zinc.py:286) routes the
    residual's gradient into this backward, where it is added to dX inside the same kernel --
    X then has a single consumer and autograd needs no separate add pass over all tuples."""

    @staticmethod
    def forward(ctx, Xv, Av, plan_xa, plan_ax, aggr, tap_residual=False, merged_bwd=None):
        n, d = Xv.shape
        cat = torch.empty((n, 3 * d), dtype=torch.float32, device=Xv.device)
        g1, g2 = plan_xa.group("a"), plan_ax.group("a")
        with _Fork(Xv.device) as fork:           # A (x) X writes its own column slice: independent
            _ops.seg_gmr_out(Av, g2.first, None, Xv, g2.second, g2.rowptr, n, aggr, cat[:, 2 * d:], False)
        if n and Av.shape[0] and fused_epilogue_ok(d, Xv, Av, cat):
            # the X (x) A launch also copies X into the first third of the buffer
            _ops.seg_gmr_fused(Xv, g1.first, None, Av, g1.second, g1.rowptr, n, aggr, None, Xv,
                               cat[:, :d], cat[:, d:2 * d])
        else:
            cat[:, :d].copy_(Xv)
            _ops.seg_gmr_out(Xv, g1.first, None, Av, g1.second, g1.rowptr, n, aggr, cat[:, d:2 * d], False)
        fork.join()
        ctx.save_for_backward(Xv, Av)
        ctx.cfg = (plan_xa, plan_ax, aggr, merged_bwd)
        if tap_residual:
            return cat, Xv.view_as(Xv)
        return cat

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g, g_res=None):
        Xv, Av = ctx.saved_tensors
        plan_xa, plan_ax, aggr, merged = ctx.cfg
        n, d = Xv.shape
        nA = Av.shape[0]
        g0, g1, g2 = g[:, :d], g[:, d:2 * d], g[:, 2 * d:]
        s1 = plan_xa.inv_count() if aggr == 1 else None
        s2 = plan_ax.inv_count() if aggr == 1 else None
        gX = gA = None
        fork = None
        if ctx.needs_input_grad[1]:      # dA on the forked stream, dX on this one
            gA = torch.empty((nA, d), dtype=torch.float32, device=g.device)
            with _Fork(g.device) as fork:
                dd = plan_xa.group("d")      # A is operand B of X (x) A
                _ops.seg_gmr_out(g1, dd.first, s1, Xv, dd.second, dd.rowptr, nA, 0, gA, False)
                c = plan_ax.group("c")       # A is operand A of A (x) X
                _ops.seg_gmr_out(g2, c.first, s2, Xv, c.second, c.rowptr, nA, 0, gA, True)
        if ctx.needs_input_grad[0] and merged is not None and aggr == 0 and n and nA \
                and g.is_contiguous() and fused_epilogue_ok(d, g, Av, g_res):
            # gX = g0 + sum over BOTH products' entries (+ residual gradient) in one launch: the
            # gradient of the concatenation is read as (3 n, d) rows, the merged plan
            # (plans.sswl_bwd_group) addresses its second and third column slice
            gX = torch.empty((n, d), dtype=torch.float32, device=g.device)
            _ops.seg_gmr_fused(g.view(3 * n, d), merged.first, None, Av, merged.second, merged.rowptr,
                               n, 0, g0, None, None, gX, g_res)
        elif ctx.needs_input_grad[0]:
            c = plan_xa.group("c")       # X is operand A of X (x) A
            if n and nA and fused_epilogue_ok(d, g, Av, g_res):
                # gX = g0 + sum(...) (+ residual gradient) in one launch: no clone, no add pass
                gX = torch.empty((n, d), dtype=torch.float32, device=g.device)
                _ops.seg_gmr_fused(g1, c.first, s1, Av, c.second, c.rowptr, n, 0, g0, None, None, gX,
                                   g_res)
            else:
                gX = g0.contiguous() if not g0.is_contiguous() else g0.clone()
                if g_res is not None:
                    gX.add_(g_res)
                _ops.seg_gmr_out(g1, c.first, s1, Av, c.second, c.rowptr, n, 0, gX, True)
            dd = plan_ax.group("d")      # X is operand B of A (x) X
            _ops.seg_gmr_out(g2, dd.first, s2, Av, dd.second, dd.rowptr, n, 0, gX, True)
        if fork is not None:
            fork.join()
        return gX, gA, None, None, None, None, None


class GatherProduct(torch.autograd.Function):
    """``out[t] = P[i_t] * Q[j_t] * V[t]``: the tuple initialisation of the reference models
    (``lin0(x)[X.indices[0]] * lin1(x)[X.indices[1]] * emb(tuplefeat)``, example/zinc.py:270-276)
    with the two gathered factors never materialised on their own: ``PQ = P[i] * Q[j]`` comes out
    of one gather-multiply launch (and is kept for the backward), the gradients of the dense
    factors are segmented reductions of ``g * V`` against the OTHER factor gathered on the fly.
    4 passes over the tuples forward and 8 backward instead of 8 and 17.
    ``pair`` = (i32, j32, rowptr_i, t_by_i, j_by_i, rowptr_j, t_by_j, i_by_j) from
    ``SparseTensor._pair_plan`` (``t_by_*`` is None when the tuples are already in that order)."""

    @staticmethod
    def forward(ctx, Pv, Qv, V, pair):
        i32, j32 = pair[0], pair[1]
        pq = _ops.seg_gmr(Pv, i32, None, Qv, j32, None, V.shape[0], 0)
        ctx.save_for_backward(Pv, Qv, V, pq)
        ctx.pair = pair
        return pq * V

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        Pv, Qv, V, pq = ctx.saved_tensors
        _i32, _j32, rp_i, t_i, j_i, rp_j, t_j, i_j = ctx.pair
        g = g.contiguous()
        gP = gQ = gV = None
        if ctx.needs_input_grad[2]:
            gV = g * pq
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
            gpq = g * V
            if ctx.needs_input_grad[0]:
                gP = _ops.seg_gmr(gpq, t_i, None, Qv, j_i, rp_i, Pv.shape[0], 0)
            if ctx.needs_input_grad[1]:
                gQ = _ops.seg_gmr(gpq, t_j, None, Pv, i_j, rp_j, Qv.shape[0], 0)
        return gP, gQ, gV, None


class EmbeddingGather(torch.autograd.Function):
    """``weight[idx]`` (``nn.Embedding``, reference example/zinc.py:233-239 encoders) through the
    gather kernel, with a deterministic weight gradient: a short chain of segmented sums over
    the cached :class:`pygho_b200.plans.EmbeddingPlan` instead of torch's per-step radix sort +
    atomic accumulation (0.66 ms per SSWL+ step for the three encoders)."""

    @staticmethod
    def forward(ctx, weight: Tensor, idx: Tensor, plan):
        n = plan.idx32.numel()
        out = _ops.seg_gmr(weight, plan.idx32, None, None, None, None, n, 0)
        ctx.plan, ctx.weight = plan, weight
        return out.reshape(tuple(idx.shape) + (weight.shape[1],))

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        plan = ctx.plan
        cur = g.reshape(-1, g.shape[-1])
        perm = plan.perm
        acc = _acc_target(ctx.weight, True)
        last = len(plan.levels) - 1
        for i, rowptr in enumerate(plan.levels):
            if i == last and acc is not None:        # last level adds into weight.grad directly
                _ops.seg_gmr_out(cur, perm, None, None, None, rowptr, rowptr.numel() - 1, 0, acc, True)
                return None, None, None
            cur = _ops.seg_gmr(cur, perm, None, None, None, rowptr, rowptr.numel() - 1, 0)
            perm = None
        return cur, None, None


ACT_CODE = {"none": 0, "silu": 1, "relu": 2}


def _tall_skinny_tn(a: Tensor, b: Tensor, chunks: int = 64, acc: Optional[Tensor] = None
                    ) -> Optional[Tensor]:
    """a^T @ b for (rows, m) and (rows, n) with rows >> m, n (weight gradients over all
    tuples).  cuBLAS does not split K for this shape and leaves most SMs idle; cutting the
    rows into `chunks` slabs turns it into one batched GEMM that fills the GPU, followed by a
    reduction over the slabs.  With ``acc`` (a (m, n) gradient buffer) the result is ADDED to it
    in the same launches (cuBLAS beta = 1 / accumulate flag of the segmented sum) and None is
    returned: no separate gradient-accumulation kernel."""
    rows = a.shape[0]
    if rows < 64 * chunks or a.shape[1] > 1024 or b.shape[1] > 1024:
        if acc is not None:
            acc.addmm_(a.t(), b)
            return None
        return a.t().mm(b)
    per = rows // chunks
    main = per * chunks
    m, n = a.shape[1], b.shape[1]
    part = torch.bmm(a[:main].view(chunks, per, m).transpose(1, 2), b[:main].view(chunks, per, n))
    if (m * n) % 4 == 0 and part.data_ptr() % 16 == 0 and (acc is None or acc.data_ptr() % 16 == 0):
        out = acc if acc is not None else torch.empty((m, n), dtype=torch.float32, device=a.device)
        _ops.sum_slabs(part, out, acc is not None)
    elif acc is not None:
        acc.add_(part.sum(0))
        out = acc
    else:
        out = part.sum(0)
    if main < rows:
        out.addmm_(a[main:].t(), b[main:])
    return None if acc is not None else out


_DIRECT_GRADS = True
_FUSED_GEMM = os.environ.get("PYGHO_B200_FUSED_GEMM", "1") != "0"
_FUSED_GEMM_MIN_ROWS = 4096
_FUSED_GEMM_WIDE = os.environ.get("PYGHO_B200_FUSED_GEMM_WIDE", "0") == "1"


def set_fused_linear_stats(flag: bool) -> None:
    """Use the TMA / tcgen05 GEMM with the statistics epilogue for Linear -> BatchNorm blocks
    (default on; off = cuBLAS GEMM + separate statistics pass)."""
    global _FUSED_GEMM
    _FUSED_GEMM = bool(flag)



def set_direct_grad_accumulation(flag: bool) -> None:
    """When a parameter already has a ``.grad`` buffer (e.g. a view of the flat all-reduce
    bucket, pygho_b200/dist.py), the fused backward kernels ADD their parameter gradients into
    it directly and hand autograd ``None`` -- no AccumulateGrad add kernel per parameter
    (90 tiny launches per SSWL+ step).  Semantics are unchanged (gradients accumulate)."""
    global _DIRECT_GRADS
    _DIRECT_GRADS = bool(flag)


def _acc_target(p: Optional[Tensor], need: bool) -> Optional[Tensor]:
    """``p.grad`` if the gradient of parameter ``p`` can be accumulated in place."""
    if not (_DIRECT_GRADS and need) or p is None:
        return None
    g = getattr(p, "grad", None)
    if g is None or g.dtype != torch.float32 or not g.is_contiguous() or g.shape != p.shape \
            or g.data_ptr() % 16 or not g.is_cuda:
        return None
    return g


class LinearBNAct(torch.autograd.Function):
    """z = act(BatchNorm_train(x @ W^T + b)) for 2-D x: the reference MLP block
    (honn/utils.py:85-142) with the normalisation/activation passes fused.  The GEMMs stay
    with cuBLAS (torch.addmm / mm); only the HBM-bound elementwise + reduction work is ours.
    Saves x and the Linear output y; the normalised tensor is recomputed in the backward.

    ``rows_dev``: device count of valid rows of capacity-padded tensors (pygho_b200/static.py).
    ``group``: a torch.distributed process group -> statistics over the rows of ALL ranks
    (SyncBN: sharded training equals single-process training on the global batch)."""

    @staticmethod
    def forward(ctx, x, weight, bias, gamma, beta, running_mean, running_var, momentum, eps, act,
                residual=None, rows_dev=None, group=None, num_batches_tracked=None):
        fused_gemm = _FUSED_GEMM and linear_stats_ok(x, weight)
        inv_n = None
        if fused_gemm:      # GEMM + statistics in one pass (TMA + tcgen05, csrc/linear_stats.cu)
            y, mean, rstd = _ops.linear_stats(x, weight, bias, eps, momentum, running_mean,
                                              running_var, rows_dev, num_batches_tracked,
                                              group is not None)
        else:
            y = torch.nn.functional.linear(x, weight, bias)
        if group is None:
            if not fused_gemm:
                mean, rstd = _ops.bn_stats(y, eps, momentum, running_mean, running_var, rows_dev,
                                           num_batches_tracked)
        else:
            import torch.distributed as dist
            local = mean if fused_gemm else _ops.bn_stats_local(y, rows_dev, num_batches_tracked)
            gathered = torch.empty((dist.get_world_size(group),) + tuple(local.shape),
                                   dtype=local.dtype, device=local.device)
            if dist.get_backend(group) == "nccl":
                dist.all_gather_into_tensor(gathered, local, group=group)
            else:       # gloo (tests) has no CUDA all-gather: sum of one-hot placed triples
                gathered.zero_()
                gathered[dist.get_rank(group)].copy_(local)
                dist.all_reduce(gathered, op=dist.ReduceOp.SUM, group=group)
            mean, rstd, inv_n = _ops.bn_sync_finalize(gathered, eps, momentum, running_mean,
                                                      running_var)
        z = _ops.bn_act_fwd(y, mean, rstd, gamma, beta, act, residual, rows_dev)  # + residual
        ctx.save_for_backward(x, weight, y, mean, rstd, gamma, beta)
        ctx.act = act
        ctx.extra = (bias, rows_dev, group, inv_n)
        return z

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dz):
        x, weight, y, mean, rstd, gamma, beta = ctx.saved_tensors
        bias, rows_dev, group, inv_n = ctx.extra
        need = ctx.needs_input_grad
        need_bias = bias is not None and need[2]
        acc_w, acc_b = _acc_target(weight, need[1]), _acc_target(bias, need_bias)
        acc_g = _acc_target(gamma, gamma is not None and need[3])
        acc_be = _acc_target(beta, beta is not None and need[4])
        if (acc_g is None) != (acc_be is None):
            acc_g = acc_be = None
        sums, dgamma, dbeta = _ops.bn_act_bwd_reduce(dz, y, mean, rstd, gamma, beta, ctx.act,
                                                     rows_dev, acc_g, acc_be)
        if group is not None:
            import torch.distributed as dist
            dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
        dy, dbias = _ops.bn_act_bwd_apply(dz, y, mean, rstd, gamma, beta, sums, inv_n, ctx.act,
                                          rows_dev, need_bias, acc_b)
        if need[0] and need[1] and acc_w is not None:
            # dW (accumulated into the gradient buffer) on the forked stream, dx on this one
            with _Fork(dy.device) as fork:
                _tall_skinny_tn(dy, x, acc=acc_w)
            dx, dw = dy.mm(weight), None
            fork.join()
        else:
            dx = dy.mm(weight) if need[0] else None
            dw = _tall_skinny_tn(dy, x, acc=acc_w) if need[1] else None
        return (dx, dw, dbias if (need_bias and acc_b is None) else None,
                dgamma if (gamma is not None and need[3] and acc_g is None) else None,
                dbeta if (beta is not None and need[4] and acc_be is None) else None,
                None, None, None, None, None,
                dz if (len(need) > 10 and need[10]) else None,   # residual: gradient passes through
                None, None, None)


# Output widths N at which the one-pass eval kernel beats cuBLAS + the bn_act_fwd pass: none on a
# B200 (1000 W).  At 230 147 rows with SiLU it takes 221 / 210 / 512 / 877 us for 384->128,
# 128->128, 384->256 and 384->384 against 132 / 98 / 201 / 308 us for the fallback
# (profiles/eval_times.txt, DESIGN.md section 4.6): the four epilogue warps, one per SM
# sub-partition, are issue-bound on scale / shift / SiLU / stores, and N > 128 re-reads W per tile.
_EVAL_GEMM_WIDTHS: tuple = ()


def linear_bn_eval_ok(x: Tensor, weight: Tensor) -> bool:
    """Whether :func:`linear_bn_eval` runs the one-pass TF32 kernel for this shape: TF32 allowed
    (as for :func:`linear_stats_ok`), enough rows, a supported shape and a width where the
    kernel was measured faster than the fallback."""
    return (torch.backends.cuda.matmul.allow_tf32 and x.dtype == torch.float32 and x.ndim == 2
            and x.is_cuda and weight.dtype == torch.float32 and x.shape[0] >= _FUSED_GEMM_MIN_ROWS
            and weight.shape[0] in _EVAL_GEMM_WIDTHS
            and bool(_lib.load().pgh_linear_stats_supported(x.shape[0], x.shape[1], weight.shape[0])))


def linear_bn_eval(x: Tensor, weight: Tensor, bias: Optional[Tensor], bn: torch.nn.BatchNorm1d,
                   act: str, residual: Optional[Tensor] = None,
                   rows_dev: Optional[Tensor] = None) -> Tensor:
    """Inference of a Linear -> BatchNorm1d (eval: running statistics) -> ``act`` block on 2-D
    ``x``, plus ``residual``: ``act((x W^T + b - running_mean) / sqrt(running_var + eps) * gamma
    + beta) (+ residual)``.  Rows >= ``rows_dev`` (capacity-padded batches) are 0.  Not
    differentiable, and never writes the BatchNorm's running statistics.

    One pass through the TMA / tcgen05 GEMM with the BatchNorm in its epilogue
    (csrc/linear_stats.cu) where :func:`linear_bn_eval_ok`; otherwise ``F.linear`` followed by the
    fused BatchNorm-apply kernel with ``mean = running_mean``, ``rstd = rsqrt(running_var + eps)``."""
    code = ACT_CODE[act]
    if linear_bn_eval_ok(x, weight):
        return _ops.linear_bn_eval(x, weight, bias, bn.weight, bn.bias, bn.running_mean,
                                   bn.running_var, bn.eps, code, residual, rows_dev)
    y = torch.nn.functional.linear(x, weight, bias)
    rstd = torch.rsqrt(bn.running_var + bn.eps)
    return _ops.bn_act_fwd(y, bn.running_mean, rstd, bn.weight, bn.bias, code, residual, rows_dev)
