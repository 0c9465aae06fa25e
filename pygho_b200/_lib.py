"""ctypes binding of ``libpygho_b200.so`` (the C ABI declared in ``include/pygho_b200.h``).

There is no CPU fallback: if the shared library is missing, or a kernel is asked to
run on a non-CUDA tensor, the call raises.  Build the library with
``python -c "import __graft_entry__ as g; g.build()"`` or ``pygho_b200/csrc/build.sh``.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpygho_b200.so")

_p, _i, _i64, _sz, _f = C.c_void_p, C.c_int, C.c_int64, C.c_size_t, C.c_float
_u64 = C.c_uint64

# name -> (restype, argtypes); mirrors include/pygho_b200.h one to one
SIGNATURES = {
    "pgh_last_error": (C.c_char_p, []),
    "pgh_abi_version": (_i, []),
    "pgh_device_info": (_i, [_p]),
    "pgh_set_tuning": (_i, [_i, _i]),
    "pgh_debug_trace": (_i, [_p, _i64]),
    "pgh_seg_gmr_f32": (_i, [_p, _p, _p, _p, _p, _p, _i64, _i64, _i64, _i, _p, _p]),
    "pgh_seg_gmr_ld_f32": (_i, [_p, _i64, _p, _p, _p, _i64, _p, _p, _i64, _i64, _i64, _i, _i, _p, _i64, _p]),
    "pgh_seg_gmr_fused_f32": (_i, [_p, _i64, _p, _p, _p, _i64, _p, _p, _i64, _i64, _i64, _i, _p, _i64,
                                   _p, _i64, _p, _i64, _p, _i64, _p, _i64, _p]),
    "pgh_seg_tie_scale_f32": (_i, [_p, _p, _p, _p, _p, _i64, _i64, _p, _p, _p, _p]),
    "pgh_seg_select_bwd_f32": (_i, [_p, _p, _p, _p, _p, _i64, _i64, _p, _p, _p, _p]),
    "pgh_inv_count_f32": (_i, [_p, _i64, _p, _p]),
    "pgh_seg_reduce_i64": (_i, [_p, _p, _p, _i64, _i64, _i, _p, _p]),
    "pgh_pack_keys": (_i, [_p, _i64, _p, _i, _i, _i64, _p, _p, _p]),
    "pgh_unpack_keys": (_i, [_p, _i64, _i, _i, _p, _i64, _p]),
    "pgh_pack_tight": (_i, [_p, _i64, _p, _p, _i, _i64, _p, _p, _p]),
    "pgh_unpack_tight": (_i, [_p, _i64, _p, _i, _p, _i64, _p]),
    "pgh_multi_copy": (_i, [_p, _p, _p, _i, _p]),
    "pgh_merge_groups_i32": (_i, [_p, _p, _p, _i64, _p, _p, _p, _i64, _i64, _i, _i, _i, _p, _p, _p, _p]),
    "pgh_embedding_plan_ws_bytes": (_sz, [_i64]),
    "pgh_embedding_plan": (_i, [_p, _i, _i64, _i64, _i64, _p, _p, _p, _i64, _p, _p, _sz, _p]),
    "pgh_acd_regroup_ws_bytes": (_sz, [_i64]),
    "pgh_acd_regroup": (_i, [_p, _i64, _i64, _i64, _i64, _i, _p] + [_p] * 9 + [_p, _sz, _p]),
    "pgh_sort_ws_bytes": (_sz, [_i64]),
    "pgh_sort_keys_perm": (_i, [_p, _i64, _i, _p, _p, _p, _sz, _p]),
    "pgh_sort_i32_perm": (_i, [_p, _i64, _i, _p, _p, _p, _sz, _p]),
    "pgh_unique_ws_bytes": (_sz, [_i64]),
    "pgh_unique_sorted": (_i, [_p, _i64, _p, _p, _p, _p, _sz, _p]),
    "pgh_rowptr_from_sorted": (_i, [_p, _i64, _i64, _p, _p]),
    "pgh_match_ws_bytes": (_sz, [_i64]),
    "pgh_match_ranges": (_i, [_p, _i64, _p, _i64, _p, _p, _p, _sz, _p]),
    "pgh_expand_pairs": (_i, [_p, _p, _p, _i64, _i64, _p, _p, _p]),
    "pgh_pair_keys": (_i, [_p, _i64, _i, _i, _p, _i64, _i, _i, _p, _p, _i64, _i, _p, _p, _p]),
    "pgh_lookup_sorted": (_i, [_p, _i64, _p, _i64, _p, _p]),
    "pgh_compact_ws_bytes": (_sz, [_i64]),
    "pgh_compact_triples": (_i, [_p, _p, _p, _p, _i64, _p, _p, _p, _p, _p, _sz, _p]),
    "pgh_i64_to_i32": (_i, [_p, _i64, _p, _p, _p]),
    "pgh_i32_to_i64": (_i, [_p, _i64, _p, _p]),
    "pgh_gather_i32": (_i, [_p, _p, _i64, _p, _p]),
    "pgh_gather_i64_as_i32": (_i, [_p, _p, _i64, _p, _p]),
    "pgh_check_sorted_i64": (_i, [_p, _i64, _i, _p, _p]),
    "pgh_mamamm_f32": (_i, [_p, _i, _p, _i, _p, _p, _p, _i64, _i64, _i64, _i64, _i64, _i, _p, _p]),
    "pgh_mask_extents": (_i, [_p, _i64, _i64, _i64, _p, _p]),
    "pgh_masked_pool_f32": (_i, [_p, _p, _i64, _i64, _i64, _i64, _i, _i, _p, _p, _p]),
    "pgh_masked_pool_bwd_f32": (_i, [_p, _p, _p, _p, _i64, _i64, _i64, _i64, _i, _i, _p, _p]),
    "pgh_masked_fill_f32": (_i, [_p, _p, _i64, _i64, _f, _p, _p]),
    "pgh_bn_ws_bytes": (_sz, [_i64, _i64]),
    "pgh_bn_stats_f32": (_i, [_p, _i64, _i64, _p, _f, _f, _p, _p, _p, _p, _p, _p, _p, _sz, _p, _p]),
    "pgh_sum_slabs_f32": (_i, [_p, _i64, _i64, _p, _i, _p]),
    "pgh_adamw_flat_f32": (_i, [_p, _p, _p, _p, _i64, _p, _f, _f, _f, _f, _f, _f, _p]),
    "pgh_linear_stats_supported": (_i, [_i64, _i64, _i64]),
    "pgh_linear_stats_ws_bytes": (_sz, [_i64]),
    "pgh_linear_stats_f32": (_i, [_p, _i64, _i64, _p, _i64, _p, _p, _p, _f, _f, _p, _p, _p, _p, _p, _p,
                                  _p, _sz, _p, _p]),
    "pgh_linear_bn_eval_f32": (_i, [_p, _i64, _i64, _p, _i64, _p, _p, _p, _p, _p, _f, _i, _p, _p, _p, _p]),
    "pgh_bn_sync_finalize_f32": (_i, [_p, _i64, _i64, _f, _f, _p, _p, _p, _p, _p, _p]),
    "pgh_bn_act_res_fwd_f32": (_i, [_p, _p, _p, _p, _p, _i64, _i64, _p, _i, _p, _p, _p]),
    "pgh_bn_act_bwd_reduce_f32": (_i, [_p, _p, _p, _p, _p, _p, _i64, _i64, _p, _i, _p, _p, _p, _i,
                                       _p, _sz, _p, _p]),
    "pgh_bn_act_bwd_apply_f32": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _i64, _i64, _p, _i, _p, _p, _i,
                                      _p, _sz, _p, _p]),
    "pgh_graph_dist_u8": (_i, [_p, _p, _p, _p, _p, _i64, _i64, _i, _p, _p, _p]),
    "pgh_khop_emit": (_i, [_p, _p, _p, _p, _p, _i64, _i64, _p, _p, _p]),
    "pgh_i2_count": (_i, [_p, _p, _p, _p, _p, _p, _i64, _i, _p, _p]),
    "pgh_i2_emit": (_i, [_p, _p, _p, _p, _p, _p, _p, _i64, _i64, _i, _p, _p, _p]),
    "pgh_spd_dense_i64": (_i, [_p, _p, _p, _i64, _i64, _i, _i64, _p, _p, _p]),
    "pgh_resistance_f32": (_i, [_p, _p, _p, _p, _p, _i64, _i64, _p, _p]),
    "pgh_rd_dense_f32": (_i, [_p, _p, _p, _i64, _i64, _f, _p, _p, _p]),
    "pgh_pad_rows": (_i, [_p, _p, _i64, _i64, _i64, _i, _u64, _p, _p, _p]),
    "pgh_dense_adj": (_i, [_p, _p, _p, _p, _p, _i64, _i64, _i64, _i64, _i, _u64, _p, _p, _p]),
}

AGGR_CODE = {"sum": 0, "mean": 1, "max": 2, "min": 3, "amax": 2, "amin": 3}

_lib: Optional[C.CDLL] = None


class KernelError(RuntimeError):
    """A C-ABI entry point returned a non-zero status."""


def load() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: the CUDA kernels are the only implementation of "
                "pygho_b200 (no CPU fallback). Run pygho_b200/csrc/build.sh first.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the ABI lost a symbol
            fn.restype = res
            fn.argtypes = args
        if os.environ.get("PYGHO_B200_NO_PDL"):
            lib.pgh_set_tuning(8, 0)     # launch every kernel fully serialised (A/B measurements)
        _lib = lib
    return _lib


def call(name: str, *args):
    """Call ``name`` and raise :class:`KernelError` on a non-zero status."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        msg = lib.pgh_last_error()
        raise KernelError(f"{name} failed with status {rc}: {msg.decode() if msg else ''}")


def size_query(name: str, n: int) -> int:
    return int(getattr(load(), name)(int(n)))


def ptr(t: Optional[torch.Tensor]):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr(device: torch.device):
    """Raw cudaStream_t of torch's current stream on ``device`` (thread-local, follows
    ``torch.cuda.stream(...)`` contexts and graph capture).  The raw getter is ~10x cheaper
    than building a ``torch.cuda.Stream`` object (0.9 ms per training step, profiles/
    host_profile.py)."""
    idx = device.index
    if idx is None:
        idx = torch.cuda.current_device()
    return torch._C._cuda_getCurrentRawStream(idx)


def require_cuda(*tensors: Optional[torch.Tensor]) -> torch.device:
    """All given tensors must live on one CUDA device; there is no CPU path."""
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError(
                "pygho_b200 operators run on CUDA tensors only (got a "
                f"{t.device} tensor); there is no CPU fallback")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f"tensors on different devices: {dev} vs {t.device}")
    if dev is None:
        raise RuntimeError("at least one tensor is required")
    return dev


_launch_count = 0


def count_launch(n: int = 1) -> None:
    global _launch_count
    _launch_count += n


def launches() -> int:
    """Number of pygho_b200 kernel-launching C calls made so far in this process."""
    return _launch_count
