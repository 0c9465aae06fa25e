"""CPU-side checks of the drop-in boundary: the C-ABI library loads without a GPU and
exports every symbol include/pygho_b200.h declares; the Python binding table matches the
header; the host-side API mirror exists with the reference's names; CUDA-only ops fail
loudly on CPU tensors (no fallback)."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "pygho_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(pgh_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from pygho_b200 import _lib
    assert os.path.exists(_lib.LIB_PATH), "run __graft_entry__.build() first"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    names = _declared()
    assert len(names) >= 35
    for name in names:
        assert hasattr(lib, name), f"{name} declared in include/pygho_b200.h but not exported"


def test_binding_table_matches_header():
    from pygho_b200 import _lib
    assert sorted(_lib.SIGNATURES) == _declared()
    lib = _lib.load()
    assert lib.pgh_abi_version() == 4
    assert lib.pgh_last_error() is not None


def test_size_queries_need_no_gpu():
    from pygho_b200 import _lib
    # (cub's own temp sizes need a device; the fixed parts of the layouts do not)
    assert _lib.size_query("pgh_sort_ws_bytes", 1000) >= 4000
    assert _lib.size_query("pgh_unique_ws_bytes", 1000) >= 0
    assert _lib.size_query("pgh_match_ws_bytes", 1000) >= 8000
    assert _lib.size_query("pgh_compact_ws_bytes", 1000) >= 8000
    assert int(_lib.load().pgh_bn_ws_bytes(100000, 128)) > 0


def test_argument_errors_are_reported():
    from pygho_b200 import _lib
    with pytest.raises(_lib.KernelError, match="a_val and out are required"):
        _lib.call("pgh_seg_gmr_f32", None, None, None, None, None, None, 4, 0, 8, 0, None, None)
    with pytest.raises(_lib.KernelError, match="aggr"):
        _lib.call("pgh_seg_gmr_f32", 16, None, None, None, None, None, 4, 0, 8, 9, 16, None)
    with pytest.raises(_lib.KernelError, match="set_tuning: key"):
        _lib.call("pgh_set_tuning", 0, 2)


def test_api_surface_names():
    import pygho_b200
    from pygho_b200 import backend
    from pygho_b200.honn import Conv, MaOperator, SpOperator, TensorOp, utils
    assert pygho_b200.SparseTensor is backend.SparseTensor
    for name in ("spspmm", "spspmpnn", "spspmm_ind", "filterind", "spsphadamard",
                 "spsphadamard_ind", "ptr2batch", "deg2batch", "spmm", "mamamm",
                 "torch_scatter_reduce", "indicehash", "decodehash", "indicehash_tight",
                 "decodehash_tight", "coalesce", "filterinf", "MaskedTensor"):
        assert hasattr(backend, name), name
    for name in ("parse_precomputekey", "KEYSEP", "OpNodeMessagePassing", "OpMessagePassing",
                 "Op2FWL", "OpMessagePassingOnSubg2D", "OpMessagePassingOnSubg3D",
                 "OpMessagePassingCrossSubg2D", "OpDiag", "OpDiag2D", "OpPooling",
                 "OpPoolingSubg2D", "OpPoolingSubg3D", "OpPoolingCrossSubg2D", "OpUnpooling",
                 "OpUnpoolingSubgNodes2D", "OpUnpoolingRootNodes2D"):
        assert hasattr(SpOperator, name), name
    for name in ("OpNodeMessagePassing", "OpSpNodeMessagePassing", "OpMessagePassing", "Op2FWL",
                 "OpMessagePassingOnSubg2D", "OpMessagePassingOnSubg3D",
                 "OpMessagePassingCrossSubg2D", "OpSpMessagePassingOnSubg2D", "OpDiag2D",
                 "OpPooling", "OpPoolingSubg2D", "OpPoolingSubg3D", "OpPoolingCrossSubg2D",
                 "OpUnpoolingSubgNodes2D", "OpUnpoolingRootNodes2D"):
        assert hasattr(MaOperator, name), name
    for name in ("OpNodeMessagePassing", "Op2FWL", "OpMessagePassingOnSubg2D",
                 "OpMessagePassingOnSubg3D", "OpMessagePassingCrossSubg2D", "OpDiag2D",
                 "OpPoolingSubg2D", "OpPoolingSubg3D", "OpPoolingCrossSubg2D",
                 "OpUnpoolingSubgNodes2D", "OpUnpoolingRootNodes2D"):
        assert hasattr(TensorOp, name), name
    for name in ("NGNNConv", "SSWLConv", "I2Conv", "DSSGNNConv", "PPGNConv", "GNNAKConv"):
        assert hasattr(Conv, name), name
    for name in ("MLP", "BatchNorm", "LayerNorm", "NoneNorm", "NormMomentumScheduler"):
        assert hasattr(utils, name), name


def test_precompute_keys_match_reference_format():
    from pygho_b200.honn import Conv
    from pygho_b200.honn.SpOperator import parse_precomputekey
    mlp = {"numlayer": 1, "tailact": True, "norm": "bn", "act": "silu"}
    assert parse_precomputekey(Conv.NGNNConv(8, 8, "sum", "SS", dict(mlp))) == ["X___X___1___A___0"]
    assert parse_precomputekey(Conv.SSWLConv(8, 8, "sum", "SS", dict(mlp))) == \
        ["X___A___1___X___0", "X___X___1___A___0"]
    assert parse_precomputekey(Conv.PPGNConv(8, 8, "sum", "SS", dict(mlp))) == ["X___X___1___X___0"]
    assert parse_precomputekey(Conv.I2Conv(8, 8, "sum", "SS", dict(mlp))) == ["X___X___2___A___0"]
    assert parse_precomputekey(Conv.PPGNConv(8, 8, "sum", "DD", dict(mlp))) == []
    with pytest.raises(AssertionError):
        Conv.PPGNConv(8, 8, "max", "DD", dict(mlp))          # dense mode is sum only


def test_mlp_state_dict_layout_matches_reference():
    """Parameter names of the MLP are the reference's (so checkpoints / goldens load)."""
    from pygho_b200.honn.utils import MLP
    keys = list(MLP(12, 4, 2, True, norm="bn", act="silu").state_dict())
    assert keys[:2] == ["lins.0.weight", "lins.0.bias"]
    assert "lins.1.norm.running_mean" in keys and "lins.3.weight" in keys and "lins.4.norm.weight" in keys
    # CPU tensors take the stock torch path (MLP is host logic), fused kernels are CUDA only
    out = MLP(12, 4, 2, True)(torch.randn(5, 12))
    assert out.shape == (5, 4)


def test_no_cpu_fallback_for_kernels():
    import pygho_b200.ops  # noqa: F401
    from pygho_b200.backend import SparseTensor, torch_scatter_reduce
    with pytest.raises(Exception):
        torch.ops.pygho_b200.seg_gmr(torch.ones(2, 4), None, None, None, None, None, 2, 0)
    with pytest.raises(Exception):
        torch_scatter_reduce(0, torch.ones(3, 4), torch.tensor([0, 1, 1]), 2, "sum")
    st = SparseTensor(torch.tensor([[0, 1], [1, 0]]), torch.ones(2, 4), (2, 2, 4), is_coalesced=True)
    assert st.nnz == 2 and st.sparseshape == (2, 2) and st.denseshape == (4,)
    with pytest.raises(Exception):
        st.sum([1])


def test_synthetic_batches_follow_the_collate_contract():
    import numpy as np
    from pygho_b200.hodata.synthetic import make_batch
    hb = make_batch(16, seed=0)
    assert hb.num_graphs == 16 and hb.x.shape[0] == hb.num_nodes == int(hb.node_ptr[-1])
    assert np.array_equal(hb.batch, np.repeat(np.arange(16), np.diff(hb.node_ptr)))
    # block diagonal: both endpoints of every edge / tuple are in the same graph
    assert np.array_equal(hb.batch[hb.edge_index[0]], hb.batch[hb.edge_index[1]])
    assert np.array_equal(hb.batch[hb.tupleid[0]], hb.batch[hb.tupleid[1]])
    key = hb.tupleid[0] * hb.num_nodes + hb.tupleid[1]
    assert np.all(np.diff(key) > 0)                      # sorted, duplicate free (coalesced)
    ek = hb.edge_index[0] * hb.num_nodes + hb.edge_index[1]
    assert np.all(np.diff(ek) > 0)
    rev = hb.edge_index[1] * hb.num_nodes + hb.edge_index[0]
    assert np.array_equal(np.sort(rev), ek)              # symmetric
    assert hb.tuplefeat.min() == 0 and hb.tuplefeat.max() <= 3
    sizes = np.diff(hb.node_ptr)
    assert sizes.min() >= 9 and sizes.max() <= 37
    hb3 = make_batch(2, seed=1, tuples="i2")
    assert hb3.tupleid.shape[0] == 3 and hb3.tuplefeat.shape[1] == 2
