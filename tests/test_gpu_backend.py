"""GPU parity: the CUDA path (through the C ABI) against the oracle and the golden vectors
produced by the real reference.  Indices bit-exact; fp32 values within 1e-5 relative."""
import numpy as np
import pytest
import torch

from oracle import pygho_oracle as O
from oracle import torch_oracle as TO

pytestmark = pytest.mark.gpu
DEV = "cuda"
RTOL = 1e-5


def T(x, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(x)).to(DEV)
    return t.to(dtype) if dtype is not None else t


def N(t):
    return t.detach().cpu().numpy()


def close(a, b, rtol=RTOL):
    a = N(a) if isinstance(a, torch.Tensor) else np.asarray(a)
    b = N(b) if isinstance(b, torch.Tensor) else np.asarray(b)
    assert a.shape == b.shape, (a.shape, b.shape)
    scale = max(1.0, float(np.abs(b).max()) if b.size else 1.0)
    err = float(np.abs(a.astype(np.float64) - b.astype(np.float64)).max(initial=0.0))
    assert err <= rtol * scale, err


def canon(plan):
    p = N(plan)
    return p[:, np.lexsort((p[2], p[1], p[0]))]


@pytest.fixture(scope="module")
def B():
    import pygho_b200.backend as B
    return B


# ------------------------------------------------------------------------------ hashing
def test_hash_roundtrip_and_golden(B, golden):
    g = golden("hash")
    for sd in (2, 3, 5):
        ind = T(g[f"ind{sd}"])
        h = B.indicehash(ind)
        assert np.array_equal(N(h), g[f"hash{sd}"])
        assert np.array_equal(N(B.decodehash(h, sd)), g[f"ind{sd}"])
        ht = B.indicehash_tight(ind, T(g[f"shape{sd}"]))
        assert np.array_equal(N(ht), g[f"tight{sd}"])
        assert np.array_equal(N(B.decodehash_tight(ht, T(g[f"shape{sd}"]))), g[f"ind{sd}"])
    assert np.array_equal(N(B.ptr2batch(T(g["ptr"]), 16)), g["ptr2batch"])
    assert np.array_equal(N(B.deg2batch(T(g["deg"]), 11)), g["deg2batch"])


def test_hash_rejects_bad_indices(B):
    with pytest.raises(AssertionError):
        B.indicehash(torch.tensor([[0, -1], [1, 2]], device=DEV))
    with pytest.raises(AssertionError):
        B.indicehash(torch.tensor([[0, 1 << 40], [1, 2]], device=DEV))


def test_no_cpu_fallback(B):
    ind = torch.tensor([[0, 1], [1, 0]])
    with pytest.raises(Exception):
        B.SparseTensor(ind, torch.ones(2, 4), (2, 2, 4), is_coalesced=False)
    with pytest.raises(Exception):
        B.torch_scatter_reduce(0, torch.ones(2, 4), torch.tensor([0, 1]), 2, "sum")


# ------------------------------------------------------------------ coalesce / create
def test_coalesce_golden(B, golden):
    g = golden("coalesce")
    for red in ("sum", "mean", "max", "min"):
        st = B.SparseTensor(T(g["ind"]), T(g["val"]), (2, 3, 5, 7), False, red)
        assert np.array_equal(N(st.indices), g[f"ind_{red}"])
        close(st.values, g[f"val_{red}"])
        si = B.SparseTensor(T(g["ind"]), T(g["ival"]), (2, 3, 5), False, red)
        assert np.array_equal(N(si.values), g[f"ival_{red}"])
        close(B.torch_scatter_reduce(0, T(g["s_src"]), T(g["s_idx"]), 50, red), g[f"s_{red}"])


def test_create_matches_torch_sparse(B):
    # reference tests/test_backend_sparse.py:62-85
    gen = torch.Generator().manual_seed(0)
    n, m, l, nnz, d = 2, 3, 5, 23, 7
    ind = torch.stack([torch.randint(0, s, (nnz,), generator=gen) for s in (n, m, l)])
    val = torch.randn((nnz, d), generator=gen)
    A1 = torch.sparse_coo_tensor(ind, val, size=(n, m, l, d)).coalesce()
    A2 = B.SparseTensor(ind.to(DEV), val.to(DEV), (n, m, l, d), False)
    assert torch.equal(A2.indices.cpu(), A1.indices())
    close(A2.values, A1.values(), 5e-5)
    A2f = B.SparseTensor.from_torch_sparse_coo(
        torch.sparse_coo_tensor(ind, val, size=(n, m, l, d)).to(DEV))
    assert torch.equal(A2f.indices, A2.indices)
    close(A2f.values, A2.values)
    close(A2.to_torch_sparse_coo().to_dense(), A1.to_dense(), 5e-5)


# -------------------------------------------------------------------------------- plans
def test_plans_golden(B, golden):
    g = golden("plans")
    for tag in ("mm10", "mm01", "mm11", "mm00", "t33", "t32"):
        d1, d2 = (int(v) for v in g[f"{tag}_dims"])
        tar, bcd = B.spspmm_ind(T(g[f"{tag}_i1"]), d1, T(g[f"{tag}_i2"]), d2)
        assert np.array_equal(N(tar), g[f"{tag}_tar"]), tag
        assert np.array_equal(canon(bcd), g[f"{tag}_bcd"]), tag
        assert np.all(np.diff(N(bcd[0])) >= 0)
        if f"{tag}_tgt" in g:
            tgt = T(g[f"{tag}_tgt"])
            assert np.array_equal(N(B.spsphadamard_ind(tgt, tar)), g[f"{tag}_b2a"])
            assert np.array_equal(canon(B.filterind(tgt, tar, bcd)), g[f"{tag}_acd"])
            # filterind on a plan that lost its cached int32 copy (fresh tensor)
            assert np.array_equal(canon(B.filterind(tgt, tar, bcd.clone())), g[f"{tag}_acd"])
    tar, bcd = B.spspmm_ind(T(g["t32_i1"]), 2, T(g["t32_i2"]), 0)
    assert np.array_equal(canon(B.filterind(T(g["t32_i1"]), tar, bcd)), g["t32_acd"])


def test_fused_filtered_plan_equals_two_step(B, golden):
    from pygho_b200 import plans as P
    g = golden("spspmm")
    ei, tid = T(g["edge_index"]), T(g["tupleid"])
    for tag, (i1, d1, i2, d2) in {"XA": (tid, 1, ei, 0), "AX": (ei, 1, tid, 0),
                                  "XX": (tid, 1, tid, 0)}.items():
        acd, plan = P.filtered_plan(tid, i1, d1, i2, d2)
        assert np.array_equal(canon(acd), g[f"{tag}_acd"]), tag
        assert plan.T == g[f"{tag}_acd"].shape[1]


def test_empty_inputs(B):
    e2 = torch.zeros((2, 0), dtype=torch.int64, device=DEV)
    ind = torch.tensor([[0, 1, 2], [1, 2, 0]], device=DEV)
    tar, bcd = B.spspmm_ind(ind, 1, e2, 0)
    assert tar.shape == (2, 0) and bcd.shape == (3, 0)
    tar, bcd = B.spspmm_ind(e2, 1, ind, 0)
    assert tar.shape == (2, 0) and bcd.shape == (3, 0)
    X = B.SparseTensor(e2, torch.zeros((0, 4), device=DEV), (3, 3, 4), True)
    assert X.sum([1]).shape == (3, 4) and float(X.sum([1]).abs().sum()) == 0.0
    out = B.torch_scatter_reduce(0, torch.zeros((0, 4), device=DEV),
                                 torch.zeros((0,), dtype=torch.int64, device=DEV), 5, "max")
    assert out.shape == (5, 4) and float(out.abs().sum()) == 0.0


def test_random_2dmm_vs_dense(B):
    # reference tests/test_backend_sparse.py:101-143
    gen = torch.Generator().manual_seed(3)
    n, m, l = 300, 200, 400
    A = torch.rand((n, m), generator=gen)
    A[torch.rand((n, m), generator=gen) > 0.1] = 0
    Bm = torch.rand((m, l), generator=gen)
    Bm[torch.rand((m, l), generator=gen) > 0.1] = 0
    As, Bs = A.to_sparse_coo(), Bm.to_sparse_coo()
    C = (A.double() @ Bm.double())
    ind1, ind2 = As.indices().to(DEV), Bs.indices().to(DEV)
    SA = B.SparseTensor(ind1, As.values().to(DEV).unsqueeze(-1), (n, m, 1), True)
    SB = B.SparseTensor(ind2, Bs.values().to(DEV).unsqueeze(-1), (m, l, 1), True)
    tar, bcd = B.spspmm_ind(ind1, 1, ind2, 0)
    with pytest.warns(UserWarning):
        out = B.spspmm(SA, 1, SB, 0, "sum")
    assert torch.equal(out.indices.cpu(), C.to_sparse_coo().coalesce().indices())
    close(out.values[:, 0], C[tuple(out.indices.cpu())].float(), 5e-5)
    tgt = torch.stack((torch.randint(0, n, (5000,), generator=gen),
                       torch.randint(0, l, (5000,), generator=gen))).to(DEV)
    tgt = B.decodehash(torch.unique(B.indicehash(tgt)), 2)
    acd = B.filterind(tgt, tar, bcd)
    out = B.spspmm(SA, 1, SB, 0, "sum", acd=acd, tar_ind=tgt)
    close(out.values[:, 0], C[tuple(tgt.cpu())].float(), 5e-5)


# ---------------------------------------------------------------------------- value ops
AGGRS = ("sum", "mean", "max", "min")


def _sp(B, ind, val, N_):
    return B.SparseTensor(ind, val, (N_, N_) + tuple(val.shape[1:]) if val is not None else (N_, N_), True)


def test_value_ops_golden(B, golden):
    g = golden("spspmm")
    Nn = int(g["N"])
    ei, tid = T(g["edge_index"]), T(g["tupleid"])
    A, X = _sp(B, ei, T(g["Av"]), Nn), _sp(B, tid, T(g["Xv"]), Nn)
    x = T(g["x"])
    ops = {"XA": (X, 1, A, 0), "AX": (A, 1, X, 0), "XX": (X, 1, X, 0)}
    for tag, (P_, d1, Q_, d2) in ops.items():
        acd = T(g[f"{tag}_acd"])
        for aggr in AGGRS:
            out = B.spspmm(P_, d1, Q_, d2, aggr, acd=acd, tar_ind=tid)
            assert out.indices is tid and out.shape == (Nn, Nn, 8)
            close(out.values, g[f"{tag}_{aggr}"])
    Aone = _sp(B, ei, None, Nn)
    close(B.spspmm(X, 1, Aone, 0, "sum", acd=T(g["XA_acd"]), tar_ind=tid).values, g["XA_sum_noB"])
    close(B.spspmm(Aone, 1, X, 0, "max", acd=T(g["AX_acd"]), tar_ind=tid).values,
          O.spspmm(None, g["Xv"], g["AX_acd"], tid.shape[1], "max"))
    with pytest.warns(UserWarning):
        full = B.spspmm(X, 1, A, 0, "sum")
    assert np.array_equal(N(full.indices), g["XA_full_tar"])
    close(full.values, g["XA_full_sum"])
    H = B.spsphadamard(X, _sp(B, T(g["had_ind2"]), T(g["had_val2"]), Nn))
    assert np.array_equal(N(H.indices), g["had_ind"])
    close(H.values, g["had_val"])
    for aggr in ("sum", "mean", "max"):
        close(B.spmm(A, 1, x, aggr), g[f"spmm1_{aggr}"])
        close(B.spmm(A, 0, x, aggr), g[f"spmm0_{aggr}"])
        close(getattr(X, aggr)([1]), g[f"pool1_{aggr}"])
        close(getattr(X, aggr)([0]), g[f"pool0_{aggr}"])
    A1 = B.SparseTensor(ei, T(g["Av"])[:, :1].contiguous(), (Nn, Nn, 1), True)
    close(B.spmm(A1, 1, x), g["spmm1_scalar"])
    close(B.spmm(Aone, 1, x), g["spmm1_noval"])
    close(X.unpooling_fromdense1dim(0, x).values, g["unpool0"])
    close(X.unpooling_fromdense1dim(1, x).values, g["unpool1"])
    close(B.torch_scatter_reduce(0, x, T(g["batch"]), int(g["batch"].max()) + 1, "sum"),
          g["readout_sum"])


def test_3d_tuples_golden(B, golden):
    g = golden("tuples3d")
    Nn = int(g["N"])
    ei, tid = T(g["edge_index"]), T(g["tupleid"])
    A = B.SparseTensor(ei, T(g["Av"]), (Nn, Nn, 4), True)
    X = B.SparseTensor(tid, T(g["Xv"]), (Nn, Nn, Nn, 4), True)
    acd = B.filterind(tid, *B.spspmm_ind(tid, 2, ei, 0))
    assert np.array_equal(canon(acd), g["acd"])
    for aggr in ("sum", "max"):
        close(B.spspmm(X, 2, A, 0, aggr, acd=acd, tar_ind=tid).values, g[f"mp_{aggr}"])
    for aggr in ("sum", "mean", "max"):
        Pp = getattr(X, aggr)([2], return_sparse=True)
        assert np.array_equal(N(Pp.indices), g[f"pool2s_ind_{aggr}"])
        close(Pp.values, g[f"pool2s_val_{aggr}"])
        close(getattr(X, aggr)([1, 2]), g[f"pool12_{aggr}"])
        close(getattr(X, aggr)([2]), g[f"pool2_{aggr}"])
    Pp = X.sum([2], return_sparse=True)
    close(Pp.unpooling([2], X).values, g["unpool_sp"])


def _rand_problem(seed, n_out=97, n_a=61, n_b=43, T_=700, d=12, ties=False):
    gen = torch.Generator().manual_seed(seed)
    acd = torch.stack((torch.randint(0, n_out, (T_,), generator=gen),
                       torch.randint(0, n_a, (T_,), generator=gen),
                       torch.randint(0, n_b, (T_,), generator=gen)))
    if ties:  # small integer values -> many equal products
        a = torch.randint(-2, 3, (n_a, d), generator=gen).float()
        b = torch.randint(-2, 3, (n_b, d), generator=gen).float()
    else:
        a, b = torch.randn((n_a, d), generator=gen), torch.randn((n_b, d), generator=gen)
    return acd, a, b


@pytest.mark.parametrize("aggr", AGGRS)
@pytest.mark.parametrize("d", [1, 3, 8, 12, 128, 200, 256, 384])
@pytest.mark.parametrize("ties", [False, True])
def test_seg_gmr_forward_backward_vs_torch(aggr, d, ties):
    """Unsorted random plan, every aggregation and width: values and both operand
    gradients against torch autograd on the CPU (the reference's own ATen ops)."""
    from pygho_b200 import plans as P
    from pygho_b200.ops import seg_gmr
    acd, a, b = _rand_problem(d * 7 + len(aggr), d=d, ties=ties)
    n_out = 97
    a_ref, b_ref = a.clone().requires_grad_(True), b.clone().requires_grad_(True)
    ref = TO.spspmm(a_ref, b_ref, acd, n_out, aggr)
    w = torch.randn(ref.shape, generator=torch.Generator().manual_seed(1))
    (ref * w).sum().backward()
    a_g, b_g = a.to(DEV).requires_grad_(True), b.to(DEV).requires_grad_(True)
    plan = P.plan_from_acd(acd.to(DEV), n_out, a.shape[0], b.shape[0])
    out = seg_gmr(a_g, b_g, plan, aggr)
    (out * w.to(DEV)).sum().backward()
    close(out, ref)
    close(a_g.grad, a_ref.grad, 2e-5)
    close(b_g.grad, b_ref.grad, 2e-5)
    # single-operand forms
    a_ref2 = a.clone().requires_grad_(True)
    ref2 = TO.spspmm(a_ref2, None, acd, n_out, aggr)
    (ref2 * w).sum().backward()
    a_g2 = a.to(DEV).requires_grad_(True)
    out2 = seg_gmr(a_g2, None, plan, aggr)
    (out2 * w.to(DEV)).sum().backward()
    close(out2, ref2)
    close(a_g2.grad, a_ref2.grad, 2e-5)
    b_ref3 = b.clone().requires_grad_(True)
    ref3 = TO.spspmm(None, b_ref3, acd, n_out, aggr)
    (ref3 * w).sum().backward()
    b_g3 = b.to(DEV).requires_grad_(True)
    out3 = seg_gmr(None, b_g3, plan, aggr)
    (out3 * w.to(DEV)).sum().backward()
    close(out3, ref3)
    close(b_g3.grad, b_ref3.grad, 2e-5)


def test_deterministic(B, golden):
    g = golden("spspmm")
    Nn = int(g["N"])
    ei, tid = T(g["edge_index"]), T(g["tupleid"])
    A, X = _sp(B, ei, T(g["Av"]), Nn), _sp(B, tid, T(g["Xv"]), Nn)
    acd = T(g["XX_acd"])
    outs = [B.spspmm(X, 1, X, 0, "sum", acd=acd.clone(), tar_ind=tid).values for _ in range(3)]
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])


@pytest.mark.parametrize("aggr", ("sum", "mean", "max"))
def test_spmm_pool_unpool_gradients(B, golden, aggr):
    g = golden("spspmm")
    Nn = int(g["N"])
    ei_c, tid_c = torch.from_numpy(g["edge_index"]), torch.from_numpy(g["tupleid"])
    Av, Xv, x = (torch.from_numpy(g[k]) for k in ("Av", "Xv", "x"))
    w = torch.randn((Nn, 8), generator=torch.Generator().manual_seed(2))
    for dim1 in (0, 1):
        av, xr = Av.clone().requires_grad_(True), x.clone().requires_grad_(True)
        (TO.spmm(ei_c, av, (Nn, Nn), dim1, xr, aggr) * w).sum().backward()
        avg, xg = Av.to(DEV).requires_grad_(True), x.to(DEV).requires_grad_(True)
        A = B.SparseTensor(ei_c.to(DEV), avg, (Nn, Nn, 8), True)
        (B.spmm(A, dim1, xg, aggr) * w.to(DEV)).sum().backward()
        close(avg.grad, av.grad, 2e-5)
        close(xg.grad, xr.grad, 2e-5)
    for keep in (0, 1):
        xv = Xv.clone().requires_grad_(True)
        (TO.sp_pool(tid_c, xv, (Nn, Nn), keep, aggr) * w).sum().backward()
        xvg = Xv.to(DEV).requires_grad_(True)
        X = B.SparseTensor(tid_c.to(DEV), xvg, (Nn, Nn, 8), True)
        (getattr(X, aggr)([1 - keep]) * w.to(DEV)).sum().backward()
        close(xvg.grad, xv.grad, 2e-5)
        xr = x.clone().requires_grad_(True)
        w2 = torch.randn((tid_c.shape[1], 8), generator=torch.Generator().manual_seed(3))
        (TO.sp_unpool(tid_c, keep, xr) * w2).sum().backward()
        xg = x.to(DEV).requires_grad_(True)
        (X.unpooling_fromdense1dim(keep, xg).values * w2.to(DEV)).sum().backward()
        close(xg.grad, xr.grad, 2e-5)


@pytest.mark.parametrize("aggr", ("sum", "mean", "max"))
@pytest.mark.parametrize("key", ("XA", "AX"))
def test_full_size_spspmm_vs_torch_oracle(B, aggr, key):
    """BASELINE-size batch (B=1024 graphs, d=128): the kernels bench.py times (lean streaming
    kernel for sum/mean, both operand-gradient groupings) compared DIRECTLY with the torch-CPU
    oracle -- values and both operand gradients, no size reduction."""
    from pygho_b200.hodata.synthetic import make_batch
    hb = make_batch(1024, seed=0)
    ei_c, tid_c = torch.from_numpy(hb.edge_index), torch.from_numpy(hb.tupleid)
    Nn, d = hb.num_nodes, 128
    gen = torch.Generator().manual_seed(5)
    Xv = torch.randn((tid_c.shape[1], d), generator=gen)
    Av = torch.randn((ei_c.shape[1], d), generator=gen)
    w = torch.randn((tid_c.shape[1], d), generator=gen)
    ei, tid = ei_c.to(DEV), tid_c.to(DEV)
    if key == "XA":
        acd = B.filterind(tid, *B.spspmm_ind(tid, 1, ei, 0))
    else:
        acd = B.filterind(tid, *B.spspmm_ind(ei, 1, tid, 0))
    xr, ar = Xv.clone().requires_grad_(True), Av.clone().requires_grad_(True)
    ops_ref = (xr, ar) if key == "XA" else (ar, xr)
    ref = TO.spspmm(ops_ref[0], ops_ref[1], acd.cpu(), tid_c.shape[1], aggr)
    (ref * w).sum().backward()
    xg, ag = Xv.to(DEV).requires_grad_(True), Av.to(DEV).requires_grad_(True)
    X, A = _sp(B, tid, xg, Nn), _sp(B, ei, ag, Nn)
    P, Q = (X, A) if key == "XA" else (A, X)
    out = B.spspmm(P, 1, Q, 0, aggr, acd=acd, tar_ind=tid).values
    (out * w.to(DEV)).sum().backward()
    close(out, ref, 1e-5)
    close(xg.grad, xr.grad, 2e-5)
    close(ag.grad, ar.grad, 2e-5)


def test_full_size_properties(B):
    """BASELINE-size batch (B=1024 graphs): properties that do not need the oracle --
    linearity of sum, mean*count == sum, max >= mean, plan totals, sortedness."""
    from pygho_b200.hodata.synthetic import make_batch
    hb = make_batch(1024, seed=0)
    ei, tid = T(hb.edge_index), T(hb.tupleid)
    Nn, d = hb.num_nodes, 128
    gen = torch.Generator(device=DEV).manual_seed(0)
    Xv = torch.randn((tid.shape[1], d), device=DEV, generator=gen)
    Av = torch.randn((ei.shape[1], d), device=DEV, generator=gen)
    tar, bcd = B.spspmm_ind(tid, 1, ei, 0)
    acd = B.filterind(tid, tar, bcd)
    assert bool((acd[0][1:] >= acd[0][:-1]).all())
    assert bool((tid[1][acd[1]] == ei[0][acd[2]]).all())          # contracted index matches
    assert bool((tid[0][acd[1]] == tid[0][acd[0]]).all()) and bool((ei[1][acd[2]] == tid[1][acd[0]]).all())
    X, A = _sp(B, tid, Xv, Nn), _sp(B, ei, Av, Nn)
    s1 = B.spspmm(X, 1, A, 0, "sum", acd=acd, tar_ind=tid).values
    X2 = _sp(B, tid, 2.0 * Xv, Nn)
    s2 = B.spspmm(X2, 1, A, 0, "sum", acd=acd, tar_ind=tid).values
    assert torch.equal(s2, 2.0 * s1)                               # exact: scaling by 2
    cnt = torch.bincount(acd[0], minlength=tid.shape[1]).clamp_min(1).unsqueeze(1)
    mean = B.spspmm(X, 1, A, 0, "mean", acd=acd, tar_ind=tid).values
    close(mean * cnt, s1, 1e-5)
    mx = B.spspmm(X, 1, A, 0, "max", acd=acd, tar_ind=tid).values
    mn = B.spspmm(X, 1, A, 0, "min", acd=acd, tar_ind=tid).values
    assert bool((mx >= mn).all()) and bool((mx + 1e-4 >= mean).all())
    # checksum of checksums: total of the sum-aggregated output == total of all messages
    tot = (Xv[acd[1]].double() * Av[acd[2]].double()).sum()
    assert abs(float(s1.double().sum() - tot)) <= 1e-6 * float(
        (Xv[acd[1]].double() * Av[acd[2]].double()).abs().sum())
    pooled = X.sum([1])
    close(pooled.double().sum(0), Xv.double().sum(0), 1e-5)


# -------------------------------------------------------------------------------- masked
@pytest.mark.parametrize("algo,tol", [(0, 1e-5), (1, 1e-2), (2, 1e-2)])
def test_masked_golden(B, golden, monkeypatch, algo, tol):
    monkeypatch.setenv("PYGHO_B200_MAMAMM_ALGO", str(algo))
    g = golden("masked")
    A, Bm, mask = T(g["A"]), T(g["B"]), T(g["mask"])
    MA, MB = B.MaskedTensor(A, mask), B.MaskedTensor(Bm, mask)
    for d1 in (1, 2):
        for d2 in (1, 2):
            close(B.mamamm(MA, d1, MB, d2, mask).data, g[f"mm_{d1}{d2}"], tol)
    for aggr in ("sum", "mean", "max"):
        for dims in ((1,), (2,), (1, 2)):
            tag = "".join(map(str, dims))
            r = getattr(MA, aggr)(list(dims))
            assert np.array_equal(N(r.mask), g[f"pool{tag}_mask"])
            sel = g[f"pool{tag}_mask"][..., None]
            close(np.where(sel, N(r.data), 0), np.where(sel, g[f"pool{tag}_{aggr}"], 0))
    close(MA.min([2]).data, g["pool2_min"])
    close(B.MaskedTensor(A, mask, padvalue=float("inf")).fill_masked(1024), g["fill1024"])
    assert np.array_equal(N(B.filterinf(T(g["filterinf_in"]))), g["filterinf_out"])


def test_masked_constructor_fills_pads(B):
    data = torch.ones((2, 3, 3, 4), device=DEV)
    mask = torch.zeros((2, 3, 3), dtype=torch.bool, device=DEV)
    mask[0, :2, :2] = True
    mt = B.MaskedTensor(data, mask)
    assert float(mt.data.sum()) == 16.0                       # intended semantics (Q1)
    assert float(mt.fill_masked(5.0).sum()) == 16.0 + 5.0 * (72 - 16)


@pytest.mark.parametrize("algo,tol", [(0, 2e-5), (1, 1e-2), (2, 1e-2), (4, 2e-5)])
@pytest.mark.parametrize("d1,d2", [(2, 1), (1, 1), (1, 2), (2, 2)])
def test_mamamm_forward_backward(B, monkeypatch, d1, d2, algo, tol):
    monkeypatch.setenv("PYGHO_B200_MAMAMM_ALGO", str(algo))
    gen = torch.Generator().manual_seed(d1 * 3 + d2)
    b, n, d = 5, 11, 40
    sizes = torch.randint(3, n + 1, (b,), generator=gen)
    ar = torch.arange(n)
    mask = (ar[None, :, None] < sizes[:, None, None]) & (ar[None, None, :] < sizes[:, None, None])
    a = torch.randn((b, n, n, d), generator=gen) * mask.unsqueeze(-1)
    bb = torch.randn((b, n, n, d), generator=gen) * mask.unsqueeze(-1)
    w = torch.randn((b, n, n, d), generator=gen)
    ar_, br_ = a.clone().requires_grad_(True), bb.clone().requires_grad_(True)
    ref = TO.mamamm(ar_ * mask.unsqueeze(-1), d1, br_ * mask.unsqueeze(-1), d2, mask)
    (ref * w).sum().backward()
    ag, bg = a.to(DEV).requires_grad_(True), bb.to(DEV).requires_grad_(True)
    mk = mask.to(DEV)
    out = B.mamamm(B.MaskedTensor(ag, mk), d1, B.MaskedTensor(bg, mk), d2, mk)
    (out.data * w.to(DEV)).sum().backward()
    close(out.data, ref, tol)
    close(ag.grad, ar_.grad, tol)
    close(bg.grad, br_.grad, tol)


@pytest.mark.parametrize("aggr", AGGRS)
@pytest.mark.parametrize("dims", [(1,), (2,), (1, 2)])
@pytest.mark.parametrize("b,n,d", [(4, 9, 24), (3, 37, 128), (2, 10, 256)])
def test_masked_pool_forward_backward(B, aggr, dims, b, n, d):
    """d = 24: thread-per-4-channels kernels; d % 128 == 0: warp-cooperative kernels (mask bits by
    ballot), n = 37 walks more than one 32-position chunk of the reduced extent."""
    gen = torch.Generator().manual_seed(5)
    mask = torch.rand((b, n, n), generator=gen) < 0.6
    mask[0] = False                                          # a fully masked graph
    data = torch.randn((b, n, n, d), generator=gen)
    ref_in = data.clone().requires_grad_(True)
    ref = TO.ma_pool(ref_in * mask.unsqueeze(-1), mask, dims, aggr)
    w = torch.randn(ref.shape, generator=gen)
    (ref * w).sum().backward()
    dg = data.to(DEV).requires_grad_(True)
    r = getattr(B.MaskedTensor(dg, mask.to(DEV)), aggr)(list(dims))
    (r.data * w.to(DEV)).sum().backward()
    close(r.data, ref, 2e-5)
    assert torch.equal(r.mask.cpu(), mask.any(dim=dims))
    close(dg.grad, ref_in.grad, 2e-5)


@pytest.mark.parametrize("n,d", [(40, 128), (37, 64), (9, 8), (23, 16), (48, 8)])
@pytest.mark.parametrize("ta,tb", [(False, False), (True, False), (False, True), (True, True)])
def test_mamamm_tcgen05_matches_fp32_kernel(n, d, ta, tb):
    """tcgen05 TF32 paths (algo 1, 2) against the exact-fp32 kernel (algo 0): 1e-2 relative
    (BASELINE.json: bf16/TF32 mamamm within a stated 1e-2), pads exactly zero."""
    import pygho_b200.ops  # noqa: F401
    gen = torch.Generator().manual_seed(n * 131 + d)
    b = 5
    sizes = torch.randint(max(2, n // 2), n + 1, (b,), generator=gen)
    sizes[0] = n
    ar = torch.arange(n)
    mask = ((ar[None, :, None] < sizes[:, None, None]) & (ar[None, None, :] < sizes[:, None, None])).to(DEV)
    A = (torch.randn((b, n, n, d), generator=gen).to(DEV) * mask.unsqueeze(-1)).contiguous()
    Bm = (torch.randn((b, n, n, d), generator=gen).to(DEV) * mask.unsqueeze(-1)).contiguous()
    ref = torch.ops.pygho_b200.mamamm(A, ta, Bm, tb, mask, None, 0)
    scale = float(ref.abs().max())
    ext = torch.stack((sizes, sizes, sizes), 1).to(torch.int32).to(DEV)
    for e in (None, ext):
        got = torch.ops.pygho_b200.mamamm(A, ta, Bm, tb, mask, e, 1)
        assert float((got - ref).abs().max()) <= 1e-2 * scale
        assert float(got[~mask].abs().max()) == 0.0
        # the pipelined kernel issues the same MMAs on the same tiles: identical bits
        # (n = 48 needs two stages of 144 KB -> it falls back to the algo-1 kernel)
        pipe = torch.ops.pygho_b200.mamamm(A, ta, Bm, tb, mask, e, 2)
        assert torch.equal(pipe, got)
        # the fp32 kernel with extents is bit-identical to the one without
        assert torch.equal(torch.ops.pygho_b200.mamamm(A, ta, Bm, tb, mask, e, 0), ref)
    from pygho_b200.ops import mask_extents
    assert torch.equal(mask_extents(mask).cpu(), torch.stack((sizes, sizes), 1).to(torch.int32))
    torch.cuda.synchronize()


@pytest.mark.parametrize("shape", [(6, 40, 40, 40, 128), (5, 37, 23, 29, 64), (7, 9, 9, 9, 16),
                                   (3, 100, 70, 100, 32), (2, 20, 300, 12, 16), (4, 16, 16, 16, 40)])
@pytest.mark.parametrize("ta,tb", [(False, False), (True, False), (False, True), (True, True)])
def test_mamamm_smem_ring_is_bit_identical_to_fp32_kernel(shape, ta, tb):
    """algo 4 (TMA-fed shared-memory ring, exact fp32, csrc/mamamm_smem.cu) against algo 0: the
    same j-ascending fmaf chains -> identical bits; rectangular extents, graphs of every size
    incl. empty ones, a mask with holes, several row passes (n = 100), dense = 40 (not a
    multiple of 16: runs on algo 0 inside the library), pads exactly zero."""
    import pygho_b200.ops  # noqa: F401
    b, n_i, n_j, n_k, d = shape
    gen = torch.Generator().manual_seed(n_i * 7 + n_j * 3 + d + 2 * ta + tb)
    si = torch.randint(0, n_i + 1, (b,), generator=gen)
    sj = torch.randint(0, n_j + 1, (b,), generator=gen)
    sk = torch.randint(0, n_k + 1, (b,), generator=gen)
    si[0], sj[0], sk[0] = n_i, n_j, n_k
    if b > 2:
        si[1] = 0
        sj[2] = 0
    def band(s1, n1, s2, n2):
        return (torch.arange(n1)[None, :, None] < s1[:, None, None]) & (torch.arange(n2)[None, None, :] < s2[:, None, None])
    mA, mB, mO = band(si, n_i, sj, n_j), band(sj, n_j, sk, n_k), band(si, n_i, sk, n_k)
    holes = (mO & (torch.rand((b, n_i, n_k), generator=gen) < 0.8)).to(DEV)
    A = torch.randn((b, n_i, n_j, d), generator=gen) * mA.unsqueeze(-1)
    Bm = torch.randn((b, n_j, n_k, d), generator=gen) * mB.unsqueeze(-1)
    A = (A.transpose(1, 2) if ta else A).contiguous().to(DEV)
    Bm = (Bm.transpose(1, 2) if tb else Bm).contiguous().to(DEV)
    ext = torch.stack((si, sj, sk), 1).to(torch.int32).to(DEV)
    ref = torch.ops.pygho_b200.mamamm(A, ta, Bm, tb, holes, None, 0)
    for e in (None, ext):
        torch.full((b, n_i, n_k, d), float("nan"), device=DEV)     # poison the next allocation
        got = torch.ops.pygho_b200.mamamm(A, ta, Bm, tb, holes, e, 4)
        assert torch.equal(got, ref), float((got - ref).abs().max())
        assert float(got[~holes].abs().max()) == 0.0
    # the queue order (largest graph first, or any permutation) never changes the result
    lpt = torch.argsort((si * sj * sk), descending=True, stable=True).to(torch.int32).to(DEV)
    for order in (lpt, torch.randperm(b, generator=gen).to(torch.int32).to(DEV)):
        got = torch.ops.pygho_b200.mamamm(A, ta, Bm, tb, holes, ext, 4, order)
        assert torch.equal(got, ref), float((got - ref).abs().max())
    # back-to-back launches re-arm their work queues (64 rotating, self-resetting)
    for _ in range(70):
        got = torch.ops.pygho_b200.mamamm(A, ta, Bm, tb, holes, ext, 4)
    assert torch.equal(got, ref)
    torch.cuda.synchronize()


def test_mamamm_pipeline_many_items():
    """The persistent pipeline with more work items than CTAs (b * dense / 8 = 800 > 148),
    graphs of every size incl. empty ones, a mask with holes: bit-identical to the
    one-CTA-per-item tcgen05 kernel, pads exactly zero, 1e-2 against exact fp32."""
    import pygho_b200.ops  # noqa: F401
    gen = torch.Generator().manual_seed(7)
    b, n, d = 50, 40, 128
    sizes = torch.randint(0, n + 1, (b,), generator=gen)
    sizes[0], sizes[1], sizes[2] = n, 0, 1
    ar = torch.arange(n)
    mask = (ar[None, :, None] < sizes[:, None, None]) & (ar[None, None, :] < sizes[:, None, None])
    holes = mask & (torch.rand((b, n, n), generator=gen) < 0.8)
    mask, holes = mask.to(DEV), holes.to(DEV)
    A = (torch.randn((b, n, n, d), generator=gen).to(DEV) * mask.unsqueeze(-1)).contiguous()
    Bm = (torch.randn((b, n, n, d), generator=gen).to(DEV) * mask.unsqueeze(-1)).contiguous()
    ext = torch.stack((sizes, sizes, sizes), 1).to(torch.int32).to(DEV)
    ref = torch.ops.pygho_b200.mamamm(A, False, Bm, False, holes, None, 0)
    for e in (None, ext):
        one = torch.ops.pygho_b200.mamamm(A, False, Bm, False, holes, e, 1)
        # poison the output allocation so unwritten positions would be noticed
        torch.full((b, n, n, d), float("nan"), device=DEV)
        pipe = torch.ops.pygho_b200.mamamm(A, False, Bm, False, holes, e, 2)
        assert torch.equal(pipe, one)
        assert float(pipe[~holes].abs().max()) == 0.0
        assert float((pipe - ref).abs().max()) <= 1e-2 * float(ref.abs().max())
    torch.cuda.synchronize()


def test_seg_gmr_strided_operands_and_out_slice():
    """Operands / output that are column slices of wider buffers (row stride > dense):
    same bits as the contiguous call, no copies needed."""
    from pygho_b200 import plans as P
    import pygho_b200.ops  # noqa: F401
    ops = torch.ops.pygho_b200
    for d in (128, 8):
        acd, a, b = _rand_problem(5, d=d)
        a, b = a.to(DEV), b.to(DEV)
        plan = P.plan_from_acd(acd.to(DEV), 97, a.shape[0], b.shape[0])
        g = plan.group("a")
        ref = ops.seg_gmr(a, g.first, None, b, g.second, g.rowptr, 97, 0)
        wide_a = torch.randn(a.shape[0], 3 * d, device=DEV)
        wide_b = torch.randn(b.shape[0], 2 * d, device=DEV)
        wide_a[:, d:2 * d] = a
        wide_b[:, d:] = b
        got = ops.seg_gmr(wide_a[:, d:2 * d], g.first, None, wide_b[:, d:], g.second, g.rowptr, 97, 0)
        assert torch.equal(got, ref)
        buf = torch.full((97, 3 * d), 7.0, device=DEV)
        ops.seg_gmr_out(a, g.first, None, b, g.second, g.rowptr, 97, 0, buf[:, 2 * d:], False)
        assert torch.equal(buf[:, 2 * d:], ref) and float(buf[:, :2 * d].min()) == 7.0
        # accumulate: out += result
        ops.seg_gmr_out(a, g.first, None, b, g.second, g.rowptr, 97, 0, buf[:, 2 * d:], True)
        assert torch.equal(buf[:, 2 * d:], ref + ref)


def test_spspmpnn_with_message_function(B, golden):
    """spspmpnn (reference Spspmm.py:334-380): a GAT-like message function that mixes the
    three gathered operands; values and gradients against the torch restatement."""
    g = golden("spspmm")
    Nn = int(g["N"])
    ei_c, tid_c, acd_c = (torch.from_numpy(g[k]) for k in ("edge_index", "tupleid", "XA_acd"))
    Av, Xv = torch.from_numpy(g["Av"]), torch.from_numpy(g["Xv"])

    def msg(a, b, c, idx):
        return torch.tanh(a + c) * b

    xr, ar = Xv.clone().requires_grad_(True), Av.clone().requires_grad_(True)
    m = msg(xr[acd_c[1]], ar[acd_c[2]], xr[acd_c[0]], acd_c[0])
    ref = TO.scatter_reduce(m, acd_c[0], tid_c.shape[1], "sum")
    w = torch.randn(ref.shape, generator=torch.Generator().manual_seed(0))
    (ref * w).sum().backward()
    xg, ag = Xv.to(DEV).requires_grad_(True), Av.to(DEV).requires_grad_(True)
    X = B.SparseTensor(tid_c.to(DEV), xg, (Nn, Nn, 8), True)
    A = B.SparseTensor(ei_c.to(DEV), ag, (Nn, Nn, 8), True)
    out = B.spspmpnn(X, 1, A, 0, X, acd_c.to(DEV), msg, "sum")
    (out.values * w.to(DEV)).sum().backward()
    close(out.values, ref, 2e-5)
    close(xg.grad, xr.grad, 5e-5)
    close(ag.grad, ar.grad, 5e-5)
    # through the operator wrapper (honn/SpOperator.py message_func path)
    from pygho_b200.honn.SpOperator import OpMessagePassingOnSubg2D
    op = OpMessagePassingOnSubg2D("sum", message_func=msg)
    out2 = op(A, X, {op.precomputekey + "___acd": acd_c.to(DEV)}, X)
    close(out2.values, ref, 2e-5)


def test_diag_add_and_sparse_unpool(B, golden):
    g = golden("spspmm")
    Nn = int(g["N"])
    tid, Xv = T(g["tupleid"]), T(g["Xv"])
    X = B.SparseTensor(tid, Xv, (Nn, Nn, 8), True)
    close(X.diag([0, 1]), O.sp_diag_dense(g["tupleid"], g["Xv"], (Nn, Nn), [0, 1]))
    from pygho_b200.honn.TensorOp import OpDiag2D
    close(OpDiag2D("S")(X), O.sp_diag_dense(g["tupleid"], g["Xv"], (Nn, Nn), [0, 1]))
    # add with a different sparsity pattern -> concatenate + coalesce (SpTensor.py:507-514)
    sub = tid[:, ::3].contiguous()
    Y = B.SparseTensor(sub.flip(1).contiguous(), Xv[::3].flip(0).contiguous(), (Nn, Nn, 8), False)
    assert torch.equal(Y.indices, sub)                       # coalesce sorted it back
    Z = X.add(Y, False)
    want_i, want_v = O.coalesce(np.concatenate([g["tupleid"], g["tupleid"][:, ::3]], 1),
                                np.concatenate([g["Xv"], g["Xv"][::3]], 0), "sum")
    assert np.array_equal(N(Z.indices), want_i)
    close(Z.values, want_v)
    # same-pattern ops
    close(X.add(X, True).values, 2 * g["Xv"])
    assert X.catvalue([X, X], True).shape == (Nn, Nn, 24)
    d = X.diagonalapply(lambda v, flag: v * flag.unsqueeze(-1))
    eq = (g["tupleid"][0] == g["tupleid"][1])[:, None]
    close(d.values, g["Xv"] * eq)


def test_dense_node_message_passing(B):
    """DD OpNodeMessagePassing (broken in the reference, Q3): A (b,n,n,d) x (b,n,d)."""
    from pygho_b200.honn.TensorOp import OpNodeMessagePassing
    gen = torch.Generator().manual_seed(1)
    b, n, d = 3, 6, 8
    sizes = torch.tensor([6, 4, 5])
    ar = torch.arange(n)
    m1 = ar[None, :] < sizes[:, None]
    m2 = m1[:, :, None] & m1[:, None, :]
    A = torch.randn(b, n, n, d, generator=gen) * m2.unsqueeze(-1)
    x = torch.randn(b, n, d, generator=gen) * m1.unsqueeze(-1)
    out = OpNodeMessagePassing("DD")(B.MaskedTensor(A.to(DEV), m2.to(DEV)), B.MaskedTensor(x.to(DEV), m1.to(DEV)))
    close(out.data, torch.einsum("bijd,bjd->bid", A, x) * m1.unsqueeze(-1), 1e-2)


def test_ragged_and_degenerate_plans():
    """Rows without entries, one giant row, a single graph, duplicated triples: the
    streaming and the row-wise kernels agree with the oracle."""
    from pygho_b200 import plans as P
    from pygho_b200.ops import seg_gmr
    gen = torch.Generator().manual_seed(11)
    n_out, n_a, n_b = 300, 50, 40
    for d in (128, 20):
        a = torch.randn(n_a, d, generator=gen)
        b = torch.randn(n_b, d, generator=gen)
        rows = torch.cat([torch.full((700,), 7), torch.randint(100, 120, (200,), generator=gen),
                          torch.tensor([299, 299, 0])])            # rows 8..99, 120..298 empty
        acd = torch.stack([rows, torch.randint(0, n_a, rows.shape, generator=gen),
                           torch.randint(0, n_b, rows.shape, generator=gen)])
        acd = torch.cat([acd, acd[:, :50]], dim=1)                  # duplicated triples
        plan = P.plan_from_acd(acd.to(DEV), n_out, n_a, n_b)
        for aggr in AGGRS:
            got = seg_gmr(a.to(DEV), b.to(DEV), plan, aggr)
            close(got, O.spspmm(a.numpy(), b.numpy(), acd.numpy(), n_out, aggr), 2e-5)
            assert float(got[8:100].abs().max()) == 0.0             # empty rows are exactly 0


def test_single_graph_batch(B):
    from pygho_b200.hodata.device import sp_datadict
    from pygho_b200.hodata.synthetic import make_batch
    hb = make_batch(1, seed=3)
    dd = sp_datadict(hb, DEV, ["X___X___1___A___0"])
    acd = dd["X___X___1___A___0___acd"]
    want = O.filterind(hb.tupleid, *O.spspmm_ind(hb.tupleid, 1, hb.edge_index, 0))
    assert np.array_equal(canon(acd), want)


@pytest.mark.parametrize("mean", [False, True])
def test_seg_gmr_fused_epilogue_matches_separate_launches(mean):
    """out = add_src + reduction and the fused row copy (pgh_seg_gmr_fused_f32) against the plain
    launch + torch arithmetic; strided column slices like the SSWL concatenated buffer."""
    ops = torch.ops.pygho_b200
    gen = torch.Generator(device=DEV).manual_seed(3)
    n_rows, nA, nB, d = 777, 500, 300, 128
    lens = torch.randint(0, 5, (n_rows,), generator=gen, device=DEV)
    rowptr = torch.zeros(n_rows + 1, dtype=torch.int32, device=DEV)
    rowptr[1:] = lens.cumsum(0)
    Tn = int(rowptr[-1])
    c = torch.randint(0, nA, (Tn,), generator=gen, device=DEV, dtype=torch.int32)
    dd = torch.randint(0, nB, (Tn,), generator=gen, device=DEV, dtype=torch.int32)
    A = torch.randn(nA, d, generator=gen, device=DEV)
    Bv = torch.randn(nB, d, generator=gen, device=DEV)
    scale = torch.rand(nA, generator=gen, device=DEV) if mean else None
    aggr = 1 if mean else 0
    want = ops.seg_gmr(A, c, scale, Bv, dd, rowptr, n_rows, aggr)
    wide = torch.randn(n_rows, 3 * d, generator=gen, device=DEV)        # add_src / copy_src slices
    buf = torch.zeros(n_rows, 3 * d, device=DEV)
    ops.seg_gmr_fused(A, c, scale, Bv, dd, rowptr, n_rows, aggr, wide[:, :d], wide[:, d:2 * d],
                      buf[:, 2 * d:], buf[:, d:2 * d])
    close(buf[:, d:2 * d], want + wide[:, :d], 1e-6)
    assert torch.equal(buf[:, 2 * d:], wide[:, d:2 * d])
    assert float(buf[:, :d].abs().max()) == 0.0                          # untouched third
    out = torch.empty(n_rows, d, device=DEV)
    ops.seg_gmr_fused(A, c, scale, Bv, dd, rowptr, n_rows, aggr, None, None, None, out)
    assert torch.equal(out, want)
    with pytest.raises(Exception):
        ops.seg_gmr_fused(A[:, :64].contiguous(), c, None, None, None, rowptr, n_rows, 0, None,
                          None, None, torch.empty(n_rows, 64, device=DEV))


@pytest.mark.parametrize("T_,with_fillers", [(0, False), (1, False), (5000, False), (5000, True)])
def test_acd_regroup_one_call_equals_lazy_groupings(T_, with_fillers):
    """pgh_acd_regroup (all three CSR groupings of a (3, T) plan in one library call) against the
    grouping-by-grouping path: identical rowptr / index arrays, incl. filler entries whose key
    equals the row count (capacity-padded plans) and the empty plan."""
    from pygho_b200 import plans as P
    gen = torch.Generator().manual_seed(T_ + 7)
    n_out, n_a, n_b = 301, 97, 1000
    hi = (n_out + 1, n_a + 1, n_b + 1) if with_fillers else (n_out, n_a, n_b)
    acd = torch.stack([torch.randint(0, h, (T_,), generator=gen) for h in hi]).to(DEV)
    lazy = P.plan_from_acd(acd.clone(), n_out, n_a, n_b)
    fused = P.plan_from_acd(acd.clone(), n_out, n_a, n_b, build_all=True)
    assert set(fused._groups) == {"a", "c", "d"}
    for k in "acd":
        assert torch.equal(fused.idx[k], lazy.idx[k])
        gl, gf = lazy.group(k), fused.group(k)
        for x, y in zip(gl, gf):
            assert x.dtype == y.dtype == torch.int32 and torch.equal(x, y), k


def test_gather_product_matches_indexing(B):
    """SparseTensor.gather_product (ops.GatherProduct: the reference models' tuple initialisation
    X0[X.indices[0]] * X1[X.indices[1]] * val, example/zinc.py:270-276) against plain torch
    indexing: values and the gradients of all three factors."""
    from pygho_b200.hodata.device import sp_datadict
    from pygho_b200.hodata.synthetic import make_batch
    dd = sp_datadict(make_batch(24, seed=9), DEV, [])
    X = dd["X"]
    n, d = X.shape[0], 32
    gen = torch.Generator(device=DEV).manual_seed(4)
    P0 = torch.randn(n, d, generator=gen, device=DEV)
    Q0 = torch.randn(n, d, generator=gen, device=DEV)
    V0 = torch.randn(X.nnz, d, generator=gen, device=DEV)
    w = torch.randn(X.nnz, d, generator=gen, device=DEV)
    res = []
    for fused in (False, True):
        Pm, Qm, Vm = (t.clone().requires_grad_(True) for t in (P0, Q0, V0))
        Xv = B.SparseTensor(X.indices, Vm, X.shape[:2] + (d,), True)
        if fused:
            out = Xv.gather_product(Pm, Qm).values
        else:
            out = Pm[X.indices[0]] * Qm[X.indices[1]] * Vm
        (out * w).sum().backward()
        res.append((out.detach(), Pm.grad, Qm.grad, Vm.grad))
    for got, want in zip(res[1], res[0]):
        close(got, want, 2e-5)


def test_merge_groups_kernel_equals_torch_version():
    """pgh_merge_groups_i32 (CUDA groupings) against the fixed-shape torch version of
    plans.merge_groups (CPU groupings, tests/test_merge_groups_cpu.py), with filler entries."""
    from pygho_b200 import plans as P
    try:
        from test_merge_groups_cpu import _group
    except ImportError:
        from tests.test_merge_groups_cpu import _group
    rng = np.random.default_rng(5)
    for n_rows, T1, cap1, T2, cap2 in ((7, 20, 20, 13, 13), (50, 300, 340, 0, 5), (9, 0, 0, 4, 4),
                                       (3000, 20000, 20480, 17000, 17000)):
        g1, _ = _group(rng, n_rows, T1, cap1, 400, 110)
        g2, _ = _group(rng, n_rows, T2, cap2, 400, 110)
        want = P.merge_groups(g1, g2, n_rows, 3, 1, 2)
        got = P.merge_groups(P.Group(*(t.to(DEV) for t in g1)), P.Group(*(t.to(DEV) for t in g2)),
                             n_rows, 3, 1, 2)
        assert torch.equal(got.rowptr.cpu(), want.rowptr)
        real = int(want.rowptr[-1])
        assert torch.equal(got.first.cpu()[:real], want.first[:real])
        assert torch.equal(got.second.cpu()[:real], want.second[:real])


@pytest.mark.parametrize("residual", [False, True])
def test_sswl_merged_gradient_plan_matches_two_launches(residual):
    """ops.SswlAggregate.backward with the merged plan (plans.sswl_bwd_group: both products'
    entries per tuple, the gradient of the concatenation read as (3 n, d) rows, ONE launch)
    against the two accumulating launches: same gradients within fp32 reassociation."""
    from pygho_b200 import plans as P
    from pygho_b200.hodata.device import sp_datadict
    from pygho_b200.hodata.synthetic import make_batch
    from pygho_b200.ops import SswlAggregate
    k1, k2 = "X___X___1___A___0", "X___A___1___X___0"
    dd = sp_datadict(make_batch(48, seed=5), DEV, [k1, k2])
    nX, nA, d = dd["X"].nnz, dd["A"].nnz, 128
    acd1, acd2 = dd[k1 + "___acd"], dd[k2 + "___acd"]
    plan_xa, plan_ax = P.plan_from_acd(acd1, nX, nX, nA), P.plan_from_acd(acd2, nX, nA, nX)
    merged = P.sswl_bwd_group(acd1, acd2, k2 + "___acd", nX, nA)
    assert int(merged.rowptr[-1]) == acd1.shape[1] + acd2.shape[1]
    gen = torch.Generator(device=DEV).manual_seed(1)
    Xv0 = torch.randn(nX, d, generator=gen, device=DEV)
    Av0 = torch.randn(nA, d, generator=gen, device=DEV)
    w = torch.randn(nX, 3 * d, generator=gen, device=DEV)
    wr = torch.randn(nX, d, generator=gen, device=DEV)
    grads = []
    for m in (None, merged):
        Xv, Av = Xv0.clone().requires_grad_(True), Av0.clone().requires_grad_(True)
        out = SswlAggregate.apply(Xv, Av, plan_xa, plan_ax, 0, residual, m)
        if residual:
            cat, tap = out
            ((cat * w).sum() + (tap * wr).sum()).backward()
        else:
            (out * w).sum().backward()
        grads.append((Xv.grad, Av.grad))
    close(grads[1][0], grads[0][0], 2e-6)
    assert torch.equal(grads[1][1], grads[0][1])


@pytest.mark.parametrize("n,V,D", [(5, 16, 8), (300, 16, 128), (70001, 28, 128), (4097, 3, 32)])
def test_embedding_matches_torch(n, V, D):
    """pygho_b200.honn.utils.Embedding: forward bit-exact, deterministic weight gradient within
    fp32 summation error of torch's (which uses atomics), absent ids get a zero gradient."""
    from pygho_b200.honn.utils import Embedding
    torch.manual_seed(0)
    emb = Embedding(V, D).to(DEV)
    ref = torch.nn.Embedding(V, D).to(DEV)
    ref.load_state_dict(emb.state_dict())
    idx = torch.randint(0, max(1, V - 2), (n,), device=DEV)              # last two ids never occur
    w = torch.randn(n, D, device=DEV)
    out, out_ref = emb(idx), ref(idx)
    assert torch.equal(out, out_ref)
    (out * w).sum().backward()
    (out_ref * w).sum().backward()
    close(emb.weight.grad, ref.weight.grad.double(), 2e-6 * max(1.0, n / V) ** 0.5)
    assert float(emb.weight.grad[V - 2:].abs().max()) == 0.0
    g1 = emb.weight.grad.clone()
    emb.weight.grad = None
    (emb(idx) * w).sum().backward()
    assert torch.equal(emb.weight.grad, g1)                               # deterministic
    idx2 = idx.reshape(-1, 1)[: n - n % 1].reshape(n)                     # other tensor object
    assert torch.equal(emb(idx2.reshape(n, 1)).squeeze(1), out_ref)


def test_spmamm_matches_reference_golden_and_oracle(B, golden):
    """SD mode: sparse batched adjacency x masked dense tuples (backend/Spmamm.py)."""
    g = golden("spmamm")
    ind, shape = T(g["ind"]), tuple(int(x) for x in g["shape"])
    for tag, dim2 in (("d1", 1), ("d2", 2)):
        Bm = B.MaskedTensor(T(g[f"{tag}_data"]), T(g[f"{tag}_mask"]), 0.0, True)
        for aggr in ("sum", "max"):
            for dim1 in (1, 2):
                A = B.SparseTensor(ind, T(g["aval"]), shape, True)
                out = B.spmamm(A, dim1, Bm, dim2, None, aggr)
                close(out.data, g[f"{tag}_{aggr}_dim{dim1}"], 1e-6)
                assert torch.equal(out.mask, Bm.mask)
    # dense features (the reference cannot run these, Q7): oracle, values None, custom mask, min
    rng = np.random.default_rng(2)
    b, n, k, d = 3, 7, 5, 8
    aval = rng.standard_normal((g["ind"].shape[1], d)).astype(np.float32)
    bmask = g["d1_mask"]
    data = rng.standard_normal(bmask.shape + (d,)).astype(np.float32) * bmask[..., None]
    omask = bmask & (rng.random(bmask.shape) < 0.8)
    for aggr in ("sum", "max", "min"):
        for av in (aval, None):
            A = B.SparseTensor(ind, None if av is None else T(av), shape + ((d,) if av is not None else ()), True)
            out = B.spmamm(A, 2, B.MaskedTensor(T(data), T(bmask), 0.0, True), 1, T(omask), aggr)
            want, _ = O.spmamm(g["ind"], av, shape, 2, data, bmask, 1, omask, aggr)
            close(out.data, want, 2e-6)
    # gradients of the sum against torch autograd on the same arithmetic
    ar = torch.from_numpy(aval).requires_grad_(True)
    br = torch.from_numpy(data).requires_grad_(True)
    it = torch.from_numpy(g["ind"])
    rows = ar.unsqueeze(1) * br[it[0], it[2]]
    ref = torch.zeros((b * n, k, d)).index_add_(0, n * it[0] + it[1], rows).reshape(b, n, k, d)
    w = torch.randn(ref.shape, generator=torch.Generator().manual_seed(1)) * torch.from_numpy(bmask).unsqueeze(-1)
    (ref * w).sum().backward()
    ag, bg = torch.from_numpy(aval).to(DEV).requires_grad_(True), torch.from_numpy(data).to(DEV).requires_grad_(True)
    out = B.spmamm(B.SparseTensor(ind, ag, shape + (d,), True), 2,
                   B.MaskedTensor(bg, T(bmask), 0.0, True), 1, None, "sum")
    (out.data * w.to(DEV)).sum().backward()
    close(ag.grad, ar.grad, 2e-5)
    close(bg.grad * T(bmask).unsqueeze(-1), br.grad * torch.from_numpy(bmask).unsqueeze(-1), 2e-5)
    # operator level (honn/MaOperator.py:45-80, 281-372)
    from pygho_b200.honn.MaOperator import OpSpMessagePassingOnSubg2D, OpSpNodeMessagePassing
    X2 = B.MaskedTensor(T(data), T(bmask), 0.0, True)
    A = B.SparseTensor(ind, T(aval), shape + (d,), True)
    o = OpSpMessagePassingOnSubg2D("sum")(A, B.MaskedTensor(T(np.swapaxes(data, 1, 2).copy()), T(np.swapaxes(bmask, 1, 2).copy()), 0.0, True), None,
                                          B.MaskedTensor(T(np.swapaxes(data, 1, 2).copy()), T(np.swapaxes(bmask, 1, 2).copy()), 0.0, True))
    want, _ = O.spmamm(g["ind"], aval, shape, 1, np.swapaxes(data, 1, 2), np.swapaxes(bmask, 1, 2), 2, None, "sum")
    close(o.data, want, 2e-6)
    xn = data[:, :, 0]
    mn = bmask[:, :, 0]
    o = OpSpNodeMessagePassing("sum")(A, B.MaskedTensor(T(xn), T(mn), 0.0, True), B.MaskedTensor(T(xn), T(mn), 0.0, True))
    want, _ = O.spmamm(g["ind"], aval, shape, 2, xn, mn, 1, None, "sum")
    close(o.data, want, 2e-6)
    assert X2.masked_dim == 3


@pytest.mark.parametrize("shape,tuples,key,graphs", [("zinc", "khop", "X___X___1___X___0", 48),
                                                      ("sr25", "khop", "X___X___1___A___0", 6),
                                                      ("sr25", "i2", "X___X___2___A___0", 2)])
@pytest.mark.parametrize("aggr", ("sum", "mean"))
def test_high_reuse_keys_match_torch_oracle(B, shape, tuples, key, graphs, aggr):
    """Plans with many entries per row (2-FWL key, sr25-shaped keys, I2 key): values and both
    operand gradients equal the torch oracle within 2e-5."""
    from pygho_b200 import ops as OPS
    from pygho_b200 import plans as P
    from pygho_b200.hodata.synthetic import make_batch
    hb = make_batch(graphs, seed=5, tuples=tuples, shape=shape)
    ei, tid = T(hb.edge_index), T(hb.tupleid)
    _o0, o1, d1, o2, d2 = key.split("___")
    pick = lambda op: ei if op == "A" else tid  # noqa: E731
    acd = B.filterind(tid, *B.spspmm_ind(pick(o1), int(d1), pick(o2), int(d2)))
    n_out, n1, n2 = tid.shape[1], pick(o1).shape[1], pick(o2).shape[1]
    gen = torch.Generator().manual_seed(11)
    av, bv = torch.randn((n1, 128), generator=gen), torch.randn((n2, 128), generator=gen)
    w = torch.randn((n_out, 128), generator=gen).to(DEV)

    plan = P.plan_from_acd(acd.clone(), n_out, n1, n2)
    a, b = av.to(DEV).requires_grad_(True), bv.to(DEV).requires_grad_(True)
    out = OPS.seg_gmr(a, b, plan, aggr)
    (out * w).sum().backward()
    ar, br = av.clone().requires_grad_(True), bv.clone().requires_grad_(True)
    ref = TO.spspmm(ar, br, acd.cpu(), n_out, aggr)
    (ref * w.cpu()).sum().backward()
    close(out.detach(), ref, 2e-5)
    close(a.grad, ar.grad, 2e-5)
    close(b.grad, br.grad, 2e-5)
