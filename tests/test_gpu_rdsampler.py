"""GPU checks of the resistance-distance sampler (``pgh_resistance_f32`` + ``pgh_rd_dense_f32``
through ``rdsampler`` / ``rd_tuplefeat``) against the fp64 numpy oracle and closed forms."""
import numpy as np
import pytest
import torch

from oracle.rd_oracle import rd_matrix

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda", 0)


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _und(pairs):
    e = np.asarray(pairs, dtype=np.int64).reshape(-1, 2).T
    return np.concatenate([e, e[::-1]], axis=1)


def _batch(graphs):
    """(edge_index, node_ptr) of a block-diagonal batch of (edge_index, n) pairs."""
    eis, ptr = [], [0]
    for ei, n in graphs:
        eis.append(np.asarray(ei, dtype=np.int64).reshape(2, -1) + ptr[-1])
        ptr.append(ptr[-1] + n)
    return np.concatenate(eis, axis=1), np.array(ptr, dtype=np.int64)


def _check_against_oracle(X, ei, node_ptr):
    data, mask = X.data.cpu().numpy(), X.mask.cpu().numpy()
    assert data.dtype == np.float32 and X.padvalue == 0
    nmax = data.shape[1]
    for g in range(node_ptr.shape[0] - 1):
        n0, n1 = int(node_ptr[g]), int(node_ptr[g + 1])
        n = n1 - n0
        sel = (ei[0] >= n0) & (ei[0] < n1)
        want = rd_matrix(ei[:, sel] - n0, n)
        got = data[g, :n, :n]
        assert np.abs(got - want).max(initial=0) <= 1e-6 * max(1.0, want.max(initial=0)), g
        m = np.zeros((nmax, nmax), dtype=bool)
        m[:n, :n] = True
        assert np.array_equal(mask[g], m) and (data[g][~m] == 0).all()
        assert np.array_equal(got, got.T) and (np.diag(got) == 0).all()


def test_zinc_batch_matches_oracle(dev):
    from pygho_b200.hodata.MaTupleSampler import rdsampler
    from pygho_b200.hodata.synthetic import make_batch
    hb = make_batch(1024, seed=0)
    X = rdsampler(_t(hb.edge_index, dev), hb.node_ptr)
    nmax = int(np.diff(hb.node_ptr).max())
    assert tuple(X.data.shape) == (1024, nmax, nmax)
    _check_against_oracle(X, hb.edge_index, hb.node_ptr)


def test_sr25_two_values(dev):
    from pygho_b200.hodata.MaTupleSampler import rdsampler
    from pygho_b200.hodata.synthetic import make_batch
    hb = make_batch(64, seed=2, shape="sr25")
    X = rdsampler(_t(hb.edge_index, dev), hb.node_ptr)
    data = X.data.cpu().numpy()
    adj = np.zeros((64, 25, 25), dtype=bool)
    adj[hb.batch[hb.edge_index[0]], hb.edge_index[0] % 25, hb.edge_index[1] % 25] = True
    eye = np.eye(25, dtype=bool)[None]
    want = np.where(adj, np.float32(4 / 25), np.float32(13 / 75)).astype(np.float32)
    want[np.broadcast_to(eye, want.shape)] = 0
    ulps = np.abs(data.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
    assert ulps.max() <= 1, ulps.max()


def test_deterministic_and_batch_independent(dev):
    from pygho_b200.hodata.MaTupleSampler import rdsampler
    from pygho_b200.hodata.synthetic import make_batch
    hb = make_batch(96, seed=7)
    ei = _t(hb.edge_index, dev)
    a, b = rdsampler(ei, hb.node_ptr), rdsampler(ei, hb.node_ptr)
    assert torch.equal(a.data, b.data) and torch.equal(a.mask, b.mask)
    perm = np.random.default_rng(1).permutation(hb.edge_index.shape[1])
    c = rdsampler(_t(hb.edge_index[:, perm], dev), _t(hb.node_ptr, dev), grouped=False)
    assert torch.equal(a.data, c.data) and torch.equal(a.mask, c.mask)
    for g in (0, 41, 95):
        n0, n1 = int(hb.node_ptr[g]), int(hb.node_ptr[g + 1])
        sel = hb.batch[hb.edge_index[0]] == g
        alone = rdsampler(_t(hb.edge_index[:, sel] - n0, dev), [0, n1 - n0])
        assert torch.equal(alone.data[0], a.data[g, :n1 - n0, :n1 - n0])


def test_edge_cases_match_oracle(dev):
    from pygho_b200.hodata.MaTupleSampler import rdsampler
    c6 = _und([(i, (i + 1) % 6) for i in range(6)])
    p5 = _und([(i, i + 1) for i in range(4)])
    disconnected = (np.concatenate([c6, p5 + 6], axis=1), 11)
    isolated = (_und([(0, 1), (1, 2), (2, 0), (2, 3)]), 5)          # node 4 has no edge
    single = (np.zeros((2, 0), dtype=np.int64), 1)
    noisy_base = _und([(i, i + 1) for i in range(8)] + [(0, 5), (2, 7)])
    noisy = np.concatenate([noisy_base, noisy_base[:, 3:9], np.stack([np.arange(4)] * 2),
                            noisy_base[:, :4][::-1]], axis=1)       # duplicates + self-loops
    ei, ptr = _batch([disconnected, isolated, single, (noisy, 9)])
    X = rdsampler(_t(ei, dev), ptr, max_num_nodes=14)
    assert tuple(X.data.shape) == (4, 14, 14)
    _check_against_oracle(X, ei, ptr)
    noisy_alone = rdsampler(_t(noisy, dev), [0, 9]).data
    assert torch.equal(noisy_alone, rdsampler(_t(noisy_base, dev), [0, 9]).data)
    # a batch without edges: all zeros, mask still the graph sizes
    X = rdsampler(torch.zeros((2, 0), dtype=torch.int64, device=dev), [0, 3, 7])
    assert tuple(X.data.shape) == (2, 4, 4) and not X.data.any()
    assert int(X.mask.sum()) == 9 + 16
    # an empty batch
    X = rdsampler(torch.zeros((2, 0), dtype=torch.int64, device=dev), [0])
    assert X.data.numel() == 0 and X.data.dtype == torch.float32
    with pytest.raises(AssertionError, match="max_num_nodes"):
        rdsampler(_t(ei, dev), ptr, max_num_nodes=10)


def test_largest_supported_graph_and_limit(dev):
    from pygho_b200 import _lib
    from pygho_b200.hodata.MaTupleSampler import rdsampler
    rng = np.random.default_rng(4)
    n = 128
    path = [(i, i + 1) for i in range(n - 1)]                         # ill-conditioned: long path
    chords = [tuple(sorted(map(int, rng.choice(n, 2, replace=False)))) for _ in range(6)]
    dense = [(int(a), int(b)) for a, b in zip(rng.integers(0, n, 2000), rng.integers(0, n, 2000))]
    ei, ptr = _batch([(_und(path), n), (_und(path + chords), n), (_und(dense), n)])
    X = rdsampler(_t(ei, dev), ptr)
    _check_against_oracle(X, ei, ptr)
    big = _und([(i, i + 1) for i in range(128)])
    with pytest.raises(_lib.KernelError, match="1..128 nodes"):
        rdsampler(_t(big, dev), [0, 129])


def test_rd_tuplefeat_and_ma_datadict(dev):
    from pygho_b200.hodata.device import ma_datadict
    from pygho_b200.hodata.MaTupleSampler import rdsampler
    from pygho_b200.hodata.SpTupleSampler import KhopSampler, rd_tuplefeat
    from pygho_b200.hodata.synthetic import make_batch
    hb = make_batch(64, seed=5)
    ei = _t(hb.edge_index, dev)
    dense = rdsampler(ei, hb.node_ptr)
    tid = KhopSampler(ei, hb.node_ptr, 3).indices
    feat = rd_tuplefeat(tid, ei, hb.node_ptr)
    g = _t(hb.batch, dev)[tid[0]]
    n0 = _t(hb.node_ptr, dev)[g]
    assert feat.dtype == torch.float32
    assert torch.equal(feat, dense.data[g, tid[0] - n0, tid[1] - n0])
    assert rd_tuplefeat(tid[:, :0], ei, hb.node_ptr).numel() == 0
    with pytest.raises(ValueError, match="one graph"):
        rd_tuplefeat(torch.tensor([[0], [int(hb.node_ptr[1])]], device=dev), ei, hb.node_ptr)
    X = ma_datadict(hb, dev, tuples="rd")["X"]
    assert torch.equal(X.data, dense.data) and torch.equal(X.mask, dense.mask)


def test_cuda_graph_replay_matches_eager(dev):
    from pygho_b200.hodata.MaTupleSampler import rdsampler
    from pygho_b200.hodata.synthetic import make_batch
    hb = make_batch(128, seed=9)
    ei = _t(hb.edge_index, dev)
    eager = rdsampler(ei, hb.node_ptr)
    # a host node_ptr in page-locked memory: sizes are read on the host, and the graph's copy
    # of it to the device reads this buffer at every replay, so it lives as long as the graph
    host_ptr = torch.from_numpy(hb.node_ptr).pin_memory()
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        rdsampler(ei, host_ptr)                                         # warm-up off the graph
    torch.cuda.current_stream(dev).wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        X = rdsampler(ei, host_ptr)
    X.data.fill_(-1.0)
    graph.replay()
    torch.cuda.synchronize(dev)
    assert torch.equal(X.data, eager.data) and torch.equal(X.mask, eager.mask)
