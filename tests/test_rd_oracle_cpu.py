"""The resistance-distance oracle (``oracle.rd_oracle.rd_matrix``) against closed forms.
No golden vectors exist for ``rdsampler``, so these pin the definition the GPU kernel is
compared with: effective resistance of the simple undirected graph, ``L+_ii + L+_jj`` across
components."""
import numpy as np
import pytest

from oracle import hodata_oracle as H
from oracle.rd_oracle import rd_matrix


def _und(pairs):
    """(2, 2m) edge_index with both directions of the undirected pairs."""
    e = np.asarray(pairs, dtype=np.int64).reshape(-1, 2).T
    return np.concatenate([e, e[::-1]], axis=1)


def test_trees_equal_hop_distance():
    rng = np.random.default_rng(0)
    for n in (1, 2, 7, 30, 128):
        path = _und([(i, i + 1) for i in range(n - 1)])
        assert np.allclose(rd_matrix(path, n), H.spd_matrix(path, n, 10 * n), atol=1e-9)
    for n in (5, 17, 40):
        tree = _und([(int(rng.integers(v)), v) for v in range(1, n)])
        assert np.allclose(rd_matrix(tree, n), H.spd_matrix(tree, n, 10 * n), atol=1e-9)


@pytest.mark.parametrize("n", [3, 4, 9, 25])
def test_cycle(n):
    R = rd_matrix(_und([(i, (i + 1) % n) for i in range(n)]), n)
    k = np.abs(np.arange(n)[:, None] - np.arange(n)[None, :])
    assert np.allclose(R, k * (n - k) / n, atol=1e-12)


@pytest.mark.parametrize("n", [2, 5, 12])
def test_complete_graph(n):
    R = rd_matrix(_und([(i, j) for i in range(n) for j in range(i + 1, n)]), n)
    assert np.allclose(R, 2.0 / n * (1 - np.eye(n)), atol=1e-12)


def test_sr25_two_values():
    """Laplacian spectrum of a (25, 12, 5, 6) graph: 0 once, 10 and 15 twelve times each, so
    adjacent pairs are 4/25 apart and non-adjacent pairs 13/75."""
    from pygho_b200.hodata.synthetic import sr25_like_graph
    rng = np.random.default_rng(3)
    for which in (0, 1):
        g = sr25_like_graph(rng, which=which)
        R = rd_matrix(g.edge_index, 25)
        adj = np.zeros((25, 25), dtype=bool)
        adj[g.edge_index[0], g.edge_index[1]] = True
        off = ~np.eye(25, dtype=bool)
        assert np.allclose(R[adj], 4 / 25, atol=1e-12)
        assert np.allclose(R[off & ~adj], 13 / 75, atol=1e-12)
        assert (np.diag(R) == 0).all()


def test_foster_theorem_on_zinc_shaped_graphs():
    """Sum of R over the undirected edges = n - #components."""
    from pygho_b200.hodata.synthetic import make_graphs
    for g in make_graphs(20, seed=5):
        R = rd_matrix(g.edge_index, g.num_nodes)
        und = g.edge_index[:, g.edge_index[0] < g.edge_index[1]]
        assert abs(R[und[0], und[1]].sum() - (g.num_nodes - 1)) < 1e-9     # connected
    # two graphs side by side: one more component
    a, b = make_graphs(2, seed=6)
    ei = np.concatenate([a.edge_index, b.edge_index + a.num_nodes], axis=1)
    n = a.num_nodes + b.num_nodes
    R = rd_matrix(ei, n)
    und = ei[:, ei[0] < ei[1]]
    assert abs(R[und[0], und[1]].sum() - (n - 2)) < 1e-9


def test_two_components():
    c5 = _und([(i, (i + 1) % 5) for i in range(5)])
    p4 = _und([(i, i + 1) for i in range(3)])
    ei = np.concatenate([c5, p4 + 5], axis=1)
    R = rd_matrix(ei, 9)
    assert np.allclose(R[:5, :5], rd_matrix(c5, 5), atol=1e-12)
    assert np.allclose(R[5:, 5:], rd_matrix(p4, 4), atol=1e-12)
    # across components: L+_ii + L+_jj, each from the component's own pseudo-inverse
    d5 = np.diag(np.linalg.pinv(np.diag([2.0] * 5) - (np.roll(np.eye(5), 1, 1) + np.roll(np.eye(5), -1, 1))))
    lp = np.diag([1.0, 2.0, 2.0, 1.0]) - (np.eye(4, k=1) + np.eye(4, k=-1))
    d4 = np.diag(np.linalg.pinv(lp))
    assert np.allclose(R[:5, 5:], d5[:, None] + d4[None, :], atol=1e-12)
    assert np.allclose(R, R.T, atol=0)


def test_isolated_node_and_edgeless_graph():
    tri = _und([(0, 1), (1, 2), (0, 2)])
    R = rd_matrix(tri, 4)                       # node 3 isolated: L+_33 = 0
    assert np.allclose(R[:3, :3], 2 / 3 * (1 - np.eye(3)), atol=1e-12)
    Lp = np.linalg.pinv(np.array([[2.0, -1, -1], [-1, 2, -1], [-1, -1, 2]]))
    assert np.allclose(R[:3, 3], np.diag(Lp), atol=1e-12) and R[3, 3] == 0
    assert (rd_matrix(np.zeros((2, 0), dtype=np.int64), 6) == 0).all()


def test_duplicates_and_self_loops_do_not_count():
    rng = np.random.default_rng(9)
    n = 12
    base = _und([(i, i + 1) for i in range(n - 1)] + [(0, 6), (3, 9)])
    noisy = np.concatenate([base, base[:, :5], np.stack([np.arange(4), np.arange(4)])], axis=1)
    noisy = noisy[:, rng.permutation(noisy.shape[1])]
    one_way = base[:, base[0] < base[1]]                       # one direction only
    R = rd_matrix(base, n)
    assert np.array_equal(rd_matrix(noisy, n), R)
    assert np.array_equal(rd_matrix(one_way, n), R)
