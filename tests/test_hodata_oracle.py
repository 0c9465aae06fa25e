"""Pin oracle/hodata_oracle.py (batch preparation: k-hop tuples, SPD features, dense padding)
to the real reference -- golden vectors from tests/golden/make_golden_hodata.py -- and check the
host-side generator of this repo against it."""
import numpy as np

from oracle import hodata_oracle as H
from pygho_b200.hodata.synthetic import collate, khop_tuples, make_graphs


def test_k_hop_subgraph_golden(golden):
    g = golden("hodata")
    for hop in (2, 3):
        for gi in range(6):
            ei, n = g[f"g{gi}_edge_index"], int(g[f"g{gi}_n"])
            subs, dists, lens = [], [], []
            for i in range(n):
                s, d = H.k_hop_subgraph(i, hop, ei, n)
                subs.append(s); dists.append(d); lens.append(s.shape[0])
            assert np.array_equal(np.array(lens), g[f"khop{hop}_g{gi}_len"])
            assert np.array_equal(np.concatenate(subs), g[f"khop{hop}_g{gi}_subset"])
            assert np.array_equal(np.concatenate(dists), g[f"khop{hop}_g{gi}_dist"])
            # KhopSampler content = the same lists with the root repeated
            tid, feat = H.khop_sampler(ei, n, hop)
            assert np.array_equal(tid[1], g[f"khop{hop}_g{gi}_subset"])
            assert np.array_equal(tid[0], np.repeat(np.arange(n), g[f"khop{hop}_g{gi}_len"]))
            assert np.array_equal(feat, g[f"khop{hop}_g{gi}_dist"])


def test_k_hop_subgraph_directed_golden(golden):
    g = golden("hodata")
    ei = g["dir_edge_index"]
    subs, dists = [], []
    for i in range(12):
        s, d = H.k_hop_subgraph(i, 2, ei, 12)
        subs.append(s); dists.append(d)
    assert np.array_equal(np.concatenate(subs), g["dir_subset"])
    assert np.array_equal(np.concatenate(dists), g["dir_dist"])


def test_spd_golden(golden):
    g = golden("hodata")
    for gi in range(4):
        assert np.array_equal(H.spd_matrix(g[f"g{gi}_edge_index"], int(g[f"g{gi}_n"]), 3),
                              g[f"spd_g{gi}"])
    # disconnected graph: the reference converts scipy's inf to int64 (INT64_MIN on x86) BEFORE
    # clamping (MaTupleSampler.py:29-30), so unreachable pairs come out as INT64_MIN and would
    # crash the embedding lookup; the intended value -- and ours -- is hop + 1 (DESIGN.md Q14)
    got, ref = H.spd_matrix(g["spd_disc_edge_index"], 6, 2), g["spd_disc"]
    reach = ref >= 0
    assert np.array_equal(got[reach], ref[reach]) and (got[~reach] == 3).all()
    assert (~reach).sum() == 6 * 6 - (9 + 4 + 1)


def test_i2_sampler_golden(golden):
    g = golden("hodata")
    for gi in range(3):
        ei, n = g[f"g{gi}_edge_index"], int(g[f"g{gi}_n"])
        tid, feat = H.i2_sampler(ei, n, 3)
        assert np.array_equal(tid[2], g[f"i2_g{gi}_subset"])
        assert np.array_equal(feat, g[f"i2_g{gi}_feat"])
        assert np.array_equal(tid[0], np.repeat(ei[0], g[f"i2_g{gi}_len"]))
        assert np.array_equal(tid[1], np.repeat(ei[1], g[f"i2_g{gi}_len"]))
        assert feat.max() <= 4                          # connected pairs: never beyond hop + 1
        from pygho_b200.hodata.synthetic import i2_tuples
        tid2, feat2 = i2_tuples(n, ei, 3)               # the generator's host sampler
        assert np.array_equal(tid, tid2) and np.array_equal(feat, feat2)


def test_dense_layout_golden(golden):
    g = golden("hodata")
    data, mask = H.to_dense_x(g["dx_x"], g["dx_ptr"])
    assert np.array_equal(data, g["dx_data"]) and np.array_equal(mask, g["dx_mask"])
    data, mask = H.to_dense_adj(g["da_ei"], g["da_eb"], g["da_ea"], 6, 4)
    assert np.array_equal(data, g["da_data"]) and np.array_equal(mask, g["da_mask"])
    data, _ = H.to_dense_adj(g["da_ei"], g["da_eb"], g["da_eaf"], 6, 4)
    assert np.array_equal(data, g["da_dataf"])
    data, mask = H.to_dense_tuplefeat(g["dt_feat"], g["dt_shape"], g["dt_ptr"])
    assert np.array_equal(data, g["dt_data"]) and np.array_equal(mask, g["dt_mask"])


def test_host_generator_matches_oracle_sampler():
    graphs = make_graphs(5, seed=3, hop=3)
    for gr in graphs:
        tid, feat = H.khop_sampler(gr.edge_index, gr.num_nodes, 3)
        tid2, feat2 = khop_tuples(gr.num_nodes, gr.edge_index, 3)
        assert np.array_equal(tid, tid2) and np.array_equal(feat, feat2)
    hb = collate(graphs)
    tid, feat = H.khop_sampler_batch(hb.edge_index, hb.node_ptr, 3)
    assert np.array_equal(tid, hb.tupleid) and np.array_equal(feat, hb.tuplefeat)
    # spd restricted to <= hop agrees with the k-hop distances
    gr = graphs[0]
    spd = H.spd_matrix(gr.edge_index, gr.num_nodes, 3)
    t, f = H.khop_sampler(gr.edge_index, gr.num_nodes, 3)
    assert np.array_equal(spd[t[0], t[1]], f)
    assert (spd <= 3).sum() == t.shape[1]


def test_sr25_like_graphs_are_strongly_regular():
    """The synthetic cfg4 graphs have the sr25 parameters (25, 12, 5, 6) and the tuple / triple
    counts SURVEY.md section 8 quotes for sr25.  The reference's sr25 dataset holds all 15
    strongly regular graphs with these parameters (Paulus), so the two Latin-square graphs are
    members of it, and distinct ones because they are not isomorphic."""
    import networkx as nx
    from pygho_b200.hodata.synthetic import make_batch, sr25_like_graph
    rng = np.random.default_rng(0)
    mats = []
    for which in (0, 1):
        g = sr25_like_graph(rng, which=which)
        A = np.zeros((25, 25), np.int64)
        A[g.edge_index[0], g.edge_index[1]] = 1
        assert (A == A.T).all() and (A.sum(0) == 12).all() and g.edge_index.shape[1] == 300
        A2 = A @ A
        off = ~np.eye(25, dtype=bool)
        assert set(A2[(A == 1) & off]) == {5} and set(A2[(A == 0) & off]) == {6}
        assert g.tupleid.shape[1] == 625 and g.tuplefeat.max() == 2
        mats.append(A)
    hb = make_batch(2, seed=1, tuples="i2", shape="sr25")
    assert hb.tupleid.shape == (3, 2 * 7500) and hb.tuplefeat.shape == (2 * 7500, 2)
    assert not nx.is_isomorphic(nx.from_numpy_array(mats[0]), nx.from_numpy_array(mats[1]))
