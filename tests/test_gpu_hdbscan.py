"""HDBSCAN in degree mode (engine.degree_mreach_mst, HSD.mutual_reachability_mst / hdbscan): the *_mreach kernels
against numpy, the Borůvka rounds against Kruskal in the order E = (d_mr, u, v) on the dense mutual-reachability
matrix (u, v and the distance bits) and the cores against the np.partition formula, a device Prim at 100k nodes,
and the model API against scikit-learn's tree_to_labels and HDBSCAN(metric="precomputed").fit."""
import numpy as np
import pytest

from test_gpu_mst import _assert_mst_equal, _graph, _key, _prim_device, _same_partition
from test_host_hdbscan import hierarchy
from test_host_mst import kruskal

pytestmark = pytest.mark.gpu

NONE = 2 ** 63 - 1


def core_device(D, min_samples, rows=4096):
    """core[i] = the min_samples-th smallest of row i of D, the zero diagonal counted (np.partition's formula), by
    row chunks: a value of D, bit for bit."""
    import torch
    return torch.cat([torch.kthvalue(D[r0:r0 + rows], min_samples, dim=1).values
                      for r0 in range(0, D.shape[0], rows)])


def mreach_device_(D, core, rows=4096):
    """D <- max(D, core[i], core[j]) in place, by row chunks."""
    import torch
    for r0 in range(0, D.shape[0], rows):
        blk = D[r0:r0 + rows]
        torch.maximum(blk, core[r0:r0 + rows, None], out=blk)
        torch.maximum(blk, core[None, :], out=blk)
    return D


def kruskal_prefix(D):
    """(u, v, dist) of Kruskal in the order E over the resident matrix D (float32 CUDA [n, n]), as numpy.  The upper
    triangle in row-major order is sorted by (u, v); a stable sort by the distance bits gives the order E.  Kruskal
    accepts the same edges from the shortest prefix of that order that connects the nodes as from the whole order,
    so scipy's MST of the prefix's ranks (distinct weights) is its tree; the prefix grows until it connects."""
    import scipy.sparse as sp
    import torch
    from scipy.sparse.csgraph import connected_components, minimum_spanning_tree
    n = D.shape[0]
    iu = torch.triu_indices(n, n, 1, device=D.device)
    order = torch.argsort(D[iu[0], iu[1]].view(torch.int32), stable=True)
    m = min(8 * n, order.numel())
    while True:
        pick = order[:m]
        a, b = iu[0][pick].cpu().numpy(), iu[1][pick].cpu().numpy()
        W = sp.csr_matrix((np.arange(1, m + 1, dtype=np.float64), (a, b)), shape=(n, n))
        if m == order.numel() or connected_components(W, directed=False)[0] == 1:
            break
        m = min(4 * m, order.numel())
    r = np.sort(minimum_spanning_tree(W).tocoo().data.astype(np.int64) - 1)
    u, v = iu[0][pick[r]], iu[1][pick[r]]
    return u.int().cpu().numpy(), v.int().cpu().numpy(), D[u, v].cpu().numpy()


def reference_mreach(dg, hops, min_samples):
    """(core numpy, Kruskal's tree of the dense d_mr) from degree_distance_device."""
    from hsd_b200 import engine
    D, _ = engine.degree_distance_device(dg, hops)
    core = core_device(D, min_samples)
    want = kruskal_prefix(mreach_device_(D, core))
    return core.cpu().numpy(), want


# ---------------------------------------------------------------- kernels
@pytest.mark.parametrize("labels", ["random", "equal", "distinct"])
@pytest.mark.parametrize("R,C,ld,node0", [(77, 301, 304, 5), (5, 37, 40, 3), (130, 130, 133, 0), (33, 1000, 1003, 9),
                                          (1, 63, 64, 2), (200, 5000, 5000, 100), (300, 300, 301, 17)])
def test_mst_panel_min_mreach_on_quantized_blocks(R, C, ld, node0, labels):
    """test_mst_panel_min_on_quantized_blocks with cores: a few levels from 0 to above every distance, so that the
    row's core, the column's core and the distance each decide some keys.  With all cores 0 the keys are
    hsd_mst_panel_min's."""
    import torch
    from hsd_b200 import engine
    from hsd_b200._lib import check, lib
    rng = np.random.default_rng(R * 7 + C + node0)
    n = node0 + C + 3
    blk = np.zeros((R, ld), np.float32)
    up = np.triu(np.ones((R, C), bool), 1)
    blk[:, :C][up] = (rng.integers(1, 5, size=(R, C)).astype(np.float32) * np.float32(0.25))[up]
    comp = {"random": rng.integers(0, 4, n), "equal": np.zeros(n), "distinct": np.arange(n)}[labels].astype(np.int32)
    prior = np.full(n, NONE, np.int64)
    some = rng.choice(n, n // 4, replace=False)
    prior[some] = _key(np.where(rng.random(some.size) < 0.5, 0.0, 0.75), rng.integers(0, n, some.size))
    rr, cc = np.nonzero(up & (comp[node0 + np.arange(R)][:, None] != comp[node0 + np.arange(C)][None, :]))
    B = torch.from_numpy(blk).cuda()
    tc = torch.from_numpy(comp).cuda()
    for cores in ("random", "zero"):
        core = (rng.integers(0, 7, n).astype(np.float32) * np.float32(0.25) if cores == "random"
                else np.zeros(n, np.float32))
        d = np.maximum(blk[rr, cc], np.maximum(core[node0 + rr], core[node0 + cc]))
        want = prior.copy()
        np.minimum.at(want, node0 + rr, _key(d, node0 + cc))
        np.minimum.at(want, node0 + cc, _key(d, node0 + rr))
        keys = torch.from_numpy(prior).cuda()
        check(lib.hsd_mst_panel_min_mreach(B.data_ptr(), ld, R, C, node0, engine._ptr(tc),
                                           engine._ptr(torch.from_numpy(core).cuda()), engine._ptr(keys),
                                           engine._stream()))
        got = keys.cpu().numpy()
        assert np.array_equal(got, want), cores
        if cores == "zero":
            plain = torch.from_numpy(prior).cuda()
            check(lib.hsd_mst_panel_min(B.data_ptr(), ld, R, C, node0, engine._ptr(tc), engine._ptr(plain),
                                        engine._stream()))
            assert np.array_equal(got, plain.cpu().numpy())
        elif labels != "equal" and rr.size > 100:         # every operand decides some keys
            assert (d == blk[rr, cc]).any() and (d > blk[rr, cc]).any()
            assert (core > blk.max()).any() and (core == 0).any()
        if labels == "equal":
            assert np.array_equal(got, prior)


@pytest.mark.parametrize("k", [1, 5, 32, 64])
def test_mst_list_candidates_mreach(k):
    """Lists ordered by (distance, id) with ties, some short (padded with -1 / +inf), some drawn from their own
    component; cores on the distances' levels, so that many d_mr equal val[k-1] exactly (keys at the bound: not
    exact).  With all cores 0 the keys are hsd_mst_list_candidates'."""
    import torch
    from hsd_b200 import engine
    from hsd_b200._lib import check, lib
    rng = np.random.default_rng(k + 100)
    n = 700
    comp = rng.integers(0, 6, n).astype(np.int32)
    idx = np.full((n, k), -1, np.int32)
    val = np.full((n, k), np.inf, np.float32)
    for i in range(n):
        length = k if rng.random() < 0.8 else int(rng.integers(0, k + 1))
        inside = rng.random() < 0.3
        pool = np.flatnonzero(comp == comp[i]) if inside else np.arange(n)
        js = rng.choice(pool[pool != i], length, replace=False)
        ds = rng.integers(0, 4, length).astype(np.float32) * np.float32(0.5)
        o = np.lexsort((js, ds))
        idx[i, :length], val[i, :length] = js[o], ds[o]
    ti, tv, tc = (torch.from_numpy(a).cuda() for a in (idx, val, comp))
    keys = torch.empty(n, dtype=torch.int64, device="cuda")
    bound = torch.empty(n, dtype=torch.float32, device="cuda")
    at_bound = 0
    for cores in ("random", "zero"):
        core = (rng.integers(0, 5, n).astype(np.float32) * np.float32(0.5) if cores == "random"
                else np.zeros(n, np.float32))
        want_key = np.full(n, NONE, np.int64)
        want_bound = np.full(n, np.inf, np.float32)
        for i in range(n):
            out = [t for t in range(k) if idx[i, t] >= 0 and comp[idx[i, t]] != comp[i]]
            ks = [_key(max(core[i], core[idx[i, t]], val[i, t]), idx[i, t]) for t in out]
            if ks:
                want_key[i] = min(ks)
            full = idx[i, k - 1] >= 0
            dk = np.int64(want_key[i]) >> 32
            exact = not full or (ks and dk < np.float32(val[i, k - 1]).view(np.int32))
            if not exact:
                want_bound[i] = val[i, k - 1]
                at_bound += bool(ks) and dk == np.float32(val[i, k - 1]).view(np.int32)
        check(lib.hsd_mst_list_candidates_mreach(engine._ptr(ti), engine._ptr(tv), n, k, engine._ptr(tc),
                                                 engine._ptr(torch.from_numpy(core).cuda()), engine._ptr(keys),
                                                 engine._ptr(bound), engine._stream()))
        assert np.array_equal(keys.cpu().numpy(), want_key), cores
        assert np.array_equal(bound.cpu().numpy(), want_bound), cores
        assert (want_key == NONE).sum() > 10 and (want_key != NONE).sum() > 10
        assert (want_bound < np.inf).sum() > 10 and (want_bound == np.inf).sum() > 10
        if cores == "zero":
            plain = torch.empty_like(keys)
            check(lib.hsd_mst_list_candidates(engine._ptr(ti), engine._ptr(tv), n, k, engine._ptr(tc),
                                              engine._ptr(plain), engine._ptr(bound), engine._stream()))
            assert np.array_equal(keys.cpu().numpy(), plain.cpu().numpy())
    assert at_bound > 10


# ---------------------------------------------------------------- Borůvka rounds == Kruskal on the dense d_mr
@pytest.mark.parametrize("hops", [1, 2, 3, 4])
@pytest.mark.parametrize("graph", ["karate", "barbell", "europe", 2000, 10000])
def test_degree_mreach_mst_equals_kruskal(golden_graphs, graph, hops):
    from hsd_b200 import engine
    from hsd_b200.graph import powerlaw_graph
    g = _graph(golden_graphs, graph) if isinstance(graph, str) else powerlaw_graph(graph, 5, seed=1)
    dg = engine.DeviceGraph.upload(g)
    try:
        engine.degree_distance_device(dg, hops)
    except engine.EmptyRingError:                           # a ring runs empty at this depth: both paths raise
        for cand_k in (0, 64):
            with pytest.raises(engine.EmptyRingError, match="Distribution can't be empty."):
                engine.degree_mreach_mst(dg, hops, 2, cand_k=cand_k, panel_rows=128)
        return
    for ms in (1, 2, 5, 17, 65):
        if ms > g.n:
            with pytest.raises(ValueError, match="min_samples"):
                engine.degree_mreach_mst(dg, hops, ms)
            continue
        core, want = reference_mreach(dg, hops, ms)
        if ms == 1:
            assert not core.any()
        for p in (None, 128):
            for cand_k in (0, 64):
                stats = {}
                u, v, d, c = engine.degree_mreach_mst(dg, hops, ms, cand_k=cand_k, panel_rows=p, stats=stats)
                _assert_mst_equal((u, v, d), want)
                assert np.array_equal(c.cpu().numpy().view(np.int32), core.view(np.int32)), (ms, p, cand_k)
                assert stats["rounds"] <= max(1, int(np.ceil(np.log2(g.n))))
                if cand_k == 0:
                    assert stats["sweeps"] == stats["rounds"]
                if ms == 1:
                    _assert_mst_equal((u, v, d), tuple(t.cpu().numpy() for t in
                                                       engine.degree_mst(dg, hops, cand_k=cand_k, panel_rows=p)))


def test_degree_mreach_mst_100k_equals_device_prim():
    """100k nodes (BA m = 5), 4 hops, min_samples = 5: the default plan against a device Prim on the resident 40 GB
    d_mr matrix; the cores against the np.partition formula."""
    from hsd_b200 import engine
    from hsd_b200.graph import powerlaw_graph
    n, hops, ms = 100000, 4, 5
    dg = engine.DeviceGraph.upload(powerlaw_graph(n, 5, seed=0))
    stats = {}
    u, v, d, c = engine.degree_mreach_mst(dg, hops, ms, stats=stats)
    got = tuple(t.cpu().numpy() for t in (u, v, d))
    c = c.cpu().numpy()
    del u, v, d
    D, _ = engine.degree_distance_device(dg, hops)
    core = core_device(D, ms)
    assert np.array_equal(c.view(np.int32), core.cpu().numpy().view(np.int32))
    _assert_mst_equal(got, _prim_device(mreach_device_(D, core)))
    assert stats["rounds"] <= 17


# ---------------------------------------------------------------- model
def _model(G, name, hop):
    from model import HSD
    return HSD(G, name, 0, hop, "wasserstein", signal="degree")


@pytest.mark.parametrize("ms", [None, 2, 17])
def test_model_hdbscan_equals_tree_to_labels(ms):
    """HSD.hdbscan against tree_to_labels of the Z of the Kruskal reference, bit for bit (labels and probability
    bits), both methods, both allow_single_cluster values, on a 2000-node graph at 2 hops."""
    import networkx as nx
    import torch
    from sklearn.cluster._hdbscan._tree import tree_to_labels
    from hsd_b200.engine import single_linkage_host
    m = _model(nx.barabasi_albert_graph(2000, 3, seed=5), "ba2k", 2)
    mcs = 8
    D = m.structural_distance_device().to(torch.float32)
    core = core_device(D, mcs if ms is None else ms)
    Z = single_linkage_host(*kruskal_prefix(mreach_device_(D, core)), m.n_node)
    del D
    for method in ("eom", "leaf"):
        for single in (False, True):
            labels, prob = m.hdbscan(min_cluster_size=mcs, min_samples=ms, cluster_selection_method=method,
                                     allow_single_cluster=single)
            want_l, want_p = tree_to_labels(hierarchy(Z), mcs, method, single, 0.0, None)
            assert labels.dtype == np.int64 and prob.dtype == np.float64
            assert np.array_equal(labels, want_l) and np.array_equal(prob.view(np.int64), want_p.view(np.int64))


@pytest.mark.parametrize("hop,ms,distinct", [(3, 1, True), (3, 2, True), (3, 5, False), (2, 1, False), (2, 2, False),
                                             (2, 5, False)])
def test_model_hdbscan_against_sklearn_fit(hop, ms, distinct):
    """HDBSCAN(metric="precomputed").fit on the same D (as float64).  The sorted heights of the tree are the same
    for every minimal tree and must equal sklearn's.  Where they are pairwise distinct (asserted per case) the
    minimal tree is unique: the partition, the noise set and the probabilities must equal sklearn's too.  On this
    graph that holds at 3 hops for min_samples <= 2; at 2 hops two of the float32 heights tie."""
    import networkx as nx
    from sklearn.cluster import HDBSCAN
    m = _model(nx.gnp_random_graph(300, 0.02, seed=1), "gnp300", hop)
    D = m.structural_distance_device().cpu().numpy().astype(np.float64)
    u, v, d = m.mutual_reachability_mst(ms)
    assert (np.unique(d).size == d.size) == distinct
    for mcs in (2, 5):
        for method in ("eom", "leaf"):
            fit = HDBSCAN(metric="precomputed", min_cluster_size=mcs, min_samples=ms, copy=True,
                          cluster_selection_method=method).fit(D)
            assert np.array_equal(np.sort(fit._single_linkage_tree_["value"]), d.astype(np.float64))
            if distinct:
                labels, prob = m.hdbscan(min_cluster_size=mcs, min_samples=ms, cluster_selection_method=method)
                assert np.array_equal(labels == -1, fit.labels_ == -1)
                assert _same_partition(labels, fit.labels_)
                assert np.array_equal(prob, fit.probabilities_)


def test_model_hdbscan_edge_cases(golden_graphs):
    import networkx as nx
    from conftest import nx_graph
    from model import HSD
    from hsd_b200.engine import EmptyRingError
    w = HSD(nx_graph(golden_graphs, "karate"), "karate", 1.0, 2, "wasserstein")
    with pytest.raises(NotImplementedError):
        w.hdbscan()
    with pytest.raises(NotImplementedError):
        w.mutual_reachability_mst()
    G = nx.barabasi_albert_graph(300, 3, seed=2)
    G.add_nodes_from([300, 301])                            # isolated nodes: their rings run empty
    m = _model(G, "iso", 2)
    with pytest.raises(EmptyRingError):
        m.hdbscan()
    with pytest.raises(EmptyRingError):
        m.mutual_reachability_mst()
    m.empty = "zero"
    labels, prob = m.hdbscan()
    assert labels.shape == prob.shape == (302,)
    m = _model(nx_graph(golden_graphs, "karate"), "karate", 2)
    n = m.n_node
    u, v, d = m.mutual_reachability_mst(n)                  # min_samples = N: every core is its row's maximum
    D = m.structural_distance_device().cpu().numpy()
    core = D.max(1)
    assert np.array_equal(d, kruskal(np.maximum(D, np.maximum(core[:, None], core[None, :])))[2])
    labels, _ = m.hdbscan(min_cluster_size=2, min_samples=n)
    assert labels.shape == (n,)
    for kw, match in (({"min_samples": n + 1}, "min_samples"), ({"min_cluster_size": 1}, "min_cluster_size"),
                      ({"cluster_selection_method": "dbscan"}, "cluster_selection_method"),
                      ({"min_samples": 0}, "min_samples")):
        with pytest.raises(ValueError, match=match):
            m.hdbscan(**kw)
    with pytest.raises(ValueError, match="min_samples"):
        m.mutual_reachability_mst(n + 1)
    two = _model(nx.path_graph(2), "two", 1)
    two.empty = "zero"
    labels, prob = two.hdbscan(min_cluster_size=2, min_samples=2)
    assert labels.shape == prob.shape == (2,)
    u, v, d = two.mutual_reachability_mst(2)
    assert u.tolist() == [0] and v.tolist() == [1]
    for g in (nx.path_graph(1), nx.Graph()):
        with pytest.raises(ValueError, match="more than one sample"):
            _model(g, "tiny", 1).hdbscan(min_cluster_size=2, min_samples=1)
