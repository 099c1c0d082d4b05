"""Minimum spanning tree and single linkage (engine.degree_mst, HSD.minimum_spanning_tree / single_linkage): the
hsd_mst_* kernels against numpy, the Borůvka sweep against Kruskal in the order E = (D[u, v], u, v) on the resident
matrix (u, v and the distance bits), a device Prim at 100k nodes, a graph beyond the device memory, and the model
API against scipy and the radius graph."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

NONE = 2 ** 63 - 1


def _graph(golden_graphs, name):
    from hsd_b200.graph import CSRGraph
    nodes = golden_graphs[f"{name}_nodes"]
    return CSRGraph.from_edges(len(nodes), golden_graphs[f"{name}_edges"], list(nodes))


def _key(d, j):
    return (np.asarray(d, np.float32).view(np.int32).astype(np.int64) << 32) | np.asarray(j, np.int64)


def kruskal_resident(D):
    """(u, v, dist) of Kruskal in the order E over the resident matrix D (float32 CUDA [n, n]), as numpy.  The
    upper triangle in row-major order is sorted by (u, v); a stable sort by the distance bits gives the order E.
    The edges' ranks in it are distinct weights, so scipy's MST of the rank matrix is that Kruskal's tree."""
    import scipy.sparse as sp
    import torch
    from scipy.sparse.csgraph import minimum_spanning_tree
    n = D.shape[0]
    iu = torch.triu_indices(n, n, 1, device=D.device)
    order = torch.argsort(D[iu[0], iu[1]].view(torch.int32), stable=True)
    rank = torch.empty_like(order)
    rank[order] = torch.arange(1, order.numel() + 1, device=D.device)
    indptr = np.concatenate([[0], np.cumsum(np.arange(n - 1, -1, -1))])
    W = sp.csr_matrix((rank.double().cpu().numpy(), iu[1].int().cpu().numpy(), indptr), shape=(n, n))
    pick = order[torch.from_numpy(np.sort(minimum_spanning_tree(W).data.astype(np.int64) - 1)).to(D.device)]
    u, v = iu[0][pick], iu[1][pick]
    return u.int().cpu().numpy(), v.int().cpu().numpy(), D[u, v].cpu().numpy()


def _assert_mst_equal(got, want):
    u, v, d = (t.cpu().numpy() if hasattr(t, "cpu") else t for t in got)
    assert u.dtype == np.int32 and v.dtype == np.int32 and d.dtype == np.float32
    assert np.array_equal(u, want[0]) and np.array_equal(v, want[1])
    assert np.array_equal(d.view(np.int32), want[2].view(np.int32))


def _components(indptr, idx, n):
    import scipy.sparse as sp
    from scipy.sparse.csgraph import connected_components
    A = sp.csr_matrix((np.ones(idx.size, np.int8), idx, indptr), shape=(n, n))   # ones: distance-0 entries count
    return connected_components(A, directed=False)[1]


def _same_partition(a, b):
    _, ia = np.unique(a, return_inverse=True)
    _, ib = np.unique(b, return_inverse=True)
    return np.unique(np.stack([ia, ib], 1), axis=0).shape[0] == ia.max() + 1 == ib.max() + 1


# ---------------------------------------------------------------- kernels
@pytest.mark.parametrize("labels", ["random", "equal", "distinct"])
@pytest.mark.parametrize("R,C,ld,node0", [(77, 301, 304, 5), (5, 37, 40, 3), (130, 130, 133, 0), (33, 1000, 1003, 9),
                                          (1, 63, 64, 2), (200, 5000, 5000, 100), (300, 300, 301, 17)])
def test_mst_panel_min_on_quantized_blocks(R, C, ld, node0, labels):
    """Few value levels (many ties), R and C not multiples of 32, node0 != 0; the lower part and the ld padding are
    poisoned with 0, which would win if read.  Some prior keys are smaller than any candidate and must stay."""
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
    want = prior.copy()
    np.minimum.at(want, node0 + rr, _key(blk[rr, cc], node0 + cc))
    np.minimum.at(want, node0 + cc, _key(blk[rr, cc], node0 + rr))
    keys = torch.from_numpy(prior).cuda()
    B = torch.from_numpy(blk).cuda()
    check(lib.hsd_mst_panel_min(B.data_ptr(), ld, R, C, node0, engine._ptr(torch.from_numpy(comp).cuda()),
                                engine._ptr(keys), engine._stream()))
    got = keys.cpu().numpy()
    assert np.array_equal(got, want)
    if labels == "equal":
        assert np.array_equal(got, prior)                       # no edge leaves the one component


@pytest.mark.parametrize("k", [1, 5, 32, 64])
def test_mst_list_candidates(k):
    """Lists ordered by (distance, id) with ties, some short (padded with -1 / +inf); a few component labels so
    that many nodes are exhausted."""
    import torch
    from hsd_b200 import engine
    from hsd_b200._lib import check, lib
    rng = np.random.default_rng(k)
    n = 700
    comp = rng.integers(0, 6, n).astype(np.int32)
    idx = np.full((n, k), -1, np.int32)
    val = np.full((n, k), np.inf, np.float32)
    for i in range(n):
        length = k if rng.random() < 0.8 else int(rng.integers(0, k + 1))
        inside = rng.random() < 0.4                         # a list drawn from its own component: exhausted
        pool = np.flatnonzero(comp == comp[i]) if inside else np.arange(n)
        js = rng.choice(pool[pool != i], length, replace=False)
        ds = rng.integers(0, 4, length).astype(np.float32) * np.float32(0.5)
        o = np.lexsort((js, ds))
        idx[i, :length], val[i, :length] = js[o], ds[o]
    want_key = np.full(n, NONE, np.int64)
    want_bound = np.full(n, np.inf, np.float32)
    for i in range(n):
        out = [t for t in range(k) if idx[i, t] >= 0 and comp[idx[i, t]] != comp[i]]
        if out:
            want_key[i] = _key(val[i, out[0]], idx[i, out[0]])
        elif idx[i, k - 1] >= 0:
            want_bound[i] = val[i, k - 1]
    keys = torch.empty(n, dtype=torch.int64, device="cuda")
    bound = torch.empty(n, dtype=torch.float32, device="cuda")
    ti, tv, tc = (torch.from_numpy(a).cuda() for a in (idx, val, comp))
    check(lib.hsd_mst_list_candidates(engine._ptr(ti), engine._ptr(tv), n, k, engine._ptr(tc), engine._ptr(keys),
                                      engine._ptr(bound), engine._stream()))
    assert np.array_equal(keys.cpu().numpy(), want_key)
    assert np.array_equal(bound.cpu().numpy(), want_bound)
    assert (want_key == NONE).sum() > 10 and (want_key != NONE).sum() > 10


# ---------------------------------------------------------------- Borůvka sweep == Kruskal on the resident matrix
@pytest.mark.parametrize("hops", [1, 2, 3, 4])
@pytest.mark.parametrize("graph", ["karate", "barbell", "europe", 2000, 10000])
def test_degree_mst_equals_kruskal(golden_graphs, graph, hops):
    from hsd_b200 import engine
    from hsd_b200.graph import powerlaw_graph
    g = _graph(golden_graphs, graph) if isinstance(graph, str) else powerlaw_graph(graph, 5, seed=1)
    dg = engine.DeviceGraph.upload(g)
    try:
        D, _ = engine.degree_distance_device(dg, hops)
    except engine.EmptyRingError:                           # a ring runs empty at this depth: both paths raise
        for cand_k in (0, 8):
            with pytest.raises(engine.EmptyRingError, match="Distribution can't be empty."):
                engine.degree_mst(dg, hops, cand_k=cand_k, panel_rows=128)
        return
    want = kruskal_resident(D)
    del D
    for p in (None, 128, 384):
        for cand_k in (0, 1, 8, 64):
            stats = {}
            got = engine.degree_mst(dg, hops, cand_k=cand_k, panel_rows=p, stats=stats)
            _assert_mst_equal(got, want)
            assert stats["rounds"] <= max(1, int(np.ceil(np.log2(g.n))))
            assert len(stats["round_ms"]) == stats["rounds"] and stats["sweeps"] == sum(stats["swept"])
            if cand_k == 0:
                assert stats["sweeps"] == stats["rounds"]
            else:
                assert not stats["swept"][0]                # round 1 is always certified


def test_degree_mst_all_distances_zero():
    """Every node of a cycle looks alike: every distance is 0 and the order E picks the star (0, j)."""
    from hsd_b200 import engine
    from hsd_b200.graph import CSRGraph
    n = 1000
    e = np.array([(i, (i + 1) % n) for i in range(n)], dtype=np.int64)
    dg = engine.DeviceGraph.upload(CSRGraph.from_edges(n, e))
    for p in (None, 128):
        for cand_k in (0, 1, 64):
            u, v, d = (t.cpu().numpy() for t in engine.degree_mst(dg, 3, cand_k=cand_k, panel_rows=p))
            assert np.array_equal(u, np.zeros(n - 1)) and np.array_equal(v, np.arange(1, n))
            assert np.array_equal(d.view(np.int32), np.zeros(n - 1, np.int32))


# ---------------------------------------------------------------- at size
def _prim_device(D):
    """Prim on the resident matrix: per-node int64 keys K(dist, u) to the tree (for a fixed outside node that is the
    order E), the global pick as in degree_mst: a minimum on (dist, lo), then on hi among the matches.  Returns
    (u, v, dist) sorted by (dist, u, v)."""
    import torch
    n, dev = D.shape[0], D.device
    node = torch.arange(n, dtype=torch.int64, device=dev)
    none = torch.full((n,), NONE, dtype=torch.int64, device=dev)
    inside = torch.zeros(n, dtype=torch.bool, device=dev)
    inside[0] = True
    key = (D[0].view(torch.int32).long() << 32) | 0
    key[0] = NONE
    eu = torch.empty(n - 1, dtype=torch.int64, device=dev)
    ev = torch.empty_like(eu)
    for t in range(n - 1):                                  # no host synchronisation inside the loop
        u = key & 0xFFFFFFFF
        k1 = torch.where(inside, none, (key >> 32) << 32 | torch.minimum(u, node))
        k2 = torch.where(k1 == k1.min(), torch.maximum(u, node), none)
        j = torch.argmin(k2).view(1)                        # the outside endpoint of the minimum edge
        uj = u.index_select(0, j)
        eu[t:t + 1].copy_(torch.minimum(uj, j))
        ev[t:t + 1].copy_(torch.maximum(uj, j))
        inside.index_fill_(0, j, True)
        row = D.index_select(0, j).squeeze(0).view(torch.int32).long() << 32 | j
        key = torch.where(inside, none, torch.minimum(key, row))
    d = D[eu, ev]
    o = np.lexsort((ev.cpu().numpy(), eu.cpu().numpy(), d.view(torch.int32).cpu().numpy()))
    return eu.int().cpu().numpy()[o], ev.int().cpu().numpy()[o], d.cpu().numpy()[o]


def test_degree_mst_100k_equals_device_prim():
    """100k nodes (BA m = 5, 2 hops): the default plan against a device Prim on the resident 40 GB matrix."""
    from hsd_b200 import engine
    from hsd_b200.graph import powerlaw_graph
    n, hops = 100000, 2
    dg = engine.DeviceGraph.upload(powerlaw_graph(n, 5, seed=0))
    stats = {}
    got = tuple(t.cpu().numpy() for t in engine.degree_mst(dg, hops, stats=stats))
    D, _ = engine.degree_distance_device(dg, hops)
    _assert_mst_equal(got, _prim_device(D))
    assert stats["rounds"] <= 17


def test_single_linkage_beyond_device_memory():
    """300k nodes, 3 hops: the float32 matrix (360 GB) exceeds the device.  The N - 1 edges form a spanning tree with
    sorted heights, and at a small radius the dendrogram's flat clusters are the radius graph's components."""
    import networkx as nx
    import torch
    from scipy.cluster.hierarchy import fcluster
    from hsd_b200.graph import powerlaw_graph
    from model import HSD
    n, hops = 300000, 3
    g = powerlaw_graph(n, 5, seed=0)
    assert 4 * n * n > torch.cuda.get_device_properties(0).total_memory
    e = np.stack([np.repeat(np.arange(n), np.diff(g.rowptr)), g.col[:g.nnz]], 1)
    G = nx.Graph()
    G.add_nodes_from(range(n))
    G.add_edges_from(map(tuple, e[e[:, 0] < e[:, 1]].tolist()))
    m = HSD(G, "pl300k", 0, hops, "wasserstein", signal="degree")
    u, v, d = m.minimum_spanning_tree()
    assert u.shape == v.shape == d.shape == (n - 1,) and np.all(u < v)
    assert np.all(np.diff(d) >= 0)
    from hsd_b200.engine import single_linkage_host
    Z = single_linkage_host(u, v, d, n)                     # refuses an edge that closes a cycle
    assert Z[-1, 3] == n
    radius = float(np.quantile(d, 0.25))
    indptr, idx, _ = m.radius_neighbors(radius)
    assert _same_partition(fcluster(Z, radius, "distance"), _components(indptr, idx, n))


# ---------------------------------------------------------------- model
@pytest.mark.parametrize("name,hop", [("karate", 2), ("europe", 3), ("barbell", 1), ("gnp8", 2)])
def test_model_single_linkage_equals_scipy(golden_graphs, name, hop):
    """The golden graphs have many equal distances: there the heights and every flat clustering must match scipy.
    gnp_random_graph(8, 0.35, seed=242) at 2 hops has 28 distinct pair distances: there Z must equal scipy's."""
    import networkx as nx
    from conftest import nx_graph
    from scipy.cluster.hierarchy import fcluster, linkage
    from scipy.spatial.distance import squareform
    from model import HSD
    G = nx.gnp_random_graph(8, 0.35, seed=242) if name == "gnp8" else nx_graph(golden_graphs, name)
    m = HSD(G, name, 0, hop, "wasserstein", signal="degree")
    D = m.structural_distance_device().cpu().numpy()
    Z = m.single_linkage()
    want = linkage(squareform(D, checks=False), "single")
    assert Z.dtype == np.float64 and Z.shape == (m.n_node - 1, 4)
    assert np.array_equal(Z[:, 2], want[:, 2])
    for h in np.unique(Z[:, 2]):
        assert _same_partition(fcluster(Z, h, "distance"), fcluster(want, h, "distance")), h
    iu = np.triu_indices(m.n_node, 1)
    tie_free = np.unique(D[iu]).size == iu[0].size
    assert tie_free == (name == "gnp8")
    if tie_free:
        assert np.array_equal(Z, want)
    u, v, d = m.minimum_spanning_tree()
    assert np.array_equal(Z[:, 2], d.astype(np.float64))


def test_model_single_linkage_cuts_are_radius_components():
    """20k nodes, 3 hops: fcluster(Z, r, "distance") is the connected components of radius_neighbors(r), at r = 0
    and the median 5-NN and 20-NN distances."""
    import networkx as nx
    from scipy.cluster.hierarchy import fcluster
    from model import HSD
    n = 20000
    G = nx.barabasi_albert_graph(n, 5, seed=3)
    m = HSD(G, "ba20k", 0, 3, "wasserstein", signal="degree")
    Z = m.single_linkage()
    _, kval = m.nearest_neighbors(20)
    for r in (0.0, float(np.median(kval[:, 4])), float(np.median(kval[:, 19]))):
        indptr, idx, _ = m.radius_neighbors(r)
        assert _same_partition(fcluster(Z, r, "distance"), _components(indptr, idx, n)), r


def test_model_mst_modes_empty_rings_and_small_graphs(golden_graphs):
    import networkx as nx
    from conftest import nx_graph
    from hsd_b200.engine import EmptyRingError
    from model import HSD
    w = HSD(nx_graph(golden_graphs, "karate"), "karate", 1.0, 2, "wasserstein")
    with pytest.raises(NotImplementedError):
        w.minimum_spanning_tree()
    with pytest.raises(NotImplementedError):
        w.single_linkage()
    G = nx.barabasi_albert_graph(300, 3, seed=2)
    G.add_nodes_from([300, 301])                            # isolated nodes: their rings run empty
    m = HSD(G, "iso", 0, 2, "wasserstein", signal="degree")
    with pytest.raises(EmptyRingError):
        m.nearest_neighbors(5)
    with pytest.raises(EmptyRingError):
        m.minimum_spanning_tree()
    with pytest.raises(EmptyRingError):
        m.single_linkage()
    m.empty = "zero"
    assert m.single_linkage().shape == (301, 4)
    for n in (1, 2):
        G = nx.path_graph(n)
        m = HSD(G, "tiny", 0, 1, "wasserstein", signal="degree")
        m.empty = "zero"
        Z = m.single_linkage()
        assert Z.shape == (n - 1, 4)
        if n == 2:
            assert np.array_equal(Z[:, [0, 1, 3]], [[0, 1, 2]])
    m = HSD(nx.Graph(), "empty", 0, 1, "wasserstein", signal="degree")
    u, v, d = m.minimum_spanning_tree()
    assert u.size == v.size == d.size == 0 and m.single_linkage().shape == (0, 4)
