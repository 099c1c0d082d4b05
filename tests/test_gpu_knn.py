"""k nearest neighbours by row panels (engine.degree_knn): the list-merge kernels against Python
sorting, and the panel sweep against the resident path — topk_rows over the full matrix — bit for bit,
on idx and on the distances."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

INF = np.float32(np.inf)


def _key(v, i):
    return (float(v), i if i >= 0 else 1 << 40)


def _sorted_list(pairs, k):
    """(val float32[k], idx int32[k]): the k first of `pairs` by (val, id), padded with +inf / -1."""
    s = sorted(pairs, key=lambda p: _key(*p))[:k]
    v = np.full(k, INF, dtype=np.float32)
    i = np.full(k, -1, dtype=np.int32)
    for t, (a, b) in enumerate(s):
        v[t], i[t] = a, b
    return v, i


def _graph(golden_graphs, name):
    from hsd_b200.graph import CSRGraph
    nodes = golden_graphs[f"{name}_nodes"]
    return CSRGraph.from_edges(len(nodes), golden_graphs[f"{name}_edges"], list(nodes))


def _resident(dg, hops, k, empty="raise"):
    from hsd_b200 import engine
    D, _ = engine.degree_distance_device(dg, hops, empty=empty)
    idx, val = engine.topk_rows(D, k)
    return idx.cpu().numpy(), val.cpu().numpy()


def _streamed(dg, hops, k, **kw):
    from hsd_b200 import engine
    idx, val = engine.degree_knn(dg, hops, k, **kw)
    return idx.cpu().numpy(), val.cpu().numpy()


def _assert_bit_equal(got, want):
    assert got[0].shape == want[0].shape and got[0].dtype == want[0].dtype == np.int32
    assert np.array_equal(got[0], want[0])
    assert np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32))


# ---------------------------------------------------------------- kernels
@pytest.mark.parametrize("n_lists", [1, 2, 3, 5, 8, 23, 64])     # 23 / 64 lists at k = 64: fewer warps per CTA
@pytest.mark.parametrize("k", [1, 7, 20, 64])
def test_topk_merge_matches_sorted(n_lists, k):
    import torch
    from hsd_b200 import engine
    rng = np.random.default_rng(100 * n_lists + k)
    n_rows, offset = 37, 1000
    cand_v = np.zeros((n_lists, n_rows, k), np.float32)
    cand_i = np.zeros((n_lists, n_rows, k), np.int32)
    run_v = np.zeros((n_rows, k), np.float32)
    run_i = np.zeros((n_rows, k), np.int32)
    want_v = np.zeros((n_rows, k), np.float32)
    want_i = np.zeros((n_rows, k), np.int32)
    for r in range(n_rows):
        # disjoint id sets per list, sizes from 0 (all padding) to 2k; values from 3 levels: big tie classes
        ids = rng.permutation(20000)
        sizes = rng.integers(0, 2 * k + 1, size=n_lists + 1)
        if r == 0:
            sizes[:] = 0
        pos, pool = 0, []
        for l in range(n_lists + 1):
            my = [(np.float32(rng.integers(0, 3) * 0.5), int(i) + offset) for i in ids[pos:pos + sizes[l]]]
            pos += sizes[l]
            pool += my
            v, i = _sorted_list(my, k)
            if l == 0:
                run_v[r], run_i[r] = v, i
            else:
                cand_v[l - 1, r], cand_i[l - 1, r] = v, np.where(i >= 0, i - offset, -1)
        want_v[r], want_i[r] = _sorted_list(pool, k)
    io_i, io_v = torch.from_numpy(run_i).cuda(), torch.from_numpy(run_v).cuda()
    engine.topk_merge(torch.from_numpy(cand_i).cuda(), torch.from_numpy(cand_v).cuda(), io_i, io_v, idx_offset=offset)
    assert np.array_equal(io_i.cpu().numpy(), want_i)
    assert np.array_equal(io_v.cpu().numpy(), want_v)


@pytest.mark.parametrize("R,n_cols,ld,c_begin,k", [(5, 300, 300, 0, 20), (130, 701, 704, 129, 7), (1000, 257, 260, 3, 64),
                                                   (300, 1000, 1001, 300, 1), (3, 50, 52, 10, 64), (77, 2000, 2000, 640, 33)])
def test_topk_merge_cols_matches_sorted(R, n_cols, ld, c_begin, k):
    """Column pass on a random quantised block (R not a power of two, ragged columns, c_begin > 0,
    R < k leaving lists partly padded); running lists partly pre-filled from disjoint ids."""
    import torch
    from hsd_b200 import engine
    rng = np.random.default_rng(R * 7 + n_cols)
    row0, col0, n_nodes = 5000, 20, 20 + n_cols + 9
    blk = np.full((R, ld), np.float32(-7.0), np.float32)                   # ld padding must never be read
    blk[:, :n_cols] = rng.integers(0, 6, size=(R, n_cols)).astype(np.float32) * 0.25
    run_v = np.full((n_nodes, k), INF, np.float32)
    run_i = np.full((n_nodes, k), -1, np.int32)
    pre = {}
    for node in range(n_nodes):
        m = int(rng.integers(0, k + 3))
        pre[node] = [(np.float32(rng.integers(0, 6) * 0.25), int(i)) for i in rng.choice(4000, m, replace=False)]
        run_v[node], run_i[node] = _sorted_list(pre[node], k)
    io_i, io_v = torch.from_numpy(run_i.copy()).cuda(), torch.from_numpy(run_v.copy()).cuda()
    engine.topk_merge_cols(torch.from_numpy(blk).cuda(), k, io_i, io_v, c_begin=c_begin, n_cols=n_cols,
                           row_node0=row0, col_node0=col0)
    got_i, got_v = io_i.cpu().numpy(), io_v.cpu().numpy()
    for node in range(n_nodes):
        c = node - col0
        if c_begin <= c < n_cols:
            wv, wi = _sorted_list(pre[node] + [(blk[r, c], row0 + r) for r in range(R)], k)
        else:                                                               # outside the column range: untouched
            wv, wi = run_v[node], run_i[node]
        assert np.array_equal(got_i[node], wi), node
        assert np.array_equal(got_v[node], wv), node


# ---------------------------------------------------------------- panel sweep == resident path
GRAPHS = ["karate", "barbell", "europe", 100, 130, 1000, 4099, 20000]


@pytest.mark.parametrize("hops", [1, 2, 3, 4])
@pytest.mark.parametrize("graph", GRAPHS)
def test_degree_knn_bit_equal_to_resident(golden_graphs, graph, hops):
    from hsd_b200 import engine
    from hsd_b200.graph import powerlaw_graph
    g = _graph(golden_graphs, graph) if isinstance(graph, str) else powerlaw_graph(graph, 5, seed=0)
    dg = engine.DeviceGraph.upload(g)
    try:
        _resident(dg, hops, 1)
    except engine.EmptyRingError:                           # a ring runs empty at this depth: both paths raise
        with pytest.raises(engine.EmptyRingError, match="Distribution can't be empty."):
            engine.degree_knn(dg, hops, 1, panel_rows=128)
        return
    for k in (1, 7, 20, 64):                                # k > N - 1 for karate (34 nodes) at 64
        want = _resident(dg, hops, k)
        for p in (128, 256, 1024, g.n, None):               # None: the default budget (one panel here)
            if p is not None and p < g.n and (g.n + p - 1) // p > 40 and k not in (1, 20):
                continue                                    # many-panel sweeps of the 20k graph: two k suffice
            _assert_bit_equal(_streamed(dg, hops, k, panel_rows=p), want)


@pytest.mark.parametrize("shape", ["cycle", "torus"])
def test_degree_knn_vertex_transitive_ties_cut_by_id(shape):
    """Every node looks alike: every distance is 0 and the k nearest are the k lowest other ids."""
    from hsd_b200 import engine
    from hsd_b200.graph import CSRGraph
    if shape == "cycle":
        n = 1000
        e = np.array([(i, (i + 1) % n) for i in range(n)], dtype=np.int64)
    else:
        s = 40
        n = s * s
        e = np.array([(r * s + c, r * s + (c + 1) % s) for r in range(s) for c in range(s)] +
                     [(r * s + c, ((r + 1) % s) * s + c) for r in range(s) for c in range(s)], dtype=np.int64)
    dg = engine.DeviceGraph.upload(CSRGraph.from_edges(n, e))
    for k in (7, 64):
        want = _resident(dg, 3, k)
        assert np.all(want[1] == 0)
        exp = np.array([[j for j in range(k + 1) if j != i][:k] for i in range(n)], dtype=np.int32)
        assert np.array_equal(want[0], exp)
        for p in (128, 384):
            _assert_bit_equal(_streamed(dg, 3, k, panel_rows=p), want)


def test_degree_knn_empty_rings():
    from hsd_b200 import engine
    from hsd_b200.graph import CSRGraph, powerlaw_graph
    base = powerlaw_graph(500, 3, seed=1)
    e = np.stack([np.repeat(np.arange(base.n), np.diff(base.rowptr)), base.col[:base.nnz]], 1)
    e = e[e[:, 0] < e[:, 1]]
    g = CSRGraph.from_edges(base.n + 3, e)                      # three isolated nodes: empty rings
    dgz = engine.DeviceGraph.upload(g, include_zero=True)
    for k in (5, 20):
        want = _resident(dgz, 2, k, empty="zero")
        for p in (128, 256):
            _assert_bit_equal(_streamed(dgz, 2, k, panel_rows=p, empty="zero"), want)
    dg = engine.DeviceGraph.upload(g)
    with pytest.raises(engine.EmptyRingError, match="Distribution can't be empty."):
        engine.degree_knn(dg, 2, 5, panel_rows=128)
    with pytest.raises(engine.EmptyRingError):
        engine.degree_knn(dg, 2, 5)


@pytest.mark.parametrize("world", [2, 3, 8])
def test_degree_knn_emulated_ranks_merge_to_one_gpu(world):
    """Each rank sweeps its dealt panels into its own lists; merging the ranks' lists gives the
    one-GPU result bit for bit (what the all-gather + hsd_topk_merge of a multi-GPU run computes)."""
    import torch
    from hsd_b200 import engine
    from hsd_b200.graph import powerlaw_graph
    dg = engine.DeviceGraph.upload(powerlaw_graph(4099, 5, seed=0))
    k = 20
    single = _streamed(dg, 3, k)
    for p in (256, None):
        parts = [engine.degree_knn(dg, 3, k, panel_rows=p, rank=r, world=world) for r in range(world)]
        idx = torch.full((dg.n, k), -1, dtype=torch.int32, device="cuda")
        val = torch.full((dg.n, k), float("inf"), dtype=torch.float32, device="cuda")
        engine.topk_merge(torch.stack([a for a, _ in parts]), torch.stack([b for _, b in parts]), idx, val)
        _assert_bit_equal((idx.cpu().numpy(), val.cpu().numpy()), single)


def test_model_nearest_neighbors_streamed_equals_default(golden_graphs):
    from conftest import nx_graph
    from model import HSD
    g = nx_graph(golden_graphs, "europe")
    m = HSD(g, "europe", 0, 3, "wasserstein", signal="degree")
    n4 = (m.n_node + 3) // 4 * 4
    want = m.nearest_neighbors(10)
    got = m.nearest_neighbors(10, block_bytes=128 * n4 * 4)     # one 128-row panel at a time
    _assert_bit_equal(got, want)
    D = m.calculate_structural_distance(0.0).astype(np.float32)
    for r in (0, 100, 398):
        assert want[0][r].tolist() == sorted((j for j in range(m.n_node) if j != r), key=lambda j: (D[r, j], j))[:10]


# ---------------------------------------------------------------- at size
def test_degree_knn_c3_forced_panels_equal_resident():
    """C3 (100k nodes, 4 hops), k = 20: the resident result first (40 GB matrix, freed), then 8192-row panels."""
    import torch
    from hsd_b200 import engine
    from hsd_b200.graph import powerlaw_graph
    dg = engine.DeviceGraph.upload(powerlaw_graph(100000, 5, seed=0))
    want = _resident(dg, 4, 20)
    torch.cuda.empty_cache()
    _assert_bit_equal(_streamed(dg, 4, 20, panel_rows=8192), want)


def test_nearest_neighbors_beyond_device_memory():
    """300k nodes, 3 hops: the float32 matrix is 360 GB, twice the device.  The model API sweeps it in
    panels; 64 sampled nodes are checked against pairwise_l1 over their aligned 4-row groups + topk_rows."""
    import networkx as nx
    import torch
    from hsd_b200 import engine
    from hsd_b200.graph import powerlaw_graph
    from model import HSD
    n, hops, k = 300000, 3, 20
    g = powerlaw_graph(n, 5, seed=0)
    assert 4 * n * n > torch.cuda.get_device_properties(0).total_memory
    e = np.stack([np.repeat(np.arange(n), np.diff(g.rowptr)), g.col[:g.nnz]], 1)
    G = nx.Graph()
    G.add_nodes_from(range(n))
    G.add_edges_from(map(tuple, e[e[:, 0] < e[:, 1]].tolist()))
    m = HSD(G, "pl300k", 0, hops, "wasserstein", signal="degree")
    idx, val = m.nearest_neighbors(k)
    assert idx.shape == (n, k) and np.all(idx >= 0) and np.all(np.diff(val, axis=1) >= 0)
    dg = m._device_graph()
    sig, _, _, _ = engine.ring_signature_degree(dg, hops)
    sigT = engine.alloc_signature_table(dg.k_used(hops), n, sig.device)
    engine.signature_transpose(sig, dg.k_used(hops), sigT, 0)
    for i in np.random.default_rng(0).choice(n, 64, replace=False).tolist():
        g0 = i // 4 * 4
        rows = min(4, n - g0)
        D = engine.pairwise_l1(sigT, n, g0, rows, 0, n, symmetric=False, k_used=dg.k_used(hops))
        ri, rv = engine.topk_rows(D, k, self_col0=g0)
        assert np.array_equal(idx[i], ri[i - g0].cpu().numpy()), i
        assert np.array_equal(val[i].view(np.uint32), rv[i - g0].cpu().numpy().view(np.uint32)), i


def test_model_nearest_neighbors_sharded_needs_a_process_group(golden_graphs):
    """Without torch.distributed a rank could only return its partial lists: the public method refuses."""
    import torch.distributed as dist
    from conftest import nx_graph
    from model import HSD
    assert not dist.is_initialized()
    m = HSD(nx_graph(golden_graphs, "europe"), "europe", 0, 3, "wasserstein", signal="degree")
    with pytest.raises(RuntimeError, match="process group"):
        m.nearest_neighbors_sharded(10, 0, 2)
    _assert_bit_equal(m.nearest_neighbors_sharded(10, 0, 1), m.nearest_neighbors(10))
