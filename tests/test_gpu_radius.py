"""Radius graph (engine.degree_radius, HSD.radius_neighbors): the hsd_radius_* kernels on random blocks, and the
panel sweep against the resident matrix — mask = D.double() <= radius with the diagonal cleared, row-major
nonzero — on indptr, indices and the distance bits."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _graph(golden_graphs, name):
    from hsd_b200.graph import CSRGraph
    nodes = golden_graphs[f"{name}_nodes"]
    return CSRGraph.from_edges(len(nodes), golden_graphs[f"{name}_edges"], list(nodes))


def _oracle(D, radius, row0=0):
    """(counts int64[rows], indices int32, dist) of rows row0 + r of D[rows][N] (a row block of the matrix)."""
    import torch
    mask = D.double() <= radius
    r = torch.arange(D.shape[0], device=D.device)
    mask[r, row0 + r] = False
    nz = mask.nonzero()
    counts = torch.bincount(nz[:, 0], minlength=D.shape[0])
    return counts, nz[:, 1].int(), D[mask]


def _assert_csr_equal(got, D, radius):
    """got (indptr, idx, dist) device tensors == the oracle over the whole resident D."""
    import torch
    indptr, idx, dist = got
    want_cnt, want_idx, want_val = _oracle(D, radius)
    assert indptr.dtype == torch.int64 and idx.dtype == torch.int32 and dist.dtype == D.dtype
    assert int(indptr[0]) == 0 and indptr.numel() == D.shape[0] + 1
    assert torch.equal(indptr.diff(), want_cnt)
    assert torch.equal(idx, want_idx)
    ibits = torch.int32 if D.dtype == torch.float32 else torch.int64
    assert torch.equal(dist.view(ibits), want_val.view(ibits))


def _assert_symmetric(indptr, idx, dist):
    """(i, j, d) present iff (j, i, d), same bits; no self pairs; rows ascending."""
    import scipy.sparse as sp
    indptr, idx, dist = (t.cpu().numpy() if hasattr(t, "cpu") else t for t in (indptr, idx, dist))
    n = indptr.size - 1
    rows = np.repeat(np.arange(n), np.diff(indptr))
    assert not np.any(rows == idx)
    bits = dist.view(np.int32 if dist.dtype == np.float32 else np.int64)
    a, b = np.lexsort((idx, rows)), np.lexsort((rows, idx))
    assert np.array_equal(rows[a], idx[b]) and np.array_equal(idx[a], rows[b]) and np.array_equal(bits[a], bits[b])
    assert np.all(np.diff(idx)[rows[1:] == rows[:-1]] > 0)
    m = sp.csr_matrix((dist, idx, indptr), shape=(n, n))
    assert m.nnz == idx.size and m.has_canonical_format


def _knn_radii(D, small):
    """0, the median over nodes of the 5th- and 20th-NN distance, and +inf on small graphs."""
    import torch
    from hsd_b200 import engine
    _, val = engine.topk_rows(D, 20)
    radii = [0.0]
    for k in (5, 20):
        v = val[:, k - 1]
        v = v[torch.isfinite(v)]
        if v.numel():
            radii.append(float(v.median()))
    if small:
        radii.append(math.inf)
    return radii


# ---------------------------------------------------------------- kernels
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("R,C,ld,r0", [(77, 301, 304, 0), (5, 37, 40, 0), (130, 130, 133, 0), (33, 1000, 1003, 9),
                                       (1, 63, 64, 0), (200, 5000, 5000, 100), (1300, 1500, 1500, 0)])
def test_radius_kernels_on_quantized_blocks(R, C, ld, r0, dtype):
    """One panel through count / emit / scatter: a few value levels so that many entries equal the radius,
    R and C not multiples of 32, the ld padding and the unread lower part poisoned with a would-be hit."""
    import torch
    from hsd_b200 import engine
    rng = np.random.default_rng(R * 31 + C)
    np_dt = np.float32 if dtype == "float32" else np.float64
    blk = np.zeros((R, ld), np_dt)                               # 0 <= any radius: padding / lower part must not count
    up = np.triu(np.ones((R, C), bool), 1)
    vals = rng.integers(0, 5, size=(R, C)).astype(np_dt) * np_dt(0.25) + np_dt(0.25)
    blk[:, :C][up] = vals[up]
    n = r0 + C
    for radius in (0.5, 0.0, 0.25, 1.25, math.inf, 0.5 + 1e-12, 0.5 - 1e-12):
        rr, cc_ = np.nonzero(up & (blk[:, :C].astype(np.float64) <= radius))
        ii = np.concatenate([r0 + rr, r0 + cc_])                  # every hit, and its mirror
        jj = np.concatenate([r0 + cc_, r0 + rr])
        vv = np.concatenate([blk[rr, cc_], blk[rr, cc_]])
        o = np.lexsort((jj, ii))
        sweep = engine._RadiusSweep(n, getattr(torch, dtype), radius, 10 ** 9, torch.device("cuda"))
        hits = torch.empty(R * ((C + 31) // 32), dtype=torch.int32, device="cuda")
        rc = torch.empty(R, dtype=torch.int32, device="cuda")
        cc = torch.empty(C * -(-R // engine.RADIUS_CHUNK_ROWS), dtype=torch.int32, device="cuda")
        B = torch.from_numpy(blk).cuda()
        assert sweep.panel(B, ld, R, C, r0, hits, rc, cc, engine._stream())
        indptr, idx, val = (t.cpu().numpy() for t in sweep.assemble())
        assert np.array_equal(np.diff(indptr), np.bincount(ii, minlength=n)), radius
        assert np.array_equal(idx, jj[o].astype(np.int32)), radius
        assert val.dtype == np_dt and np.array_equal(val, vv[o]), radius
        _assert_symmetric(indptr, idx, val)


# ---------------------------------------------------------------- panel sweep == resident matrix
GRAPHS = ["karate", "barbell", "europe", 100, 130, 1000, 4099, 20000]


@pytest.mark.parametrize("hops", [1, 2, 3, 4])
@pytest.mark.parametrize("graph", GRAPHS)
def test_degree_radius_equals_resident(golden_graphs, graph, hops):
    from hsd_b200 import engine
    from hsd_b200.graph import powerlaw_graph
    g = _graph(golden_graphs, graph) if isinstance(graph, str) else powerlaw_graph(graph, 5, seed=0)
    dg = engine.DeviceGraph.upload(g)
    try:
        D, _ = engine.degree_distance_device(dg, hops)
    except engine.EmptyRingError:                           # a ring runs empty at this depth: both paths raise
        with pytest.raises(engine.EmptyRingError, match="Distribution can't be empty."):
            engine.degree_radius(dg, hops, 1.0, panel_rows=128)
        return
    for radius in _knn_radii(D, g.n <= 4099):
        for p in (128, 256, 1024, g.n, None):               # None: the default budget (one panel here)
            if p is not None and p < g.n and (g.n + p - 1) // p > 40 and radius not in (0.0,) and p != 128:
                continue                                    # many-panel sweeps of the 20k graph: 128 rows suffice
            got = engine.degree_radius(dg, hops, radius, panel_rows=p)
            _assert_csr_equal(got, D, radius)
            if g.n <= 1000:
                _assert_symmetric(*got)


@pytest.mark.parametrize("shape", ["cycle", "torus"])
def test_degree_radius_all_zero_distances_and_the_cap(shape):
    """Every node looks alike: every distance is 0, radius 0 lists all N (N - 1) ordered pairs.  A smaller
    max_pairs raises, leaves no device memory behind, and the next call works."""
    import torch
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
    D, _ = engine.degree_distance_device(dg, 3)
    assert bool((D == 0).all())
    for p in (128, 384, None):
        indptr, idx, dist = engine.degree_radius(dg, 3, 0.0, panel_rows=p)
        assert idx.numel() == n * (n - 1) and bool((dist == 0).all())
        _assert_csr_equal((indptr, idx, dist), D, 0.0)
    del indptr, idx, dist, D
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    for p, cap in ((128, n * (n - 1) - 1), (384, 1000), (None, 0)):
        with pytest.raises(ValueError, match="max_pairs") as ei:
            engine.degree_radius(dg, 3, 0.0, panel_rows=p, max_pairs=cap)
        assert str(cap) in str(ei.value) and "radius 0.0" in str(ei.value)
        assert torch.cuda.memory_allocated() == before      # the call's buffers are gone, traceback alive or not
    indptr, idx, _ = engine.degree_radius(dg, 3, 0.0, panel_rows=128, max_pairs=n * (n - 1))
    assert idx.numel() == n * (n - 1)


def test_degree_radius_empty_rings():
    from hsd_b200 import engine
    from hsd_b200.graph import CSRGraph, powerlaw_graph
    base = powerlaw_graph(500, 3, seed=1)
    e = np.stack([np.repeat(np.arange(base.n), np.diff(base.rowptr)), base.col[:base.nnz]], 1)
    e = e[e[:, 0] < e[:, 1]]
    g = CSRGraph.from_edges(base.n + 3, e)                      # three isolated nodes: empty rings
    dgz = engine.DeviceGraph.upload(g, include_zero=True)
    D, _ = engine.degree_distance_device(dgz, 2, empty="zero")
    for radius in _knn_radii(D, True):
        for p in (128, 256, None):
            _assert_csr_equal(engine.degree_radius(dgz, 2, radius, panel_rows=p, empty="zero"), D, radius)
    dg = engine.DeviceGraph.upload(g)
    with pytest.raises(engine.EmptyRingError, match="Distribution can't be empty."):
        engine.degree_radius(dg, 2, 1.0, panel_rows=128)
    with pytest.raises(engine.EmptyRingError):
        engine.degree_radius(dg, 2, 1.0)


def test_model_radius_neighbors_degree(golden_graphs):
    """The public API: numpy CSR, scipy-canonical, bad radii refused, and rows holding the k-NN ids when the
    radius is a node's k-th NN distance."""
    import scipy.sparse as sp
    from conftest import nx_graph
    from model import HSD
    g = nx_graph(golden_graphs, "europe")
    m = HSD(g, "europe", 0, 3, "wasserstein", signal="degree")
    for bad in (math.nan, -0.5):
        with pytest.raises(ValueError, match="radius"):
            m.radius_neighbors(bad)
    D = m.calculate_structural_distance(0.0).astype(np.float32)
    kidx, kval = m.nearest_neighbors(10)
    for i in (0, 100, 398):
        for k in (1, 5, 10):
            indptr, idx, dist = m.radius_neighbors(float(kval[i, k - 1]))
            assert indptr.dtype == np.int64 and idx.dtype == np.int32 and dist.dtype == np.float32
            row = set(idx[indptr[i]:indptr[i + 1]].tolist())
            assert set(kidx[i, :k].tolist()) <= row
            assert row == {j for j in range(m.n_node) if j != i and D[i, j] <= kval[i, k - 1]}
    n4 = (m.n_node + 3) // 4 * 4
    r = float(np.median(kval[:, 4]))
    a = m.radius_neighbors(r)
    b = m.radius_neighbors(r, block_bytes=128 * n4 * 4)          # 128-row panels
    for x, y in zip(a, b):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
    M = sp.csr_matrix((a[2], a[1], a[0]), shape=(m.n_node, m.n_node))
    assert M.nnz == a[1].size and M.has_canonical_format
    assert np.array_equal(M.toarray() != 0, (D <= r) & (D != 0) & ~np.eye(m.n_node, dtype=bool))


@pytest.mark.parametrize("name", ["karate", "europe"])
def test_model_radius_neighbors_wavelet(golden_graphs, name):
    """Wavelet mode thresholds the resident float64 matrix with the double kernels."""
    import torch
    from conftest import nx_graph
    from model import HSD
    m = HSD(nx_graph(golden_graphs, name), name, 1.0, 2, "wasserstein")
    m.init()
    D = m.structural_distance_device(1.0)
    assert D.dtype == torch.float64 and torch.equal(D, D.T)
    for radius in _knn_radii(D.float(), True) + [float(D[0, 1])]:
        got = m.radius_neighbors(radius, scale=1.0)
        assert got[2].dtype == np.float64
        _assert_csr_equal(tuple(torch.from_numpy(t).cuda() for t in got), D, radius)
        _assert_symmetric(*got)
    with pytest.raises(ValueError, match="max_pairs"):
        m.radius_neighbors(math.inf, scale=1.0, max_pairs=10)
    assert m.radius_neighbors(math.inf, scale=1.0)[1].size == m.n_node * (m.n_node - 1)


# ---------------------------------------------------------------- at size
def test_degree_radius_c3_forced_panels_equal_resident():
    """C3 (100k nodes, 4 hops): 8192-row panels against the resident 40 GB matrix, checked in row blocks."""
    import torch
    from hsd_b200 import engine
    from hsd_b200.graph import powerlaw_graph
    n, hops = 100000, 4
    dg = engine.DeviceGraph.upload(powerlaw_graph(n, 5, seed=0))
    _, val = engine.degree_knn(dg, hops, 20)
    radius = float(val[:, 19].median())
    indptr, idx, dist = engine.degree_radius(dg, hops, radius, panel_rows=8192)
    D, _ = engine.degree_distance_device(dg, hops)
    for b0 in range(0, n, 8192):
        b1 = min(b0 + 8192, n)
        cnt, wi, wv = _oracle(D[b0:b1], radius, row0=b0)
        s, e = int(indptr[b0]), int(indptr[b1])
        assert torch.equal(indptr[b0:b1 + 1].diff(), cnt)
        assert torch.equal(idx[s:e], wi)
        assert torch.equal(dist[s:e].view(torch.int32), wv.view(torch.int32))
    assert 10 * n <= idx.numel()                             # about 20 per node at the median 20th-NN distance


def test_radius_neighbors_beyond_device_memory():
    """300k nodes, 3 hops: the float32 matrix (360 GB) exceeds the device.  64 sampled nodes are checked
    against pairwise_l1 over their aligned 4-row groups."""
    import networkx as nx
    import torch
    from hsd_b200 import engine
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
    _, kval = m.nearest_neighbors(20)
    radius = float(np.median(kval[:, 19]))
    indptr, idx, dist = m.radius_neighbors(radius)
    assert indptr.shape == (n + 1,) and idx.size == indptr[-1] and dist.dtype == np.float32
    dg = m._device_graph()
    sig, _, _, _ = engine.ring_signature_degree(dg, hops)
    sigT = engine.alloc_signature_table(dg.k_used(hops), n, sig.device)
    engine.signature_transpose(sig, dg.k_used(hops), sigT, 0)
    for i in np.random.default_rng(0).choice(n, 64, replace=False).tolist():
        g0 = i // 4 * 4
        rows = min(4, n - g0)
        D = engine.pairwise_l1(sigT, n, g0, rows, 0, n, symmetric=False, k_used=dg.k_used(hops))
        cnt, wi, wv = _oracle(D, radius, row0=g0)
        off = int(cnt[:i - g0].sum())
        k = int(cnt[i - g0])
        assert indptr[i + 1] - indptr[i] == k, i
        assert np.array_equal(idx[indptr[i]:indptr[i + 1]], wi[off:off + k].cpu().numpy()), i
        assert np.array_equal(dist[indptr[i]:indptr[i + 1]].view(np.uint32),
                              wv[off:off + k].cpu().numpy().view(np.uint32)), i
