"""Radius graph over several ranks (engine.degree_radius with world > 1, engine.radius_merge,
HSD.radius_neighbors_sharded): hsd_radius_merge_parts against a numpy stable merge, and ranks emulated in one
process — each sweeps its dealt panels into a partial CSR, and merging the partials must give the one-GPU
graph bit for bit (what the gather + merge of a multi-GPU run computes)."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------- the merge kernel
def _random_parts(rng, n_parts, n_rows, hub_row, dup):
    """n_parts CSRs over n_rows rows: about a third of the parts after the first empty, every tenth row empty in
    all parts, row `hub_row` holding thousands of entries in the first part and in about half of the others;
    ids of a row disjoint across parts unless `dup`."""
    parts = []
    for p in range(n_parts):
        indptr = np.zeros(n_rows + 1, np.int64)
        ids = []
        empty = p > 0 and rng.random() < 0.3
        for i in range(n_rows):
            k = 0 if empty or i % 10 == 1 or rng.random() < 0.4 else int(rng.integers(1, 12))
            if i == hub_row and not empty and (p == 0 or rng.random() < 0.5):
                k = int(rng.integers(1000, 4000))
            if dup:          # a small id range: the same id lands in several parts' rows
                row = np.sort(rng.choice(5000, size=k, replace=False))
            else:            # id classes by part: disjoint across parts
                row = np.sort(rng.choice(1 << 16, size=k, replace=False)) * n_parts + p
            ids.append(row)
            indptr[i + 1] = indptr[i] + k
        parts.append((indptr, np.concatenate(ids).astype(np.int32)))
    return parts


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("dup", [False, True])
@pytest.mark.parametrize("n_parts", [1, 2, 3, 8, 64])
def test_radius_merge_parts_stable_merge(n_parts, dup, dtype):
    """Parts placed with gaps in one buffer (part_base), output at an offset inside garbage-filled padding that
    must survive; each row of the result is the numpy stable merge by id (ties by part index)."""
    import torch
    from hsd_b200 import engine
    from hsd_b200._lib import check, lib
    rng = np.random.default_rng(n_parts * 7 + dup)
    n_rows = 64 if n_parts == 64 else 300
    parts = _random_parts(rng, n_parts, n_rows, hub_row=n_rows // 3, dup=dup)
    np_dt = np.dtype(dtype)
    ibits = np.int32 if np_dt.itemsize == 4 else np.int64
    vals = [rng.integers(-2 ** 30, 2 ** 30, size=ix.size).astype(ibits).view(np_dt) for _, ix in parts]
    gap = 17
    base, pos = [], 0
    for _, ix in parts:
        pos += gap
        base.append(pos)
        pos += ix.size
    idx_buf = np.full(pos + gap, -7, np.int32)
    val_buf = np.full(pos + gap, -9, ibits).view(np_dt)
    for b, (_, ix), v in zip(base, parts, vals):
        idx_buf[b:b + ix.size] = ix
        val_buf[b:b + ix.size] = v
    lens = sum(np.diff(ip) for ip, _ in parts)
    off = 5                                                   # the merged offsets need not start at 0
    indptr = off + np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    total = int(lens.sum())
    pad = 23
    out_idx = torch.full((total + off + pad,), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
    out_val = torch.full((total + off + pad,), -3, dtype=torch.int32 if ibits == np.int32 else torch.int64,
                         device="cuda")
    ins = [torch.from_numpy(np.ascontiguousarray(a)).cuda()        # kept alive until the launch has run
           for a in (np.stack([ip for ip, _ in parts]), np.array(base, np.int64), idx_buf, val_buf.view(ibits), indptr)]
    check(lib.hsd_radius_merge_parts(n_parts, n_rows, *(engine._ptr(t) for t in ins[:4]), np_dt.itemsize,
                                     engine._ptr(ins[4]), engine._ptr(out_idx), engine._ptr(out_val),
                                     engine._stream()))
    got_i, got_v = out_idx.cpu().numpy(), out_val.cpu().numpy()
    assert np.all(got_i[:off] == 0x5A5A5A5A) and np.all(got_i[off + total:] == 0x5A5A5A5A)
    assert np.all(got_v[:off] == -3) and np.all(got_v[off + total:] == -3)
    for i in range(n_rows):
        ids = np.concatenate([ix[ip[i]:ip[i + 1]] for ip, ix in parts])
        vv = np.concatenate([v[ip[i]:ip[i + 1]] for (ip, _), v in zip(parts, vals)]).view(ibits)
        o = np.argsort(ids, kind="stable")                    # concatenated in part order: ties keep the part order
        s, e = indptr[i], indptr[i + 1]
        assert np.array_equal(got_i[s:e], ids[o]), i
        assert np.array_equal(got_v[s:e], vv[o]), i
    assert lens[n_rows // 3] >= 1000 and np.any(lens == 0)


# ---------------------------------------------------------------- emulated ranks == one GPU
def _graph(golden_graphs, name):
    from hsd_b200.graph import CSRGraph, powerlaw_graph
    if isinstance(name, int):
        return powerlaw_graph(name, 5, seed=0)
    nodes = golden_graphs[f"{name}_nodes"]
    return CSRGraph.from_edges(len(nodes), golden_graphs[f"{name}_edges"], list(nodes))


def _bit_equal(a, b):
    import torch
    return (torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
            and torch.equal(a[2].view(torch.int32), b[2].view(torch.int32)))


def _check_partials(parts, n):
    """Each partial is a valid CSR over all n rows (from 0, monotone, ids in range, no self pair, rows strictly
    ascending); the union of the partials holds no (i, j) twice."""
    import torch
    keys = []
    for indptr, idx, dist in parts:
        assert indptr.dtype == torch.int64 and indptr.numel() == n + 1 and int(indptr[0]) == 0
        assert bool((indptr.diff() >= 0).all()) and int(indptr[-1]) == idx.numel() == dist.numel()
        rows = torch.repeat_interleave(torch.arange(n, device=idx.device), indptr.diff())
        assert bool(((idx >= 0) & (idx < n) & (idx != rows)).all())
        same = rows[1:] == rows[:-1]
        assert bool((idx[1:][same] > idx[:-1][same]).all())
        keys.append(rows * n + idx)
    keys = torch.cat(keys)
    assert torch.unique(keys).numel() == keys.numel()


@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("graph", ["karate", "barbell", "europe", 4099])
def test_emulated_ranks_merge_to_one_gpu(golden_graphs, graph, world):
    """radius_merge of the ranks' partials == one-GPU degree_radius bit for bit, with forced 256-row panels and
    with the default plan (panels capped for `world` ranks).  The small graphs have fewer panels than ranks,
    so some ranks have nothing to sweep."""
    from hsd_b200 import engine
    g = _graph(golden_graphs, graph)
    hops = 3 if isinstance(graph, int) else 2
    dg = engine.DeviceGraph.upload(g)
    try:
        single = engine.degree_radius(dg, hops, 0.0)
    except engine.EmptyRingError:
        pytest.skip("a ring runs empty at this depth")
    _, kval = engine.degree_knn(dg, hops, 5)
    for radius in (0.0, float(kval[:, 4].median()), math.inf):
        single = engine.degree_radius(dg, hops, radius)
        for p in (256, None):
            parts = [engine.degree_radius(dg, hops, radius, panel_rows=p, rank=r, world=world) for r in range(world)]
            _check_partials(parts, g.n)
            assert _bit_equal(engine.radius_merge(parts), single), (radius, p)
    if g.n > 256:        # at radius +inf (the last) every panel has entries: each rank that swept one holds some
        assert sum(parts[r][1].numel() > 0 for r in range(world)) > 1      # the work really was split


def test_emulated_ranks_cap_and_arguments():
    """A partial past max_pairs raises like one GPU does; rank must be in 0..world-1; radius_merge takes
    1..64 parts of one shape."""
    import torch
    from hsd_b200 import engine
    from hsd_b200.graph import powerlaw_graph
    dg = engine.DeviceGraph.upload(powerlaw_graph(1000, 5, seed=0))
    with pytest.raises(ValueError, match="max_pairs = 10"):
        engine.degree_radius(dg, 2, math.inf, panel_rows=128, rank=1, world=2, max_pairs=10)
    with pytest.raises(ValueError, match="rank"):
        engine.degree_radius(dg, 2, 1.0, rank=2, world=2)
    with pytest.raises(ValueError, match="1..64"):
        engine.radius_merge([])
    a = engine.degree_radius(dg, 2, 0.0)
    with pytest.raises(ValueError, match="parts"):
        engine.radius_merge([a, (a[0][:-1], a[1], a[2])])
    assert _bit_equal(engine.radius_merge([a]), a)
    empty = (torch.zeros(dg.n + 1, dtype=torch.int64, device="cuda"), a[1][:0], a[2][:0])
    assert _bit_equal(engine.radius_merge([empty, a, empty]), a)


def test_model_radius_neighbors_sharded(golden_graphs):
    """world = 1 is radius_neighbors; world > 1 needs a process group; bad rank / mode refused."""
    import torch.distributed as dist
    from conftest import nx_graph
    from model import HSD
    assert not dist.is_initialized()
    m = HSD(nx_graph(golden_graphs, "europe"), "europe", 0, 3, "wasserstein", signal="degree")
    _, kval = m.nearest_neighbors(10)
    for r in (0.0, float(np.median(kval[:, 4])), math.inf):
        got, want = m.radius_neighbors_sharded(r, 0, 1), m.radius_neighbors(r)
        for x, y in zip(got, want):
            assert x.dtype == y.dtype and np.array_equal(x.view(np.uint8), y.view(np.uint8))
    with pytest.raises(RuntimeError, match="process group"):
        m.radius_neighbors_sharded(1.0, 0, 2)
    with pytest.raises(ValueError, match="rank"):
        m.radius_neighbors_sharded(1.0, 1, 1)
    with pytest.raises(ValueError, match="radius"):
        m.radius_neighbors_sharded(-1.0, 0, 1)
    w = HSD(nx_graph(golden_graphs, "karate"), "karate", 1.0, 2, "wasserstein")
    with pytest.raises(NotImplementedError):
        w.radius_neighbors_sharded(1.0, 0, 1)


# ---------------------------------------------------------------- at size
def test_emulated_ranks_c3_forced_panels_equal_one_gpu():
    """C3 (100k nodes, 4 hops), radius = median 20th-NN distance: 8 emulated ranks over 4096-row panels, merged,
    equal the one-GPU sweep with its default plan bit for bit."""
    import torch
    from hsd_b200 import engine
    from hsd_b200.graph import powerlaw_graph
    n, hops, world = 100000, 4, 8
    dg = engine.DeviceGraph.upload(powerlaw_graph(n, 5, seed=0))
    _, val = engine.degree_knn(dg, hops, 20)
    radius = float(val[:, 19].median())
    del val
    single = engine.degree_radius(dg, hops, radius)
    parts = [engine.degree_radius(dg, hops, radius, panel_rows=4096, rank=r, world=world) for r in range(world)]
    _check_partials(parts, n)
    assert all(p[1].numel() for p in parts)
    assert _bit_equal(engine.radius_merge(parts), single)
    assert 10 * n <= single[1].numel()
    torch.cuda.empty_cache()
