"""Parity of the degree-mode hot path (BFS rings -> degree CDF -> pairwise L1)
against the oracle (scipy W1 over degree multisets of the reference's rings)."""
import numpy as np
import pytest

from oracle import hsd_oracle as O

pytestmark = pytest.mark.gpu


def _graph(golden_graphs, name):
    from hsd_b200.graph import CSRGraph
    nodes = golden_graphs[f"{name}_nodes"]
    return CSRGraph.from_edges(len(nodes), golden_graphs[f"{name}_edges"], list(nodes))


def _oracle_adj(g):
    return [g.neighbors(i).astype(np.int64) for i in range(g.n)]


def _rings_from_bitmaps(bitmaps, orig_of, n):
    """uint32 bitmaps [rows, H+1, words] in degree-order ids -> sorted original-id lists."""
    bm = bitmaps.view(np.uint32)
    bits = np.unpackbits(bm.view(np.uint8), axis=-1, bitorder="little")[..., :n]
    out = []
    for r in range(bits.shape[0]):
        out.append([sorted(orig_of[np.nonzero(bits[r, h])[0]].tolist()) for h in range(bits.shape[1])])
    return out


@pytest.mark.parametrize("name,hops", [("karate", 3), ("barbell", 2), ("mkarate", 3), ("tree", 4), ("europe", 3)])
def test_rings_match_reference_bfs(golden_graphs, name, hops):
    import torch
    from hsd_b200 import engine
    g = _graph(golden_graphs, name)
    dg = engine.DeviceGraph.upload(g)
    _, sizes, bitmaps, _ = engine.ring_signature_degree(dg, hops, want_sig=False, want_bitmaps=True)
    torch.cuda.synchronize()
    rings = _rings_from_bitmaps(bitmaps.cpu().numpy(), g.degree_order().orig_of, g.n)
    ref = O.all_rings(_oracle_adj(g), hops)
    for i in range(g.n):
        assert rings[i] == ref[i], f"ring mismatch at node {i}"
        assert sizes[i].tolist() == [len(l) for l in ref[i]]


def test_ring_sizes_match_reference_run(golden_graphs, golden_runs):
    import torch
    from hsd_b200 import engine
    for name in ["karate", "europe", "usa"]:
        g = _graph(golden_graphs, name)
        hop = int(golden_runs[f"{name}_hop"])
        dg = engine.DeviceGraph.upload(g)
        _, sizes, _, _ = engine.ring_signature_degree(dg, hop, want_sig=False)
        assert np.array_equal(sizes.cpu().numpy(), golden_runs[f"{name}_ring_sizes"])


@pytest.mark.parametrize("name,hops", [("karate", 3), ("mkarate", 2), ("europe", 3)])
def test_degree_distance_small_graphs(golden_graphs, name, hops):
    import torch
    from hsd_b200 import engine
    g = _graph(golden_graphs, name)
    dg = engine.DeviceGraph.upload(g)
    D, _ = engine.degree_distance_device(dg, hops)
    D = D.cpu().numpy().astype(np.float64)
    rows = list(range(g.n)) if g.n <= 80 else [0, 1, 17, 200, g.n - 1]
    ref = O.degree_distance_rows(_oracle_adj(g), hops, rows)
    got = D[rows]
    # north-star tolerance: 1e-5 relative (fp32 accumulation of <= ~600 terms), plus an
    # absolute floor of 1e-6 * max|D| for near-zero distances between near-automorphic nodes
    np.testing.assert_allclose(got, ref, rtol=1e-5, atol=1e-6 * ref.max())
    assert np.array_equal(D, D.T)
    assert np.all(np.diag(D) == 0)


def test_degree_distance_powerlaw_2k():
    import torch
    from hsd_b200 import engine
    from hsd_b200.graph import powerlaw_graph
    g = powerlaw_graph(2000, 5, seed=0)
    dg = engine.DeviceGraph.upload(g)
    D, sizes = engine.degree_distance_device(dg, 3)
    D = D.cpu().numpy().astype(np.float64)
    rows = [0, 3, 500, 1999]
    ref = O.degree_distance_rows(_oracle_adj(g), 3, rows)
    np.testing.assert_allclose(D[rows], ref, rtol=1e-5, atol=1e-6 * ref.max())
    assert np.array_equal(D, D.T)


def test_automorphic_nodes_have_zero_distance(golden_graphs):
    """K-A2: mirrored-karate nodes v and v+34 are automorphic -> D == 0 exactly
    (the property asserted at tests/graphwave_test/main.py:47-50)."""
    import torch
    from hsd_b200 import engine
    g = _graph(golden_graphs, "mkarate")
    labels = golden_graphs["mkarate_labels"]
    dg = engine.DeviceGraph.upload(g)
    D, _ = engine.degree_distance_device(dg, 3)
    D = D.cpu().numpy()
    for lab in np.unique(labels):
        idx = np.nonzero(labels == lab)[0]
        assert np.all(D[np.ix_(idx, idx)] == 0.0)


def test_empty_ring_policy():
    """A node whose BFS exhausts early: 'raise' mirrors scipy's ValueError, 'zero' is the
    point mass at 0 (tools/metrics.py zero padding)."""
    import torch
    from hsd_b200 import engine
    from hsd_b200.graph import CSRGraph
    edges = np.array([[0, 1], [1, 2], [3, 4]])
    g = CSRGraph.from_edges(6, edges)  # node 5 isolated
    dg = engine.DeviceGraph.upload(g)
    with pytest.raises(ValueError):
        engine.degree_distance_device(dg, 2)
    dgz = engine.DeviceGraph.upload(g, include_zero=True)
    D, sizes = engine.degree_distance_device(dgz, 2, empty="zero")
    ref = O.degree_distance_rows(_oracle_adj(g), 2, list(range(6)), empty="zero")
    np.testing.assert_allclose(D.cpu().numpy(), ref, rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("n,m,hops", [(700, 3, 1), (700, 3, 2), (3000, 5, 3), (5000, 2, 4)])
def test_dense_and_frontier_ring_variants_agree_bitwise(n, m, hops, monkeypatch):
    """hsd_ring_signature_degree_dense (bitmap dynamic programming over all nodes) against
    hsd_ring_signature_degree (frontier BFS per source): signatures, ring sizes, ring bitmaps and the
    empty-ring flag must be identical — also with isolated nodes, a self-loop and a source subset."""
    import torch
    from hsd_b200 import engine
    from hsd_b200.graph import CSRGraph, powerlaw_graph
    g0 = powerlaw_graph(n, m, seed=n)
    rows = np.repeat(np.arange(g0.n), np.diff(g0.rowptr))
    e = np.stack([rows, g0.col], 1)
    e = np.concatenate([e[rows < g0.col], [[5, 5]]])               # one self-loop
    g = CSRGraph.from_edges(n + 3, e)                              # three isolated nodes (empty rings)
    dg = engine.DeviceGraph.upload(g, include_zero=True)
    subset = torch.arange(0, g.n, 2, dtype=torch.int32, device="cuda")   # >= half the nodes
    out = {}
    for algo in ("frontier", "dense"):
        monkeypatch.setenv("HSD_RING_ALGO", algo)
        assert engine.ring_algorithm(g.n, g.n, hops, "cuda") == algo
        full = engine.ring_signature_degree(dg, hops, want_bitmaps=True, empty="zero")
        raising = engine.ring_signature_degree(dg, hops, empty="raise", want_sizes=False)
        part = engine.ring_signature_degree(dg, hops, rows=subset, want_bitmaps=True, empty="zero")
        torch.cuda.synchronize()
        out[algo] = (full, raising, part)
    for a, b in zip(out["frontier"], out["dense"]):
        for x, y in zip(a, b):
            assert (x is None) == (y is None)
            if x is not None:
                assert torch.equal(x, y)
    assert int(out["dense"][1][3].item()) & 1                      # isolated nodes raise the empty-ring flag


def test_repeated_sources_fall_back_to_the_frontier_variant(monkeypatch):
    """The dense variant emits one output row per node; a caller-supplied source list with repeats
    must still fill every output row (the dispatcher keeps it on the frontier kernel)."""
    import torch
    from hsd_b200 import engine
    from hsd_b200.graph import powerlaw_graph
    g = powerlaw_graph(900, 4, seed=1)
    dg = engine.DeviceGraph.upload(g)
    monkeypatch.setenv("HSD_RING_ALGO", "dense")
    rows = torch.arange(900, dtype=torch.int32, device="cuda").repeat_interleave(2)[:1500]
    sig, sizes, _, _ = engine.ring_signature_degree(dg, 3, rows=rows)
    ref_sig, ref_sizes, _, _ = engine.ring_signature_degree(dg, 3)
    assert torch.equal(sig, ref_sig[rows.long()]) and torch.equal(sizes, ref_sizes[rows.long()])


def test_bench_dump_outputs_hold_the_timed_path_result(tmp_path):
    """bench.py --dump-outputs: within 64 MB, the seeded sample of rows and the row sums it writes are
    those of the distance matrix the hot path computes on the same graph; --steps sets the step count."""
    import json
    import os
    import subprocess
    import sys
    import torch
    from hsd_b200 import engine
    from hsd_b200.graph import powerlaw_graph
    from hsd_b200.sharded import ShardedDegreeHSD
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    n, hops = 5000, 3                      # the matrix (100 MB) exceeds the dump budget: rows are sampled
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", f"{n}x{hops}", "--steps", "2",
                          "--warmup", "0", "--no-extras", "--no-cpu-baseline", "--no-e2e",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["gpu_launches"] % 2 == 0
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 * 1000 * 1000
    rows = np.load(tmp_path / "distances_rows.npy")
    sample = np.load(tmp_path / "distances_sample.npy")
    sums = np.load(tmp_path / "distances_row_sums.npy")
    assert rows.dtype == np.float64 and sample.dtype == np.float32 and sums.dtype == np.float64
    assert 0 < rows.size < n and sample.shape == (rows.size, n) and sums.shape == (n,)
    D = ShardedDegreeHSD(engine.DeviceGraph.upload(powerlaw_graph(n, 5, seed=0)), hops).step()
    torch.cuda.synchronize()
    D = D.cpu().numpy()
    assert np.array_equal(sample, D[rows.astype(np.int64)])
    np.testing.assert_allclose(sums, D.astype(np.float64).sum(1), rtol=1e-12)
