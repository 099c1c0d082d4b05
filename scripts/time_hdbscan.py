"""Times HDBSCAN's mutual-reachability minimum spanning tree in degree mode (engine.degree_mreach_mst) at several
min_samples against the plain MST (engine.degree_mst) in the same run, then the host labelling
(engine.single_linkage_host + engine.hdbscan_host) at 10^5 and 10^6 nodes; one JSON line per record, with the device
name and power limit read in the same run.

  python scripts/time_hdbscan.py N HOPS [--ms 1,5,17] [--steps S] [--warmup W]
  python scripts/time_hdbscan.py --host [--sizes 100000,1000000]

Graph: powerlaw_graph(N, 5, seed=0).  Every step is one whole call (signatures, k-NN lists, rounds; no copy to the
host), timed with CUDA events after a 256 MB write that evicts L2, modes alternated step by step.  Per mode it
reports the call time, the time before round 1 (signatures, lists and cores), the rounds, the sweeps (rounds the
lists could not certify) and which rounds swept (degree_mreach_mst's stats of the last step).  The host records
time the labelling of a random spanning tree's dendrogram (edges in random order, heights on 1000 levels: many
ties) with a host clock, best of three."""
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def host(sizes):
    from hsd_b200 import engine
    for n in sizes:
        rng = np.random.default_rng(n)
        u = np.arange(1, n, dtype=np.int32)
        v = (rng.random(n - 1) * u).astype(np.int32)        # a random tree: node t joins an earlier node
        perm = rng.permutation(n - 1)                       # merged in random order
        u, v = u[perm], v[perm]
        d = np.sort(rng.integers(0, 1000, n - 1).astype(np.float32) / np.float32(64))
        best = {}
        for _ in range(3):
            t0 = time.perf_counter()
            Z = engine.single_linkage_host(np.minimum(u, v), np.maximum(u, v), d, n)
            best["single_linkage_host_ms"] = min(best.get("single_linkage_host_ms", 1e30),
                                                 (time.perf_counter() - t0) * 1e3)
            for method in ("eom", "leaf"):
                t0 = time.perf_counter()
                labels, _ = engine.hdbscan_host(Z, n, 5, method)
                key = f"hdbscan_host_{method}_ms"
                best[key] = min(best.get(key, 1e30), (time.perf_counter() - t0) * 1e3)
        print(json.dumps({"mode": "host_labelling", "n": n, "min_cluster_size": 5, "clusters": int(labels.max() + 1),
                          **best}), flush=True)


def main():
    from time_knn import opt
    if "--host" in sys.argv:
        sizes = sys.argv[sys.argv.index("--sizes") + 1] if "--sizes" in sys.argv else "100000,1000000"
        host([int(s) for s in sizes.split(",")])
        return
    import torch
    from hsd_b200 import engine
    from hsd_b200.graph import powerlaw_graph
    from time_knn import device_info
    args = [a for i, a in enumerate(sys.argv[1:], 1) if not a.startswith("--") and not sys.argv[i - 1].startswith("--")]
    n, hops = int(args[0]), int(args[1])
    steps, warmup = opt("--steps", 2), opt("--warmup", 1)
    mss = [int(c) for c in (sys.argv[sys.argv.index("--ms") + 1] if "--ms" in sys.argv else "1,5,17").split(",")]
    dev = torch.device("cuda", torch.cuda.current_device())
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    dg = engine.DeviceGraph.upload(powerlaw_graph(n, 5, seed=0), device=dev)

    def plain():
        st = {}
        return engine.degree_mst(dg, hops, stats=st), st

    def mreach(ms):
        def run():
            st = {}
            return engine.degree_mreach_mst(dg, hops, ms, stats=st), st
        return run

    modes = {"degree_mst": plain, **{f"mreach_ms_{ms}": mreach(ms) for ms in mss}}
    times = {m: [] for m in modes}
    stats_of = {}
    for step in range(warmup + steps):
        for m, fn in modes.items():
            flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out, st = fn()
            e1.record()
            e1.synchronize()
            if step >= warmup:
                times[m].append(e0.elapsed_time(e1))
                stats_of[m] = st
            if m == "mreach_ms_1":                       # min_samples = 1 is the plain tree
                ref = modes["degree_mst"]()[0]
                assert all(torch.equal(a.view(torch.int32), b.view(torch.int32)) for a, b in zip(out[:3], ref))
            del out
    rec = {"n": n, "hops": hops, "k_used": dg.k_used(hops), "steps": steps, "warmup": warmup,
           "l2": "256 MB written before every step", **device_info(dev)}
    base = float(np.median(times["degree_mst"]))
    for m in modes:
        t = np.array(times[m])
        st = stats_of[m]
        print(json.dumps(dict(rec, mode=m, call_ms_median=float(np.median(t)), call_ms_min=float(t.min()),
                              call_ms_max=float(t.max()), over_degree_mst=float(np.median(t)) / base,
                              rounds=st["rounds"], sweeps=st["sweeps"], setup_ms=st["setup_ms"], swept=st["swept"],
                              round_ms=[round(x, 3) for x in st["round_ms"]])), flush=True)
    torch.cuda.synchronize()


if __name__ == "__main__":
    main()
