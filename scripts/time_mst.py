"""Times the minimum spanning tree in degree mode (engine.degree_mst) for several candidate-list sizes against one
k-nearest-neighbour sweep (engine.degree_knn, k = 20) in the same run, one JSON line per configuration, with the
device name and power limit read in the same run.

  python scripts/time_mst.py N HOPS [--cand 0,16,32,64] [--steps S] [--warmup W]

Graph: powerlaw_graph(N, 5, seed=0).  Every step is one whole call (signatures, k-NN lists when cand_k > 0, rounds;
no copy to the host), timed with CUDA events after a 256 MB write that evicts L2, modes alternated step by step.
Per cand_k it reports the call time, the time before round 1 (signatures and lists), the rounds, the sweeps
(rounds the lists could not certify) and the mean wall time of a sweep round and of a certified round (from
degree_mst's stats of the last step).  A last record
times hsd_mst_panel_min alone on the first default panel (CUDA events over 5 launches) with the bytes it reads
(the panel's upper part), so its share of a sweep shows beside the pairwise launches."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from hsd_b200 import engine
from hsd_b200._lib import check, lib
from hsd_b200.graph import powerlaw_graph

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from time_knn import device_info, opt  # noqa: E402


def panel_min_kernel(dg, n, hops, dev):
    """Event time of hsd_mst_panel_min on the first panel of the default k-NN plan (random labels)."""
    sigT, _ = engine._knn_table(dg, hops, "raise", 0, 1, None)
    R = engine.knn_panel_rows(n, int(engine._free_bytes(dev) * engine.KNN_BLOCK_FRACTION))
    ld = engine.roundup(n, 4)
    B = torch.empty((R, ld), dtype=torch.float32, device=dev)
    st = engine._stream()
    engine._panel_pairwise(sigT, dg.k_used(hops), n, 0, R, B, ld, st)
    comp = torch.randint(0, 1 << 20, (n,), dtype=torch.int32, device=dev)
    keys = torch.empty(n, dtype=torch.int64, device=dev)
    reps = 5
    keys.fill_(engine.MST_KEY_NONE)
    check(lib.hsd_mst_panel_min(B.data_ptr(), ld, R, n, 0, engine._ptr(comp), engine._ptr(keys), st))   # warm-up
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        check(lib.hsd_mst_panel_min(B.data_ptr(), ld, R, n, 0, engine._ptr(comp), engine._ptr(keys), st))
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / reps
    upper = R * n - R * (R + 1) // 2                     # elements with c > r
    return {"mode": "panel_min_kernel", "panel_rows": R, "n_cols": n, "kernel_ms": ms,
            "bytes_read": 4 * upper, "gb_per_s": 4 * upper / (ms * 1e-3) / 1e9}


def main():
    args = [a for i, a in enumerate(sys.argv[1:], 1) if not a.startswith("--") and not sys.argv[i - 1].startswith("--")]
    n, hops = int(args[0]), int(args[1])
    steps, warmup = opt("--steps", 2), opt("--warmup", 1)
    cands = [int(c) for c in (sys.argv[sys.argv.index("--cand") + 1] if "--cand" in sys.argv else "0,16,32,64").split(",")]
    dev = torch.device("cuda", torch.cuda.current_device())
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    dg = engine.DeviceGraph.upload(powerlaw_graph(n, 5, seed=0), device=dev)

    def mst(cand_k):
        def run():
            st = {}
            out = engine.degree_mst(dg, hops, cand_k=cand_k, stats=st)
            return out, st
        return run

    def knn():
        return engine.degree_knn(dg, hops, 20), None

    modes = {"knn_k20": knn, **{f"mst_cand_{c}": mst(c) for c in cands}}
    times = {m: [] for m in modes}
    stats_of = {}
    ref = None
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
                if st is not None:
                    stats_of[m] = st
            if st is not None:                           # every cand_k must give the same tree
                got = tuple(t.cpu() for t in out)
                if ref is None:
                    ref = got
                assert all(torch.equal(a, b) for a, b in zip(got[:2], ref[:2])) and \
                    torch.equal(got[2].view(torch.int32), ref[2].view(torch.int32)), m
            del out
    rec = {"n": n, "hops": hops, "k_used": dg.k_used(hops), "steps": steps, "warmup": warmup,
           "l2": "256 MB written before every step", **device_info(dev)}
    knn_ms = float(np.median(times["knn_k20"]))
    for m in modes:
        t = np.array(times[m])
        r = dict(rec, mode=m, call_ms_median=float(np.median(t)), call_ms_min=float(t.min()),
                 call_ms_max=float(t.max()))
        if m in stats_of:
            st = stats_of[m]
            sw = [ms for ms, s in zip(st["round_ms"], st["swept"]) if s]
            cert = [ms for ms, s in zip(st["round_ms"], st["swept"]) if not s]
            r.update(rounds=st["rounds"], sweeps=st["sweeps"], setup_ms=st["setup_ms"], swept=st["swept"],
                     round_ms=[round(x, 3) for x in st["round_ms"]],
                     sweep_round_ms_mean=float(np.mean(sw)) if sw else None,
                     certified_round_ms_mean=float(np.mean(cert)) if cert else None,
                     knn_k20_ms=knn_ms, call_over_knn=float(np.median(t)) / knn_ms)
        print(json.dumps(r), flush=True)
    print(json.dumps(dict(rec, **panel_min_kernel(dg, n, hops, dev))), flush=True)
    torch.cuda.synchronize()


if __name__ == "__main__":
    main()
