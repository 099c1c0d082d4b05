"""Times the radius graph of every node in degree mode (engine.degree_radius) against k nearest neighbours
(engine.degree_knn, k = 20) in the same run, one JSON line per configuration, with the device name and
power limit read in the same run.

  python scripts/time_radius.py compare N HOPS     degree_radius and degree_knn, each with the default panel
                                                   budget and with forced 2048-row panels
  python scripts/time_radius.py sweep N HOPS       both with the default budget only (N beyond the device memory)
  python scripts/time_radius.py profile N HOPS [R] one degree_radius call (R-row panels, default budget without R)
                                                   under torch.profiler: CUDA time and launches per kernel name

The radius is the median over nodes of the 20th-NN distance, so a node has about 20 neighbours, as many as
the k-NN lists hold.  Every step is the whole call (signatures, pairwise panels, selection, assembly; no
copy to the host), timed with CUDA events after a 256 MB write that evicts L2, modes alternated step by
step.  It reports the pairwise launches' summed event time, the time outside them (for degree_radius:
count, scans, emits, the one device-to-host count per panel, assembly; for degree_knn: row and column
passes, merges) — both include the signature phase — nnz and the panels.
Options: --steps S (default 3), --warmup W (default 1)."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from hsd_b200 import engine
from hsd_b200.graph import powerlaw_graph

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from time_knn import device_info, opt  # noqa: E402


def profile(dg, n, hops, radius, panel_rows, dev):
    """Per-kernel CUDA time of one degree_radius call after a warm-up call (a run of its own: tracing slows
    the host, so these are not end-to-end numbers)."""
    from torch.profiler import ProfilerActivity
    from torch.profiler import profile as tprofile
    engine.degree_radius(dg, hops, radius, panel_rows=panel_rows)
    torch.cuda.synchronize()
    with tprofile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        out = engine.degree_radius(dg, hops, radius, panel_rows=panel_rows)
        torch.cuda.synchronize()
    kernels = []
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
        if t and e.device_type.name == "CUDA":
            kernels.append({"name": e.key[:120], "cuda_ms": t / 1e3, "calls": e.count})
    kernels.sort(key=lambda k: -k["cuda_ms"])
    print(json.dumps({"n": n, "hops": hops, "radius": radius, "mode": "profile", "panel_rows": panel_rows,
                      "nnz": int(out[1].numel()), **device_info(dev), "kernels": kernels}), flush=True)


def main():
    args = [a for i, a in enumerate(sys.argv[1:], 1) if not a.startswith("--") and not sys.argv[i - 1].startswith("--")]
    mode, n, hops = args[0], int(args[1]), int(args[2])
    k = 20
    steps, warmup = opt("--steps", 3), opt("--warmup", 1)
    dev = torch.device("cuda", torch.cuda.current_device())
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    dg = engine.DeviceGraph.upload(powerlaw_graph(n, 5, seed=0), device=dev)
    _, val = engine.degree_knn(dg, hops, k)
    radius = float(val[:, k - 1].median())
    del val

    def knn(panel_rows):
        def run():
            ev = []
            out = engine.degree_knn(dg, hops, k, panel_rows=panel_rows, pair_events=ev)
            return out, ev
        return run

    def radius_graph(panel_rows):
        def run():
            ev = []
            out = engine.degree_radius(dg, hops, radius, panel_rows=panel_rows, pair_events=ev)
            return out, ev
        return run

    if mode == "profile":
        profile(dg, n, hops, radius, int(args[3]) if len(args) > 3 else None, dev)
        return
    if mode == "compare":
        modes = {"knn_default": knn(None), "radius_default": radius_graph(None),
                 "knn_panels_2048": knn(2048), "radius_panels_2048": radius_graph(2048)}
    else:
        modes = {"knn_default": knn(None), "radius_default": radius_graph(None)}
    times = {m: [] for m in modes}
    pair = {m: [] for m in modes}
    panels_of, nnz_of = {}, {}
    for step in range(warmup + steps):
        for m, fn in modes.items():
            flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out, ev = fn()
            e1.record()
            e1.synchronize()
            if step >= warmup:
                times[m].append(e0.elapsed_time(e1))
                pair[m].append(sum(a.elapsed_time(b) for _, _, a, b in ev))
                panels_of[m] = [(r0, r1) for r0, r1, _, _ in ev]
                if m.startswith("radius"):
                    nnz_of[m] = int(out[1].numel())
            del out
    rec = {"n": n, "hops": hops, "k": k, "radius": radius, "k_used": dg.k_used(hops), "steps": steps,
           "warmup": warmup, "l2": "256 MB written before every step", **device_info(dev)}
    for m in modes:
        t, p = np.array(times[m]), np.array(pair[m])
        panels = panels_of[m]
        r = dict(rec, mode=m, step_ms_median=float(np.median(t)), step_ms_min=float(t.min()),
                 step_ms_max=float(t.max()), pairwise_ms_median=float(np.median(p)),
                 outside_pairwise_ms=float(np.median(t)) - float(np.median(p)),
                 panel_rows=panels[0][1] - panels[0][0], n_panels=len(panels))
        if m in nnz_of:
            r.update(nnz=nnz_of[m], nnz_per_node=nnz_of[m] / n)
        print(json.dumps(r), flush=True)
    torch.cuda.synchronize()


if __name__ == "__main__":
    main()
