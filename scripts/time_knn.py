"""Times k nearest neighbours of every node in degree mode (engine.degree_knn), one JSON line per
configuration, with the device name and power limit read in the same run.

  python scripts/time_knn.py compare N HOPS [K]      today's resident path (full matrix + topk_rows)
                                                     against degree_knn with the default panel budget
                                                     and with forced 2048-row panels
  python scripts/time_knn.py sweep N HOPS [K]        degree_knn alone (N beyond the device memory);
  torchrun --nproc_per_node G scripts/time_knn.py sweep N HOPS [K]   the same on G GPUs
  python scripts/time_knn.py emulate N HOPS [K] --world W
                                                     one GPU runs each of W ranks' panel sweeps in turn
                                                     (the default W-rank panel plan and dealing): the
                                                     sweep's strong-scaling efficiency without the
                                                     signature phase and the all-gather

Every step is the whole call (signatures, pairwise panels, selection, merges; no copy to the host),
timed with CUDA events after a 256 MB write that evicts L2, modes alternated step by step.  For the
panel sweep it also reports the pairwise launches' summed event time, their share of the live-measured
FP32 issue peak (flops = 2 x pairs x signature length), and the time outside them (row pass, column
pass, merges, signatures).  Options: --steps S (default 3), --warmup W (default 1)."""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

from hsd_b200 import engine
from hsd_b200.graph import powerlaw_graph


def opt(name, default):
    return int(sys.argv[sys.argv.index(name) + 1]) if name in sys.argv else default


def device_info(dev):
    info = {"device": torch.cuda.get_device_name(dev)}
    try:   # read-only query of the board's power limit
        out = subprocess.run(["nvidia-smi", "-i", str(dev.index or 0), "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in out.split(",")]
    except Exception as e:
        info["power_limit"] = f"unavailable ({type(e).__name__})"
    return info


def timed(fn, flush):
    flush.fill_(1.0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def emulate(dg, n, hops, k, world, steps, warmup, flush, rec):
    """Time the 1-GPU call, the signature phase alone, and every rank's call of a `world`-rank plan
    (no process group: each call builds the whole table here, then sweeps that rank's panels)."""
    ones, sigs, ranks = [], [], [[] for _ in range(world)]
    for step in range(warmup + steps):
        t1 = timed(lambda: engine.degree_knn(dg, hops, k), flush)
        ts = timed(lambda: engine._knn_table(dg, hops, "raise", 0, 1, None), flush)
        tr = [timed(lambda: engine.degree_knn(dg, hops, k, rank=r, world=world), flush) for r in range(world)]
        if step >= warmup:
            ones.append(t1)
            sigs.append(ts)
            for r in range(world):
                ranks[r].append(tr[r])
    t1, ts = float(np.median(ones)), float(np.median(sigs))
    tr = [float(np.median(x)) for x in ranks]
    free = torch.cuda.mem_get_info(dg.rowptr.device)[0]
    rows = engine.knn_panel_rows(n, int(free * engine.KNN_BLOCK_FRACTION), world)
    deal = engine.knn_deal(n, engine.knn_panels(n, rows), world)
    print(json.dumps(dict(rec, mode="emulate", emulated_world=world, one_gpu_ms=t1, signature_ms=ts,
                          rank_call_ms=tr, panel_rows=rows, panels_per_rank=[len(d) for d in deal],
                          sweep_efficiency=(t1 - ts) / (world * (max(tr) - ts)))), flush=True)


def main():
    args = [a for i, a in enumerate(sys.argv[1:], 1) if not a.startswith("--") and not sys.argv[i - 1].startswith("--")]
    mode, n, hops = args[0], int(args[1]), int(args[2])
    k = int(args[3]) if len(args) > 3 else 20
    steps, warmup = opt("--steps", 3), opt("--warmup", 1)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if world > 1:
        lr = int(os.environ["LOCAL_RANK"])
        torch.cuda.set_device(lr)
        dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
    dev = torch.device("cuda", torch.cuda.current_device())
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    peak = engine.fp32_issue_peak()
    dg = engine.DeviceGraph.upload(powerlaw_graph(n, 5, seed=0), device=dev)
    k_used = dg.k_used(hops)

    if mode == "emulate":
        rec = {"n": n, "hops": hops, "k": k, "k_used": k_used, "steps": steps, "warmup": warmup,
               "l2": "256 MB written before every call", **device_info(dev)}
        emulate(dg, n, hops, k, opt("--world", 8), steps, warmup, flush, rec)
        return

    def resident():
        D, _ = engine.degree_distance_device(dg, hops)
        out = engine.topk_rows(D, k)
        del D
        return out, []

    def sweep(panel_rows):
        def run():
            ev = []
            out = engine.degree_knn(dg, hops, k, panel_rows=panel_rows, rank=rank, world=world, pair_events=ev)
            return out, ev
        return run

    modes = {"resident": resident, "knn_default": sweep(None), "knn_panels_2048": sweep(2048)} \
        if mode == "compare" else {"knn_default": sweep(None)}
    panels_of = {}
    times = {m: [] for m in modes}
    pair = {m: [] for m in modes}
    results = {}
    for step in range(warmup + steps):
        for m, fn in modes.items():
            flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            if world > 1:
                dist.barrier()
            e0.record()
            out, ev = fn()
            e1.record()
            e1.synchronize()
            if step >= warmup:
                t = e0.elapsed_time(e1)
                p = sum(a.elapsed_time(b) for _, _, a, b in ev)
                panels_of[m] = [(r0, r1) for r0, r1, _, _ in ev]
                if world > 1:   # the step ends when the slowest rank ends
                    tt = torch.tensor([t, p], dtype=torch.float64, device=dev)
                    allr = [torch.zeros_like(tt) for _ in range(world)]
                    dist.all_gather(allr, tt)
                    t = max(float(a[0]) for a in allr)
                    p = [float(a[1]) for a in allr]
                times[m].append(t)
                pair[m].append(p)
            results[m] = out
            del out
    ref = results.get("resident")
    rec = {"n": n, "hops": hops, "k": k, "k_used": k_used, "world": world, "steps": steps, "warmup": warmup,
           "l2": "256 MB written before every step", "fp32_issue_peak_lane_ops_per_s": peak, **device_info(dev)}
    for m in modes:
        t = np.array(times[m])
        r = dict(rec, mode=m, step_ms_median=float(np.median(t)), step_ms_min=float(t.min()),
                 step_ms_max=float(t.max()))
        if ref is not None:
            r["bit_equal_to_resident"] = bool(torch.equal(results[m][0], ref[0]) and
                                              torch.equal(results[m][1].view(torch.int32), ref[1].view(torch.int32)))
        if m != "resident":
            mine = panels_of[m]                          # the panels this rank swept (rank 0)
            panel_rows = mine[0][1] - mine[0][0] if len(mine) > 1 or world > 1 else n
            deal = engine.knn_deal(n, engine.knn_panels(n, panel_rows), world)
            assert deal[rank] == mine
            pairs = [sum(engine.knn_panel_work(n, *p) for p in d) for d in deal]
            pms = np.array(pair[m])          # [steps] or [steps, world]
            pms = pms.reshape(len(t), -1)
            frac = [2.0 * pairs[q] * k_used / (float(np.median(pms[:, q])) * 1e-3) / peak for q in range(pms.shape[1])]
            r.update(panel_rows=panel_rows, n_panels=sum(len(d) for d in deal),
                     pairwise_ms_median_per_rank=[float(np.median(pms[:, q])) for q in range(pms.shape[1])],
                     pairwise_frac_of_fp32_issue_peak_per_rank=frac,
                     outside_pairwise_ms=float(np.median(t)) - float(np.median(pms.max(1))),
                     outside_pairwise_share=1.0 - float(np.median(pms.max(1))) / float(np.median(t)))
        if rank == 0:
            print(json.dumps(r), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
