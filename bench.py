#!/usr/bin/env python
"""bench.py — HSD node-pairs/sec for the degree-mode 3-hop distance matrix.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--workload c2|c3|NODESxHOPS]
                    [--dump-outputs DIR]

One "step" = one full pass of the hot path over the workload graph: k-hop rings
(bitmap dynamic programming over all nodes, or one frontier BFS per source) -> per-ring degree CDF signatures -> (N>1: one NCCL all-gather of
the signature table, or peer-memory stores fused into the BFS kernel) -> pairwise W1 (L1
between signatures) for this rank's share of the symmetric tiles.
`value` is whole-job unordered node pairs / second with the graph already in HBM;
`e2e` is the same job through the host-buffer pipeline (pinned host CSR in, pinned
host float32 matrix out, copies inside the timed region).  Both legs time K steps.

Workload (BASELINE.json configs[1]): networkx.barabasi_albert_graph(20000, 5, seed=0),
3 hops, full N x N.  With N>1 ranks the SAME graph is row-block sharded (strong scaling).

`--impl reference` times the reference's CPU algorithm for this path (the oracle
port: Python BFS rings of tools/hierarchy.py + scipy.stats.wasserstein_distance per
pair and hop, model/HSD.py:98-114) on the box's host cores on a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "HSD node-pairs/sec (3-hop distance matrix)"
UNIT = "node-pairs/s"
CPU_SAMPLE_NODES = 160   # 12 720 sampled pairs x (hops + 1) scipy calls ~ 10-30 s of CPU work per step


def parse_workload(spec: str):
    if spec == "c2":
        return 20000, 3
    if spec == "c3":
        return 100000, 4
    n, h = spec.lower().split("x")
    return int(n), int(h)


# ------------------------------------------------------------------------------
# CPU baseline / reference arm: the oracle port on host cores, bounded sample
# ------------------------------------------------------------------------------
_POOL_STATE = {}


def _cap_threads():
    """One thread per worker process: scipy's W1 ends in a BLAS dot, and a forked worker otherwise
    inherits a BLAS/OpenMP pool as wide as the machine — `cores` processes x `cores` spinning threads
    made the round-1 reference arm 85x slower without torchrun (which exports OMP_NUM_THREADS=1)
    than with it.  Environment for pools created later, threadpoolctl for the ones already loaded."""
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        os.environ[k] = "1"
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)
    except Exception:
        pass


def _pool_init(n, edges, hops):
    _cap_threads()
    from oracle import hsd_oracle as O
    _POOL_STATE["adj"] = O.adjacency_from_edges(n, edges)
    _POOL_STATE["hops"] = hops
    _POOL_STATE["deg"] = np.array([len(a) for a in _POOL_STATE["adj"]], dtype=np.float64)


def _pool_rings(src):
    from oracle import hsd_oracle as O
    t = time.perf_counter()
    layers = O.rings_of(_POOL_STATE["adj"], int(src), _POOL_STATE["hops"])
    deg = _POOL_STATE["deg"]
    sig = [deg[np.asarray(l, dtype=np.int64)] for l in layers]
    return int(src), sig, time.perf_counter() - t


def _pool_pairs(args):
    from oracle import hsd_oracle as O
    sig_i, sig_js = args
    t = time.perf_counter()
    out = [sum(O.w1(sig_i[h], sj[h]) for h in range(len(sig_i))) for sj in sig_js]
    return out, time.perf_counter() - t


class CpuReference:
    """model/HSD.py:98-114 with a degree-valued ring signal, through the oracle, on all host cores."""

    def __init__(self, n, hops, sample_nodes=48, seed=0):
        import multiprocessing as mp
        import networkx as nx
        self.n, self.hops = n, hops
        g = nx.barabasi_albert_graph(n, 5, seed=seed)
        self.edges = np.array(g.edges(), dtype=np.int64)
        self.n_bins = int(np.unique(np.bincount(self.edges.ravel(), minlength=n)).size)   # distinct degrees
        self.cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        _cap_threads()      # before the fork: the workers inherit single-threaded BLAS/OpenMP pools
        self.sample = np.sort(np.random.default_rng(seed).choice(n, size=min(sample_nodes, n), replace=False))
        self.pool = mp.get_context("fork").Pool(self.cores, initializer=_pool_init,
                                                initargs=(n, self.edges, hops))

    def step(self):
        """One bounded pass: rings of the sampled sources + all pairs among them.
        Returns (extrapolated full-workload pairs/s, details)."""
        t0 = time.perf_counter()
        res = self.pool.map(_pool_rings, list(self.sample), chunksize=max(1, len(self.sample) // (4 * self.cores)))
        t_rings_wall = time.perf_counter() - t0
        sigs = [r[1] for r in res]
        ring_cpu = sum(r[2] for r in res)
        s = len(sigs)
        t1 = time.perf_counter()
        jobs = [(sigs[i], sigs[i + 1:]) for i in range(s - 1)]
        out = self.pool.map(_pool_pairs, jobs, chunksize=1)
        t_pairs_wall = time.perf_counter() - t1
        pair_cpu = sum(o[1] for o in out)
        n_pairs = s * (s - 1) // 2
        # full job on `cores` cores: N ring builds + N(N-1)/2 pair evaluations
        full_pairs = self.n * (self.n - 1) / 2
        t_full = (self.n * (ring_cpu / s) + full_pairs * (pair_cpu / n_pairs)) / self.cores
        return full_pairs / t_full, dict(sample_nodes=s, sample_pairs=n_pairs, rings_wall_s=t_rings_wall,
                                         pairs_wall_s=t_pairs_wall, ring_cpu_s_per_source=ring_cpu / s,
                                         pair_cpu_s=pair_cpu / n_pairs, step_wall_s=time.perf_counter() - t0)

    def describe(self, d):
        return (f"{d['sample_nodes']} sampled sources: Python BFS rings ({d['ring_cpu_s_per_source']*1e3:.1f} ms/source) + "
                f"{d['sample_pairs']} pairs x {self.hops + 1} hops of scipy wasserstein_distance "
                f"({d['pair_cpu_s']*1e6:.0f} us/pair), extrapolated to N={self.n} on {self.cores} worker processes, "
                f"one thread each (OMP/MKL/OPENBLAS_NUM_THREADS=1 + threadpoolctl; perfect scaling assumed)")

    def close(self):
        self.pool.close()
        self.pool.join()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n, hops = parse_workload(args.workload)
    ref = CpuReference(n, hops, sample_nodes=CPU_SAMPLE_NODES)
    for _ in range(args.warmup):
        ref.step()
    vals, last = [], None
    t0 = time.perf_counter()
    for _ in range(args.steps):
        v, last = ref.step()
        vals.append(v)
    wall = time.perf_counter() - t0
    ref.close()
    value = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall / max(args.steps, 1) * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": workload_config(n, hops, max(args.gpus, 1), args.gpus > 1 and not args.no_peer, ref.n_bins),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": ref.cores, "kind": "port",
                         "sample": ref.describe(last)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------
# clocks sampling (NVML) during the timed region
# ------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def bind_to_gpu_numa_node(index):
    """Restrict this process to the CPUs NVML reports as local to GPU `index`, so that pinned
    host buffers (first touch) and the copy threads sit on the socket the GPU's PCIe link hangs
    off.  With 4-8 ranks streaming results to the host at once, remote-socket buffers otherwise
    halve the device-to-host rate.  Best effort: returns the CPU count bound, or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n_cpu = os.cpu_count() or 1
        words = (n_cpu + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {w * 64 + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


# ------------------------------------------------------------------------------
# native arm
# ------------------------------------------------------------------------------
class Ctx:
    """Per-process state of the native arm: rank / device / collectives helpers / peaks."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args = torch, dist, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py (native arm) needs a CUDA device: hsd_b200 has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.numa = bind_to_gpu_numa_node(self.local_rank)   # pinned host buffers land on the GPU's own socket
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.peer = self.world > 1 and not args.no_peer
        self.flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=self.dev)  # > 126 MB L2
        from hsd_b200 import engine
        self.fp32_peak = engine.fp32_issue_peak()    # live FP32 CUDA-core issue peak (pairwise roofline denominator)
        self.peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                self.peaks = json.load(f)
        except Exception:
            pass
        self.hbm_peak = float(self.peaks.get("hbm_gbs", 6650.0))
        self.hbm_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if self.peaks else "fallback 6650 GB/s (of fallback)"

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())


def measure_degree_path(ctx, g, hops, steps, warmup, workload_key):
    """The hot path (rings -> signatures -> [fused all-gather] -> pairwise) on graph `g`, sharded over
    ctx.world ranks: warm-up, then `steps` timed steps (CUDA events, barrier + synchronize on both
    sides, max over ranks, L2 flushed before every step).  Returns (record, plan, dg, block): block is this
    rank's rows of the distance matrix as the last timed step left them."""
    torch = ctx.torch
    from hsd_b200 import engine
    from hsd_b200.sharded import ShardedDegreeHSD
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    n = g.n
    dg = engine.DeviceGraph.upload(g, device=dev)
    peer = ctx.peer
    try:
        plan = ShardedDegreeHSD(dg, hops, rank, world, peer=peer)
    except Exception as e:   # symmetric memory unavailable: every rank computes its full row block
        if rank == 0:
            print(f"[bench] peer-memory result blocks unavailable ({type(e).__name__}: {e}); "
                  "falling back to independent row blocks", file=sys.stderr)
        peer = False
        plan = ShardedDegreeHSD(dg, hops, rank, world, peer=False)
    pairs = n * (n - 1) / 2

    def one_step(ev=None):
        if ev is not None:
            ev[4].record()
        ctx.flush.fill_(1.0)               # evict the previous step's tables from L2
        if ev is not None:
            ev[0].record()
        plan.signatures()
        if ev is not None:
            ev[1].record()
        plan.gather()
        if ev is not None:
            out = plan.distances(ev[2], ev[3])   # (N > 1: ends with the device-side barrier that completes the blocks)
            ev[5].record()
            return out
        return plan.distances()

    for _ in range(max(warmup, 0)):
        one_step()
    torch.cuda.synchronize()
    plan.check()

    events = [[torch.cuda.Event(enable_timing=True) for _ in range(6)] for _ in range(steps)]
    sampler = ClockSampler(ctx.local_rank)
    ctx.barrier()
    torch.cuda.synchronize()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(steps):
        block = one_step(events[k])
    e1.record()
    torch.cuda.synchronize()
    ctx.barrier()
    clocks = sampler.stop()
    ms_per_step = ctx.max_over_ranks(e0.elapsed_time(e1)) / steps
    value = pairs / (ms_per_step * 1e-3)
    bfs_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in events]))
    gather_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in events]))
    pair_ms = float(np.mean([e[2].elapsed_time(e[3]) for e in events]))
    flush_ms = float(np.mean([e[4].elapsed_time(e[0]) for e in events]))
    tail_ms = float(np.mean([e[3].elapsed_time(e[5]) for e in events]))

    per_rank = None
    if world > 1:   # the same stage times on every rank (rank skew shows up as waiting at the barriers)
        mine = torch.tensor([bfs_ms, gather_ms, pair_ms, tail_ms], dtype=torch.float64, device=dev)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        ctx.dist.all_gather(allr, mine)
        per_rank = {k: [round(float(t[i]), 4) for t in allr]
                    for i, k in enumerate(("bfs_signature", "allgather_transpose", "pairwise", "final_barrier"))}

    # ---- roofline of the dominant kernel (pairwise L1) ----
    # algorithmic flops per launch = 2 (subtract, |.|-accumulate) x unordered pairs this launch
    # covers x signature length; hop 0 is one scalar (the kernel treats it so), every later hop B-1 gaps
    k_alg = plan.k_used
    if world == 1:
        launch_pairs = pairs
    elif peer:
        launch_pairs = pairs / world        # this rank's share of the upper-triangle tiles
    else:
        launch_pairs = plan.n_rows * n      # ordered (row, col) pairs of this rank's block
    flops = 2.0 * launch_pairs * k_alg
    achieved = flops / (pair_ms * 1e-3) / 1e12 if pair_ms > 0 else 0.0
    traffic = None   # DRAM bytes per launch from the committed ncu --set full capture of this workload
    try:
        with open(os.path.join(ROOT, "profiles", "pairwise_ncu_traffic.json")) as f:
            cap = json.load(f)
        if world == 1 and cap.get("workload") == workload_key:
            traffic = cap["dram_bytes_read"] + cap["dram_bytes_write"]
    except Exception:
        pass
    fp32_peak = ctx.fp32_peak
    pair_kernel = ("pairwise_l1_n64_kernel (128 x 64 tiles, one per CTA)" if getattr(plan, "tile_list", None) is not None
                   and getattr(plan, "tile_n", 128) == 64 else "pairwise_l1_v2_kernel")
    roofline = {
        "kernel": pair_kernel, "bound": "fp32", "achieved": achieved, "peak": fp32_peak / 1e12,
        "unit": "TFLOP/s", "frac": achieved / (fp32_peak / 1e12), "traffic": traffic,
        "peak_source": "measured live: hsd_fp32_peak_probe (register-only FADD sub+|.|-accumulate), "
                       "1 flop per lane per clock; MEASURED_PEAKS.json has no FP32 CUDA-core entry",
        "flops_per_launch": flops, "ms_per_launch": pair_ms,
        "note": "tensor cores not applicable (|a-b| is not a contraction); FMA-counted peak would be 2x this",
    }
    # ---- secondary: ring + signature phase against HBM/L2 ----
    own = slice(plan.rank * plan.per, plan.rank * plan.per + plan.n_src)   # this rank's sources in the table
    variant = "cols" if getattr(plan, "ring_mode", "rows") == "cols" else engine.ring_algorithm(n, plan.n_src, hops, dev)
    if variant == "cols":
        # column-split dense variant: every level for all nodes on 1/world of the bitmap words, then one integer
        # all-reduce of the partial counts (N x (hops (B-1) + hops) int32) and the signature build for all nodes
        row_b = ((n + 31) // 32 + 3) // 4 * 4 * 4.0 / world
        nnz = float(dg.nnz)
        ring_bytes = 2 * n * row_b + (hops - 1) * ((nnz + n) * row_b + n * row_b + 2 * n * row_b)
        counts_b = 4.0 * n * (hops * (dg.n_bins - 1) + hops)
        ring_bytes += hops * counts_b / hops + 2 * counts_b + 4.0 * k_alg * n      # counts written, all-reduced, read; table written
        ring_kernel = "ball_or_kernel + ring_count_cols_kernel + signature_from_counts_kernel (column-split dense variant) + NCCL all-reduce of the counts"
        ring_note = (f"each rank runs the bitmap recursion for all nodes on 1/{world} of the bitmap columns; "
                     f"{counts_b/1e6:.0f} MB of int32 partial counts are summed by one all-reduce")
        edges_scanned = None
    elif variant == "dense":
        # bitmap dynamic programming: level h >= 2 reads (entries + rows) N-bit rows of the previous table and
        # writes one row per computed node; intermediate levels cover all nodes, the last one this rank's sources
        row_b = ((n + 31) // 32 + 3) // 4 * 4 * 4.0
        nnz = float(dg.nnz)
        ring_bytes = n * row_b + plan.n_src * row_b                      # level 1: table build + CDF read
        for h in range(2, hops + 1):
            rows_h = n if h < hops else plan.n_src
            ring_bytes += (nnz * rows_h / n + rows_h) * row_b + rows_h * row_b
        ring_bytes += 4.0 * k_alg * plan.n_src
        ring_kernel = "ball_or_cdf_kernel + ring_cdf_kernel (dense ring variant)"
        ring_note = ("bitmap dynamic programming over all nodes: (H-1) levels of (2E+N) row reads of N/8 bytes; hub rows "
                     "are re-read from L2, so DRAM traffic is below the algorithmic bytes")
        edges_scanned = None
    else:
        sig_rows = plan.sig_all[own, 1:k_alg].double()
        nb1 = dg.n_bins - 1
        sizes = plan.sizes[own].double()
        sup_max = float(dg.support[-1])
        edges_scanned = float((plan.sig_all[own, 0].double()).sum().item())  # hop 0 expands the source
        for h in range(1, hops):   # rings 1..H-1 are expanded; sum of member degrees = n * mean = n * (max - sum_b CDF*delta)
            mean_deg = sup_max - sig_rows[:, (h - 1) * nb1:h * nb1].sum(1)
            edges_scanned += float((sizes[:, h] * mean_deg).sum().item())
        ring_bytes = 4.0 * edges_scanned + 4.0 * k_alg * plan.n_src
        ring_kernel = "bfs_ring_signature_kernel (frontier ring variant)"
        ring_note = "CSR and bitmaps are L2/SMEM resident, so the HBM fraction is structurally small (SURVEY H4)"
    roofline_bfs = {
        "kernel": ring_kernel, "bound": "hbm", "achieved": ring_bytes / (bfs_ms * 1e-3) / 1e9,
        "peak": ctx.hbm_peak, "unit": "GB/s", "frac": ring_bytes / (bfs_ms * 1e-3) / 1e9 / ctx.hbm_peak, "traffic": None,
        "peak_source": ctx.hbm_src,
        "bytes_per_launch": ring_bytes, "ms_per_launch": bfs_ms, "edges_scanned_per_launch": edges_scanned,
        "note": ring_note,
    }
    rec = {"ms_per_step": ms_per_step, "value": value, "pairs": pairs, "peer": peer, "k_alg": k_alg,
           "n_bins": dg.n_bins, "stage_ms": {"l2_flush": flush_ms, "bfs_signature": bfs_ms, "allgather_transpose": gather_ms, "pairwise": pair_ms,
                        "final_barrier": tail_ms},
           "stage_ms_per_rank": per_rank,
           "roofline": roofline, "roofline_bfs": roofline_bfs, "clocks": clocks,
           # ring phase: scatter + hops CDF passes + (hops - 1) OR passes (dense, unfused; the fused build for 32k < N <= 131k
           # launches hops + 2), or one BFS kernel (two with the hub split); then transpose + pairwise
           "launches_per_step": ((2 * hops + 1) if variant == "cols" else
                                 (2 * hops if n <= 32768 or n > 131072 else hops + 2) if variant == "dense"
                                 else (2 if plan.hub_split is not None else 1)) + (2 if plan.n_rows else 1)}
    return rec, plan, dg, block


def workload_config(n, hops, world, peer, n_bins):
    """`config` of the JSON line — identical in the native and the reference arm (the driver compares
    them); the l2 / symmetric / multi_gpu entries describe how the NATIVE arm runs this workload."""
    return {"workload": f"barabasi_albert_graph({n}, 5, seed=0), {hops} hops, degree-valued ring signal, full NxN",
            "n_nodes": n, "hops": hops, "support_bins": int(n_bins), "signature_len": int(1 + hops * (n_bins - 1)),
            "l2": "native arm: 256 MB buffer written before every step (flush) + each step writes a result > L2",
            "symmetric": world == 1 or peer, "sharded_over_gpus": world,
            "multi_gpu": None if world == 1 else (
                "BFS kernel stores each signature row into every rank's table over NVLink peer memory "
                "(fused all-gather, no collective; from 32k nodes: column-split bitmap recursion + one integer all-reduce "
                "of the partial counts); every symmetric tile computed once in the job by the owner of its row or "
                "column block, mirrored store local, direct store into the other owner's row block through NVLink "
                "peer memory (torch symmetric memory allocations)" if peer else
                "independent row blocks (every rank computes rows x all columns); one NCCL all-gather")}


def extra_c1(ctx):
    """BASELINE config 1: model/HSD.py 3-hop distance matrix on the bundled airport graphs through the
    reference-faithful wavelet signal (exact heat kernel, FP64, scipy-W1 semantics), checked against rows /
    the full matrix the UNMODIFIED reference produced (tests/golden/reference_runs.npz; reference CPU
    times measured at survey time on one core: europe 18.1 s, usa 256.2 s)."""
    torch = ctx.torch
    import networkx as nx
    from model import HSD
    gz = np.load(os.path.join(ROOT, "tests", "golden", "graphs.npz"))
    runs = np.load(os.path.join(ROOT, "tests", "golden", "reference_runs.npz"))
    out = []
    for name in ("europe", "usa"):
        nodes = [str(v) for v in gz[f"{name}_nodes"]]
        G = nx.Graph()
        G.add_nodes_from(nodes)
        G.add_edges_from((nodes[u], nodes[v]) for u, v in gz[f"{name}_edges"])
        hop, scale = int(runs[f"{name}_hop"]), float(runs[f"{name}_scale"])
        m = HSD(G, name, scale, hop, "wasserstein", device=ctx.dev)
        m.calculate_structural_distance(scale, approx=False)           # warm-up (cuSOLVER handles, rings)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        D = m.calculate_structural_distance(scale, approx=False)        # float64 ndarray on the host, like the reference
        wall = time.perf_counter() - t0
        n = m.n_node
        if name == "europe":
            ref, got = np.asarray(runs["europe_D"]), D[np.triu_indices(n, 1)]    # the golden holds the upper triangle
        else:
            ref, got = runs["usa_Drows"], D[runs["usa_rows"]]
        diff = np.abs(got - ref)
        big = np.abs(ref) > 1e-3 * np.abs(ref).max()
        err = float(np.max(diff[big] / np.abs(ref[big])))
        ok = bool(np.all(diff <= 1e-5 * np.abs(ref) + 1e-10))       # the parity tests' tolerance (tests/test_gpu_models.py)
        out.append({"graph": name, "n_nodes": n, "hops": hop, "scale": scale, "ms": wall * 1e3,
                    "node_pairs_per_s": n * (n - 1) / 2 / wall, "max_rel_err_vs_reference_output": err,
                    "max_abs_err_vs_reference_output": float(diff.max()), "within_rtol_1e-5_atol_1e-10": ok,
                    "reference_cpu_s_one_core_survey": {"europe": 18.1, "usa": 256.2}[name]})
        del m
    return {"workload": "bundled airport graphs, exact heat-kernel wavelet signal, 3 hops (model/HSD.py:98-114)",
            "dtype": "f64", "cases": out,
            "note": "wall time of HSD.calculate_structural_distance(scale, approx=False) incl. eigh (cuSOLVER), "
                    "the fused wavelet kernel, ring gather + sort, the W1 merge kernel and the copy of the float64 matrix to the host"}


def extra_c4(ctx):
    """BASELINE config 4: MultiHSD heat-kernel wavelets, Chebyshev order 30, 4 scales, 50 000 nodes.
    (i) one 256-column block of hsd_cheb_spmm on rank 0's GPU, with both byte counts; (ii) the whole
    embedding (all 50k impulse columns + ring reduce), impulse columns sharded over the ranks."""
    torch = ctx.torch
    import networkx as nx
    from hsd_b200 import wavelets as wv
    from hsd_b200.graph import powerlaw_graph
    from model import MultiHSD
    n, order, S, hop, C = 50000, 30, 4, 3, 256
    g = powerlaw_graph(n, 5, seed=0)
    lmax = wv.estimate_lmax(g, device=ctx.dev)
    scales = np.exp(np.linspace(np.log(0.01), np.log(40.0 / lmax), S))
    coeffs = np.stack([wv.cheby_coefficients(float(s), lmax, order) for s in scales])
    csr = wv.DeviceCSR(g, ctx.dev)
    C = wv.column_block(n, S)
    work = torch.empty((3, n, C), dtype=torch.float64, device=ctx.dev)
    outb = torch.empty((S, n, C), dtype=torch.float64, device=ctx.dev)
    times = []
    for it in range(4):
        ctx.flush.fill_(1.0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        wv.cheb_wavelet_block(csr, lmax, coeffs, 0, C, 1e-4 / n, work, outb)
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    ms = float(np.median(times[1:]))
    # SURVEY §8(d): every step reads T_{k-1}, T_{k-2}, writes T_k and reads + writes S accumulators;
    # compulsory: the kernel defers accumulation (3 terms at once), i.e. 174 plane sweeps per block at order 30
    bytes_survey = order * (8.0 * g.nnz + 4 * (n + 1) + (3 + 2 * S) * 8.0 * n * C)
    acc_passes = len([k for k in range(2, order + 1) if k % 3 == 2 or k == order])
    bytes_compulsory = order * (8.0 * g.nnz + 4 * (n + 1) + 3 * 8.0 * n * C) + acc_passes * 2 * S * 8.0 * n * C
    del work, outb
    m = MultiHSD(nx.barabasi_albert_graph(n, 5, seed=0), "ba50k", hop, S, device=ctx.dev)
    m.lmax, m.scales, m.CHEB_ORDER = lmax, scales, order
    m._rings()
    torch.cuda.synchronize()
    ctx.barrier()
    t0 = time.perf_counter()
    emb = m.embed_device_sharded(ctx.rank, ctx.world) if ctx.world > 1 else m.embed_device()
    torch.cuda.synchronize()
    full_s = ctx.max_over_ranks(time.perf_counter() - t0)
    rec = {"workload": f"barabasi_albert_graph({n}, 5, seed=0), Chebyshev order {order}, {S} scales in [0.01, 40/lmax], hop {hop}",
           "kernel": "cheb_step_kernel (FP64)", "block_cols": C, "block_ms": ms,
           "frac_hbm_survey_bytes": bytes_survey / (ms * 1e-3) / 1e9 / ctx.hbm_peak,
           "frac_hbm_compulsory_bytes": bytes_compulsory / (ms * 1e-3) / 1e9 / ctx.hbm_peak,
           "gbs_survey_bytes": bytes_survey / (ms * 1e-3) / 1e9, "gbs_compulsory_bytes": bytes_compulsory / (ms * 1e-3) / 1e9,
           "hbm_peak_gbs": ctx.hbm_peak, "peak_source": ctx.hbm_src,
           "full_embedding_s": full_s, "n_gpus": ctx.world,
           "full_embedding": "all 50k impulse columns + ring [sum, mean] reduce"
                             + (", impulse columns sharded over the ranks + one all-gather" if ctx.world > 1 else ""),
           "checksum": float(emb.sum().item())}
    del m, emb
    torch.cuda.empty_cache()
    return rec


def extra_c5(ctx):
    """BASELINE config 5: DynamicHSD on the 100 000-node graph, edges inserted with default_rng(1):
    time of the incremental update against a from-scratch step (1 GPU: structural_distance_update;
    N GPUs: structural_distance_update_sharded)."""
    torch = ctx.torch
    import networkx as nx
    from model import DynamicHSD
    n = 100000
    out = []
    for hop, batches in ((4, (5000,)), (2, (5, 5000))):
        m = DynamicHSD(nx.barabasi_albert_graph(n, 5, seed=0), "ba100k", hop, 1, "wasserstein", signal="degree",
                       device=ctx.dev)

        def update():
            if ctx.world > 1:
                return m.structural_distance_update_sharded(ctx.rank, ctx.world, peer=ctx.peer)
            return m.structural_distance_update()
        update()
        torch.cuda.synchronize()
        ctx.barrier()
        if ctx.world == 1:
            m._D = None          # forget the previous matrix: the next call is a from-scratch step
            m._sig_prev = None
            t0 = time.perf_counter()
            update()
        else:
            t0 = time.perf_counter()
            m._plan.step()       # from scratch on the existing plan (buffers and peer mappings kept)
        torch.cuda.synchronize()
        full_ms = ctx.max_over_ranks((time.perf_counter() - t0) * 1e3)
        rng = np.random.default_rng(1)
        # one untimed 1-edge update first: the first update of a plan pays one-time costs (large temporaries from
        # the caching allocator, peer views, NCCL's first all-reduce of that size) that are not the update's own
        wu = np.random.default_rng(7)
        while True:
            u, v = (int(x) for x in wu.integers(0, n, 2))
            if u != v and not m.graph.has_edge(u, v):
                break
        m.dynamic_add_edges([(u, v)])
        update()
        torch.cuda.synchronize()
        ctx.barrier()
        for k_ins in batches:
            edges = set()
            while len(edges) < k_ins:
                u, v = (int(x) for x in rng.integers(0, n, 2))
                if u != v and not m.graph.has_edge(u, v):
                    edges.add((min(u, v), max(u, v)))
            t0 = time.perf_counter()
            m.dynamic_add_edges(sorted(edges))
            edit_ms = (time.perf_counter() - t0) * 1e3
            ctx.barrier()
            t0 = time.perf_counter()
            update()
            torch.cuda.synchronize()
            upd_ms = ctx.max_over_ranks((time.perf_counter() - t0) * 1e3)
            out.append({"hop": hop, "inserted_edges": k_ins, "affected_rows": int(m.last_affected.numel()),
                        "from_scratch_ms": full_ms, "update_ms": upd_ms, "host_graph_edit_ms": edit_ms})
        del m
        torch.cuda.empty_cache()
    return {"workload": f"barabasi_albert_graph({n}, 5, seed=0) + edge insertions (numpy default_rng(1)), degree signal; "
                        "one untimed 1-edge warm-up update before the timed batches",
            "n_gpus": ctx.world, "cases": out,
            "note": "hop 4: any insertion changes every signature (SURVEY H8), the update is a full recompute; "
                    "wall-clock ms incl. host-side support check"}


def _time_e2e(ctx, step, steps, pairs, pipe, api, host_out):
    torch = ctx.torch
    for _ in range(2):
        step()
    ctx.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    torch.cuda.synchronize()
    mine_ms = (time.perf_counter() - t0) * 1e3 / steps
    e2e_ms = ctx.max_over_ranks(mine_ms)
    ctx.barrier()
    return {"value": pairs / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
            "h2d_bytes_per_step": int(pipe.h2d_bytes), "d2h_bytes_per_step": int(pipe.d2h_bytes),
            "d2h_gbs_this_rank": pipe.d2h_bytes / (mine_ms * 1e-3) / 1e9,
            "d2h_gbs_all_ranks": ctx.world * pipe.d2h_bytes / (e2e_ms * 1e-3) / 1e9,
            "api": api, "cpus_bound_to_gpu_numa_node": ctx.numa,
            "note": "PCIe/host-memory bound: the float32 result (N^2 x 4 B over all ranks) crosses PCIe inside the timed "
                    "region; kernels are ~20 % of it at N = 1 and overlap the copies",
            "checksum": float(host_out[: min(64, pipe.n_rows)].double().sum().item())}


def run_e2e_single(ctx, n, hops, args, pairs):
    """N = 1: literally the call a user of the reference makes — the drop-in class,
    HSD.calculate_structural_distance(scale, out=<pinned host buffer>) -> engine.HostDegreePipeline:
    pinned host CSR -> H2D -> kernels -> D2H of finished row panels overlapped with the panels still computing."""
    torch = ctx.torch
    import networkx as nx
    from model import HSD
    model = HSD(nx.barabasi_albert_graph(n, 5, seed=0), f"ba{n}", 0, hops, "wasserstein", signal="degree")
    host_out = torch.empty((n, n), dtype=torch.float32).pin_memory()

    def step():
        model.calculate_structural_distance(0.0, out=host_out)   # synchronises: the result is in host memory
    step()
    api = "model.HSD(graph, name, 0, hop, metric, signal='degree').calculate_structural_distance(0.0, out=pinned)"
    return _time_e2e(ctx, step, args.steps, pairs, model._host_pipe, api, host_out)


def run_e2e_sharded(ctx, g, hops, plan, args, pairs):
    """N > 1: every rank runs the same host pipeline for its row shard (rows x all columns, panels
    streamed out while later panels compute)."""
    torch = ctx.torch
    from hsd_b200 import engine
    pipe = engine.HostDegreePipeline(g, hops, device=ctx.dev, row0=plan.row0, n_rows=plan.n_rows)
    host_out = torch.empty((pipe.n_rows, g.n), dtype=torch.float32).pin_memory()
    api = "hsd_b200.engine.HostDegreePipeline.run on each rank's row shard (what HSD.calculate_structural_distance(out=) calls)"
    return _time_e2e(ctx, lambda: pipe.run(host_out), args.steps, pairs, pipe, api, host_out)


DUMP_BYTES = 64 * 1000 * 1000     # --dump-outputs: upper bound on the size of the .npy files together


def dump_outputs(ctx, block, row0, n, out_dir):
    """--dump-outputs: what the timed path computed in its last step, as .npy files in out_dir, so that two
    builds of the project can be compared output for output (the workload graph is seeded, so the inputs
    are identical from run to run).  The N x N float32 matrix is too large to store whole; the files are
      distances_rows.npy      float64 [R]     sampled row ids: numpy default_rng(0), sorted; every row when N is small
      distances_sample.npy    float32 [R, N]  those rows of the matrix, as computed
      distances_row_sums.npy  float64 [N]     every row of the matrix summed in float64 (touches the unsampled rows)
    With N > 1 ranks each rank contributes the rows of its block and rank 0 writes the files."""
    torch = ctx.torch
    n_rows = block.shape[0]
    r = max(1, min(n, (DUMP_BYTES - 8 * n - 4096) // (4 * n + 8)))     # 4096: slack for the three .npy headers
    rows = np.sort(np.random.default_rng(0).choice(n, size=r, replace=False))
    sample = torch.zeros((r, n), dtype=torch.float32, device=ctx.dev)
    sums = torch.zeros(n, dtype=torch.float64, device=ctx.dev)
    mine = np.nonzero((rows >= row0) & (rows < row0 + n_rows))[0]
    if mine.size:
        sample[torch.from_numpy(mine).to(ctx.dev)] = block[torch.from_numpy(rows[mine] - row0).to(ctx.dev)]
    for c in range(0, n_rows, 4096):
        end = min(c + 4096, n_rows)
        sums[row0 + c:row0 + end] = block[c:end].sum(1, dtype=torch.float64)
    if ctx.world > 1:      # every row is nonzero on exactly one rank
        ctx.dist.all_reduce(sample)
        ctx.dist.all_reduce(sums)
    if ctx.rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, "distances_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(out_dir, "distances_sample.npy"), sample.cpu().numpy())
        np.save(os.path.join(out_dir, "distances_row_sums.npy"), sums.cpu().numpy())


def run_native(args):
    ctx = Ctx(args)
    torch, dist = ctx.torch, ctx.dist
    from hsd_b200 import engine
    from hsd_b200.graph import powerlaw_graph
    world, rank, dev = ctx.world, ctx.rank, ctx.dev

    n, hops = parse_workload(args.workload)
    g = powerlaw_graph(n, 5, seed=0)       # same deterministic graph on every rank
    rec, plan, dg, block = measure_degree_path(ctx, g, hops, args.steps, args.warmup, args.workload)
    peer = rec["peer"]
    pairs = rec["pairs"]
    if args.dump_outputs:
        dump_outputs(ctx, block, plan.row0, n, args.dump_outputs)
    del block

    # ---- e2e: host buffers in, host matrix out, copies inside the timed region ----
    # N = 1: literally the call a user of the reference makes — the drop-in class,
    # HSD.calculate_structural_distance(scale, out=<pinned host buffer>) — which runs
    # engine.HostDegreePipeline.  N > 1: every rank runs the same pipeline for its row shard.
    if args.no_e2e:
        e2e = None
    elif world == 1:
        e2e = run_e2e_single(ctx, n, hops, args, pairs)
    else:
        e2e = run_e2e_sharded(ctx, g, hops, plan, args, pairs)
    # ---- the other BASELINE.json configs, as sub-records (outside the timed region above) ----
    extras = {}
    want = [] if args.no_extras else [x for x in args.extras.split(",") if x]
    del plan, dg
    torch.cuda.empty_cache()
    for key in want:
        try:
            if key == "c3" and args.workload != "c3":
                g3 = powerlaw_graph(100000, 5, seed=0)
                r3, p3, d3, _ = measure_degree_path(ctx, g3, 4, 3, 1, "c3")
                extras["north_star_c3"] = {
                    "config": workload_config(100000, 4, world, r3["peer"], r3["n_bins"]), "n_gpus": world, "steps": 3, "warmup": 1,
                    "ms_per_step": r3["ms_per_step"], "value": r3["value"], "unit": UNIT, "stage_ms": r3["stage_ms"], "stage_ms_per_rank": r3["stage_ms_per_rank"],
                    "frac": r3["roofline"]["frac"], "roofline": r3["roofline"], "roofline_bfs": r3["roofline_bfs"],
                    "clocks": r3["clocks"]}
                del p3, d3, g3
                torch.cuda.empty_cache()
            elif key == "c1":
                if rank == 0:
                    try:
                        extras["c1"] = extra_c1(ctx)
                    except Exception as e:      # rank-local: must not desynchronise the other ranks
                        extras["c1"] = {"error": f"{type(e).__name__}: {e}"}
            elif key == "c4":
                extras["c4"] = extra_c4(ctx)
            elif key == "c5":
                extras["c5"] = extra_c5(ctx)
        except Exception as e:      # an extra must never take the headline line down with it
            extras[key] = {"error": f"{type(e).__name__}: {e}"}
            if world > 1:
                raise

    # ---- CPU baseline beside it (rank 0, N=1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ref = CpuReference(n, hops, sample_nodes=CPU_SAMPLE_NODES)
        v, d = ref.step()
        ref.close()
        cpu = {"value": v, "unit": UNIT, "cores": ref.cores, "kind": "port", "sample": ref.describe(d)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": rec["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": rec["ms_per_step"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(n, hops, world, peer, rec["n_bins"]),
            "stage_ms": rec["stage_ms"], "stage_ms_per_rank": rec["stage_ms_per_rank"],
            "roofline": rec["roofline"], "roofline_bfs": rec["roofline_bfs"], "cpu_baseline": cpu, "e2e": e2e,
            "gpu_launches": int(args.steps * rec["launches_per_step"]),
            "clocks": rec["clocks"],
        }
        line.update(extras)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="c2")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-peer", action="store_true", help="N>1: independent row blocks instead of peer-memory mirroring")
    ap.add_argument("--extras", default="c1,c3,c4,c5",
                    help="other BASELINE.json configs measured after the headline workload, as sub-records of the line")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer e2e leg (NVLink byte-count runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a seeded sample of the distance matrix the last step computed "
                         "(and its row sums) to DIR/*.npy, at most 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the native arm's outputs; the reference arm computes a sample of pairs only")
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.warmup < 3:
            args.warmup = 3
        run_native(args)


if __name__ == "__main__":
    main()
