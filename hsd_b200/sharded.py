"""Row-block sharding of the degree-mode path over the GPUs of one box.

One process per GPU (torch.distributed, NCCL).  Every D[i, j] depends only on
signature rows i and j (SURVEY.md §8 e).  The RESULT is row-block sharded: rank r
owns rows [r*per, (r+1)*per).  The WORK is dealt differently so that it balances:

* BFS sources are dealt round-robin (node s -> rank s % world; contiguous blocks
  would give one rank all the hubs);
* peer mode (default under bench.py): the signature table and the result blocks are
  torch symmetric-memory allocations mapped into every rank over NVLink.  The BFS
  kernel stores each signature row into all ranks' tables as it is produced (fused
  all-gather), and the pairwise kernel computes each symmetric tile once in the whole
  job and stores it, mirrored, into the owners' blocks.  No collective is issued;
  two device-side barriers per step order the stores;
* fallback (peer=False): ONE in-place NCCL all-gather of the signature table, then
  every rank computes its rows against all columns (twice the arithmetic).

The reference's counterpart is multiprocessing.Pool over rows with the whole
model pickled per task (model/HSD.py:118-137).
"""
from __future__ import annotations

import os
from typing import Tuple

import torch

from . import engine


HUB_DEGREE = 64


def shard_rows(n: int, world: int, rank: int) -> Tuple[int, int, int]:
    """(row0, n_rows, rows_per_rank): contiguous blocks of ceil(n / world) rows rounded up to
    a multiple of 4 (the pairwise kernel's TMA tile origins must be 16-byte aligned), the last
    ranks may own fewer (or zero) rows; rows_per_rank is the all-gather chunk."""
    per = ((n + world - 1) // world + 3) // 4 * 4
    row0 = min(rank * per, n)
    return row0, max(0, min(per, n - row0)), per


def deal_affected(aff: torch.Tensor, n: int, world: int, rank: int):
    """Incremental update: the affected nodes `aff` (ascending ids, identical on every rank) are dealt
    round-robin; returns (dealt, segments) with dealt = aff[rank::world] and segments a list of
    (owner, lo, hi, row0_of_owner): dealt[lo:hi] are the rows owned by `owner` (row blocks are
    contiguous, dealt is ascending, so each owner's share is one slice)."""
    dealt = aff[rank::world].contiguous()
    segments = []
    if dealt.numel():
        bounds = [shard_rows(n, world, r)[0] for r in range(world)] + [n]
        cut = torch.searchsorted(dealt, torch.tensor(bounds, dtype=dealt.dtype, device=dealt.device)).tolist()
        for r in range(world):
            if cut[r + 1] > cut[r]:
                segments.append((r, cut[r], cut[r + 1], bounds[r]))
    return dealt, segments


def agree_status(status: torch.Tensor, world: int, group=None) -> int:
    """OR of every rank's status flags (a MAX all-reduce of the bit field would lose bits, so the
    flags are summed per bit).  world == 1, or no process group: the local value."""
    if world > 1:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            bits = torch.stack([(status.reshape(-1)[0] >> b) & 1 for b in range(8)]).to(torch.int32)
            dist.all_reduce(bits, op=dist.ReduceOp.SUM, group=group)
            return int(sum((1 << b) for b, v in enumerate(bits.tolist()) if v))
    return int(status.reshape(-1)[0].item())


def agree_all(flag: bool, world: int, group=None, device=None) -> bool:
    """True on every rank iff `flag` is true on every rank (a MIN all-reduce); world == 1, or no process
    group: the local value.  Used for decisions that select which collectives the ranks issue next."""
    if world > 1:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            t = torch.tensor([1 if flag else 0], dtype=torch.int32, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MIN, group=group)
            return bool(t.item())
    return bool(flag)


def agree_min(values, group=None, device=None):
    """Element-wise MIN over the ranks of a list of integers (one int64 all-reduce): the value every rank
    uses for a decision that must not differ between ranks, such as a plan derived from free memory."""
    import torch.distributed as dist
    t = torch.tensor([int(v) for v in values], dtype=torch.int64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MIN, group=group)
    return [int(v) for v in t.tolist()]


def agree_radius_cap(nnz: int, stopped: bool, max_pairs: int, radius, group=None, device=None) -> int:
    """Global nnz of a radius graph swept by several ranks: one SUM all-reduce of (this rank's nnz, whether it
    stopped at the cap).  Raises the same ValueError (engine.radius_cap_error) on every rank when the sum
    exceeds max_pairs or any rank stopped; a rank past the cap must still join, or the others would hang."""
    import torch.distributed as dist
    t = torch.tensor([int(nnz), 1 if stopped else 0], dtype=torch.int64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    total, n_stopped = t.tolist()
    if n_stopped or total > max_pairs:
        raise engine.radius_cap_error(radius, total, max_pairs)
    return total


def gather_csr_parts(indptr: torch.Tensor, idx: torch.Tensor, val: torch.Tensor, world: int, group=None):
    """Every rank's CSR (indptr int64[N+1] from 0, idx[nnz_r], val[nnz_r]) on every rank, without padding:
    one all_gather_into_tensor of the indptrs gives each rank's entry count, then each rank's entries are
    broadcast into its exact slice of one buffer per array (ranks with no entries are skipped by all ranks
    alike).  Returns (part_indptr int64[world, N+1], part_base int64[world]: where rank r's entries start,
    idx_all, val_all), on the inputs' device (any device the group's backend serves)."""
    import torch.distributed as dist
    me = dist.get_rank(group)
    part_indptr = torch.empty(world * indptr.numel(), dtype=torch.int64, device=indptr.device)
    dist.all_gather_into_tensor(part_indptr, indptr.contiguous(), group=group)
    part_indptr = part_indptr.view(world, indptr.numel())
    sizes = part_indptr[:, -1].tolist()
    starts = [0]
    for c in sizes:
        starts.append(starts[-1] + c)
    idx_all = torch.empty(starts[-1], dtype=idx.dtype, device=idx.device)
    val_all = torch.empty(starts[-1], dtype=val.dtype, device=val.device)
    for r in range(world):
        if not sizes[r]:
            continue
        for mine, out in ((idx, idx_all), (val, val_all)):
            piece = out[starts[r]:starts[r + 1]]
            if r == me:
                piece.copy_(mine)
            dist.broadcast(piece, group=group, group_src=r)
    part_base = torch.tensor(starts[:-1], dtype=torch.int64).to(indptr.device)
    return part_indptr, part_base, idx_all, val_all


def cols_workspace_words(n: int, world: int) -> int:
    """Workspace words (hsd_ring_cols_workspace_words) of the column-split ring phase on the rank that
    owns the most bitmap pieces: the same number on every rank."""
    from ._lib import lib as _lib_
    return max(int(_lib_.hsd_ring_cols_workspace_words(n, *engine.ring_cols_range(n, r, world)))
               for r in range(world))


def symmetric_tile_list(n: int, world: int, per: int, rank: int, tile_n: int = 128):
    """Rank `rank`'s share of the upper-triangle 128 x 128 tiles of the N x N matrix, as int32[m, 3] rows
    {first row, first column, mirror flag} of 128 x tile_n tiles (tile_n = 64 splits every tile in two).

    Every tile {I, J} is computed by the owner of row block I or of row block J (checkerboard on I + J, then
    a rebalancing pass that moves tiles between their two possible owners until every rank has the same
    count), and is ORIENTED so that its mirrored store — the short-run one — lands in the computing rank's
    own block and only the direct store (256-byte runs) crosses NVLink.  Against round-robin dealing
    (hsd_pairwise_l1_sharded) that halves the peer traffic and removes every 32-byte remote write.
    Deterministic: every rank derives the same global assignment."""
    import numpy as np
    T = (n + 127) // 128
    I, J = np.triu_indices(T)
    own = lambda t: np.minimum(t * 128 // per, world - 1)
    oI, oJ = own(I), own(J)
    comp = np.where(((I + J) & 1) == 0, oI, oJ)
    cnt = np.bincount(comp, minlength=world).astype(np.int64)
    target = -(-len(I) // world)
    for _ in range(10 * world):                 # move tiles from the fullest rank to their other possible owner
        hi = int(cnt.argmax())
        if cnt[hi] <= target:
            break
        cand = np.nonzero((comp == hi) & (oI != oJ))[0]
        other = np.where(oI[cand] == hi, oJ[cand], oI[cand])
        moved = False
        for r in np.argsort(cnt, kind="stable"):
            if cnt[r] >= target or r == hi:
                continue
            c = cand[other == r]
            k = int(min(len(c), cnt[hi] - target, target - cnt[r]))
            if k > 0:
                comp[c[:k]] = r
                cnt[hi] -= k
                cnt[r] += k
                moved = True
                break
        if not moved:
            break
    mine = comp == rank
    I, J, by_row_owner = I[mine], J[mine], (comp == oI)[mine]
    # rows of the listed tile = the REMOTE block (direct store), columns = the local block (mirrored store)
    X = np.where(by_row_owner, J, I)
    Y = np.where(by_row_owner, I, J)
    order = np.lexsort((Y, X))                 # consecutive tiles share their A rows (L2)
    X, Y = X[order], Y[order]
    mirror = (X != Y).astype(np.int64)
    if tile_n == 128:
        out = np.stack([X * 128, Y * 128, mirror], 1)
    else:
        lo = np.stack([X * 128, Y * 128, mirror], 1)
        hi_half = np.stack([X * 128, Y * 128 + 64, mirror], 1)
        hi_half = hi_half[hi_half[:, 1] < n]
        out = np.concatenate([lo, hi_half])
        out = out[np.lexsort((out[:, 1], out[:, 0]))]
    return torch.from_numpy(np.ascontiguousarray(out.astype(np.int32)))


class ShardedDegreeHSD:
    """Plan + buffers for repeated evaluation of one graph on `world` ranks."""

    def __init__(self, dg: engine.DeviceGraph, hops: int, rank: int = 0, world: int = 1,
                 group=None, empty: str = "raise", peer: bool = False, peer_blocks=None,
                 peer_tables=None, reuse: "ShardedDegreeHSD" = None):
        """peer=True (world > 1): the result blocks are allocated as symmetric memory and mapped
        into every rank over NVLink; the pairwise kernel then computes each symmetric tile once
        in the whole job and stores its mirror straight into the owner's block
        (hsd_pairwise_l1_sharded).  peer=False: every rank computes its full row block.
        The signature table is symmetric memory as well and the BFS kernel stores every row it
        produces into all ranks' copies (hsd_ring_signature_degree_allgather), so no collective is
        issued at all — only two barriers per step.
        peer_blocks / peer_tables: lists of `world` local tensors standing in for the peers'
        result blocks / signature tables (single-GPU emulation in the tests).
        reuse: a previous plan of the same node count / rank / world / peer mode whose symmetric-memory
        allocations (result block, and the signature table when the new one fits its capacity) are
        taken over instead of allocated and rendezvous-ed again — what an incremental update needs
        when an insertion adds a distinct degree and every signature changes length."""
        self.dg, self.hops, self.rank, self.world, self.group, self.empty = dg, hops, rank, world, group, empty
        n = dg.n
        dev = dg.rowptr.device
        self.row0, self.n_rows, self.per = shard_rows(n, world, rank)
        self.k_used = dg.k_used(hops)
        self.ld = engine.roundup(self.k_used, 4)
        # row-major signature table, padded to world * per rows so every rank's chunk is equal
        self.peer = bool(peer) and world > 1
        self.sig_symm = None
        self.sig_peer_ptrs = None
        if self.peer and peer_tables is not None:
            self.sig_all = peer_tables[rank]
            self.sig_peer_ptrs = torch.tensor([t.data_ptr() for r, t in enumerate(peer_tables) if r != rank],
                                              dtype=torch.int64, device=dev)
        elif self.peer and peer_blocks is None:
            import torch.distributed as dist
            import torch.distributed._symmetric_memory as symm_mem
            need = world * self.per * self.ld
            ok = (reuse is not None and reuse.peer and reuse.sig_symm is not None and reuse.world == world
                  and reuse.rank == rank and reuse.dg.n == n and getattr(reuse, "_sig_flat", None) is not None
                  and reuse._sig_flat.numel() >= need)
            if ok:
                self._sig_flat, self.sig_symm = reuse._sig_flat, reuse.sig_symm
                dist.barrier(group=group)  # nobody is still storing rows of the old layout into it
            else:
                # capacity for a few more distinct degrees per hop than the graph has now
                cap = world * self.per * engine.roundup(self.k_used + 16 * hops, 4)
                self._sig_flat = symm_mem.empty((cap,), dtype=torch.float32, device=dev)
                self.sig_symm = symm_mem.rendezvous(self._sig_flat, group if group is not None else dist.group.WORLD)
            self._sig_flat.zero_()
            self.sig_all = self._sig_flat[:need].view(world * self.per, self.ld)
            self.sig_peer_ptrs = torch.tensor([int(p) for r, p in enumerate(self.sig_symm.buffer_ptrs) if r != rank],
                                              dtype=torch.int64, device=dev)
            torch.cuda.synchronize(dev)
            dist.barrier(group=group)      # every table is zeroed before any peer may store into it
        else:
            self.sig_all = torch.zeros((world * self.per, self.ld), dtype=torch.float32, device=dev)
        self.sigT = engine.alloc_signature_table(self.k_used, n, dev)
        self.side = None
        # Ring phase across ranks.  "cols": every rank runs the dense bitmap recursion for ALL nodes on its own
        # 1/world of the bitmap columns (no exchange), the partial integer counts are summed by ONE all-reduce and
        # every rank builds the whole signature table from the sums — 1/world of the ring work per rank instead
        # of the intermediate levels being recomputed everywhere.  Needs a real process group and is taken from
        # 32k nodes (below, the phase is latency-bound and the frontier / dense-by-rows kernels win);
        # HSD_RING_SHARD_MODE=cols|rows overrides.
        self.ring_mode = "rows"
        if world > 1 and peer_blocks is None and peer_tables is None and hops >= 1:
            import torch.distributed as dist
            want = os.environ.get("HSD_RING_SHARD_MODE", "cols" if n >= 32768 else "rows")
            if want == "cols" and dist.is_available() and dist.is_initialized():
                # the two modes issue different collectives, so every rank must take the same one
                if agree_all(self._cols_workspace_fits(), world, group, dev):
                    self.ring_mode = "cols"
        self.update_mode = os.environ.get("HSD_DYN_PEER_MODE", "rows")   # see update_finish()
        self._plan_sources(dg)
        node = torch.arange(n, dtype=torch.int32, device=dev)
        self.table_row = ((node % world) * self.per + node // world).to(torch.int32).contiguous()
        self.sizes = torch.zeros((world * self.per, hops + 1), dtype=torch.int32, device=dev)
        self.status = torch.zeros(1, dtype=torch.int32, device=dev)
        self.launches_per_step = 3
        self.symm = None
        self.ld_out = engine.roundup(n, 4)
        if self.peer and peer_blocks is not None:
            self.blocks = peer_blocks
            self.out_full = peer_blocks[rank]
            self.ptrs = torch.tensor([b.data_ptr() for b in peer_blocks], dtype=torch.int64, device=dev)
        elif self.peer:
            import torch.distributed as dist
            import torch.distributed._symmetric_memory as symm_mem
            if (reuse is not None and reuse.peer and reuse.symm is not None and reuse.world == world
                    and reuse.rank == rank and reuse.dg.n == n):
                self.out_full, self.symm = reuse.out_full, reuse.symm      # the result block does not depend on the support
            else:
                self.out_full = symm_mem.empty((self.per, self.ld_out), dtype=torch.float32, device=dev)
                self.symm = symm_mem.rendezvous(self.out_full, group if group is not None else dist.group.WORLD)
            self.ptrs = torch.tensor([int(p) for p in self.symm.buffer_ptrs], dtype=torch.int64, device=dev)
        self.tile_list = None
        if self.peer and os.environ.get("HSD_PAIR_SHARD_TILES", "owner") == "owner":
            # tiles dealt to the owners of their row / column blocks, mirrored store local (symmetric_tile_list);
            # 128 x 64 tiles when a rank has few tiles per CTA slot, like the single-GPU dispatch
            sms = torch.cuda.get_device_properties(dev).multi_processor_count
            t128 = ((n + 127) // 128) * ((n + 127) // 128 + 1) // 2 // world
            self.tile_n = 64 if t128 < sms * 2 * 8 else 128
            self.tile_list = symmetric_tile_list(n, world, self.per, rank, self.tile_n).to(dev)
        if self.peer:
            self.out = self.out_full[:max(self.n_rows, 1), :n]
        else:
            self._out = None      # allocated on first use: a plan that only builds signatures never needs it

    @property
    def out(self) -> torch.Tensor:
        """This rank's result rows (non-peer mode: float32[n_rows, N], allocated on first use)."""
        if self._out is None:
            self._out = torch.empty((max(self.n_rows, 1), self.dg.n), dtype=torch.float32,
                                    device=self.dg.rowptr.device)
        return self._out

    @out.setter
    def out(self, value: torch.Tensor) -> None:
        self._out = value

    def _cols_workspace_fits(self) -> bool:
        """This rank's vote for the column-split ring phase.  It keeps two N x (N / world)-bit tables per rank:
        take it only when the largest rank's tables fit in a quarter of this device's free memory (the rule
        engine.ring_algorithm applies to the dense variant); otherwise the row-split phase runs, with the same
        signatures.  The ranks combine their votes with agree_all."""
        words = cols_workspace_words(self.dg.n, self.world)
        dev = self.dg.rowptr.device
        ws = engine._DENSE_WS.get(("cols", dev.index if dev.index is not None else torch.cuda.current_device()))
        have = ws.numel() * 4 if ws is not None else 0     # this rank's cached tables are reused / replaced
        if have >= words * 4:
            return True
        free, _ = torch.cuda.mem_get_info(dev)
        return words * 4 <= (free + have) // 4

    def _plan_sources(self, dg: engine.DeviceGraph) -> None:
        """Deal this rank's BFS sources for graph `dg` (called again by update(): the degree order,
        hence the relabelled source ids and the hubs, change with the graph)."""
        n, rank, world = dg.n, self.rank, self.world
        dev = dg.rowptr.device
        # BFS sources are DEALT round-robin (node s -> rank s % world): contiguous blocks would give
        # one rank all the hubs of a preferential-attachment graph (its BFS then takes 2x longer).
        # Table row of node s in the gathered table: (s % world) * per + s // world.
        self.all_src = dg.new_of.contiguous()      # every node, original order -> degree-order id (cols mode)
        self.rows = torch.arange(rank, n, world, dtype=torch.int32, device=dev)
        self.n_src = int(self.rows.numel())
        self.src = dg.new_of[self.rows.long()].contiguous()
        self.out_rows = (rank * self.per + torch.arange(self.n_src, dtype=torch.int32, device=dev)).contiguous()
        # Latency regime (few sources per rank): one hub source is latency-bound inside its CTA and sets
        # the floor of the whole BFS phase, so hubs (degree > HUB_DEGREE) get 1024-thread CTAs on a side
        # stream while the rest run with the default CTA size.
        self.hub_split = None
        # (not when the BFS bitmaps live in the shared global workspace: two concurrent launches would race on it)
        from ._lib import lib as _lib_
        if 0 < self.n_src <= 4096 and int(_lib_.hsd_bfs_workspace_words(n)) == 0:
            deg = (dg.rowptr[1:] - dg.rowptr[:-1])[self.src.long()]
            hub = deg > HUB_DEGREE
            if bool(hub.any()) and not bool(hub.all()):
                self.hub_split = (self.src[hub].contiguous(), self.out_rows[hub].contiguous(),
                                  self.src[~hub].contiguous(), self.out_rows[~hub].contiguous())
                if self.side is None:
                    self.side = torch.cuda.Stream(device=dev)

    def ring_sizes(self) -> torch.Tensor:
        """int32[N, hops+1] in node order (valid after gather for world > 1 only for own sources)."""
        return self.sizes[self.table_row.long()] if self.world > 1 else self.sizes[:self.dg.n]

    def signatures(self) -> None:
        """BFS + degree CDF for this rank's sources, written straight into its slice of the
        gathered table."""
        from ._lib import check, lib
        dg = self.dg
        if self.ring_mode == "cols":
            import torch.distributed as dist
            self._counts = engine.ring_counts_cols(dg, self.hops, self.rank, self.world,
                                                   getattr(self, "_counts", None))
            dist.all_reduce(self._counts, op=dist.ReduceOp.SUM, group=self.group)
            engine.signature_from_counts(dg, self.hops, self._counts, self.all_src, self.table_row, self.sig_all,
                                         self.sizes, self.empty, self.status)
            return
        if self.n_src == 0:
            return
        engine.ensure_bfs_workspace(dg.n, dg.rowptr.device)

        def launch(src, out_rows, threads, stream):
            if self.sig_peer_ptrs is not None:
                check(lib.hsd_ring_signature_degree_allgather(
                    engine._ptr(dg.rowptr), engine._ptr(dg.col), dg.n, engine._ptr(src),
                    engine._ptr(out_rows), int(src.numel()), self.hops,
                    engine._ptr(dg.bin_end), engine._ptr(dg.delta), dg.n_bins,
                    engine._ptr(self.sig_all), self.ld, engine._ptr(self.sig_peer_ptrs),
                    int(self.sig_peer_ptrs.numel()), engine._ptr(self.sizes),
                    1 if self.empty == "zero" else 0, engine._ptr(self.status), threads, stream))
            else:
                check(lib.hsd_ring_signature_degree(
                    engine._ptr(dg.rowptr), engine._ptr(dg.col), dg.n, engine._ptr(src),
                    engine._ptr(out_rows), int(src.numel()), self.hops,
                    engine._ptr(dg.bin_end), engine._ptr(dg.delta), dg.n_bins,
                    engine._ptr(self.sig_all), self.ld, engine._ptr(self.sizes), None,
                    1 if self.empty == "zero" else 0, engine._ptr(self.status), threads, stream))

        if engine.ring_algorithm(dg.n, self.n_src, self.hops, dg.rowptr.device) == "dense":
            # (world <= 2) most nodes are this rank's sources: bitmap dynamic programming over all nodes,
            # signature rows stored into the peers' tables by its CDF pass like the frontier kernel does
            engine.launch_ring_signature(dg.rowptr, dg.col, dg.n, dg.nnz, self.src, self.out_rows, self.n_src,
                                         self.hops, dg.bin_end, dg.delta, dg.n_bins, self.sig_all, self.ld,
                                         self.sizes, None, 1 if self.empty == "zero" else 0, self.status,
                                         dg.rowptr.device, peers=self.sig_peer_ptrs)
            return
        if self.hub_split is None:
            launch(self.src, self.out_rows, 0, engine._stream())
            return
        hub_src, hub_rows, rest_src, rest_rows = self.hub_split
        cur = torch.cuda.current_stream()
        self.side.wait_stream(cur)
        launch(hub_src, hub_rows, 1024, self.side.cuda_stream)
        launch(rest_src, rest_rows, 0, cur.cuda_stream)
        cur.wait_stream(self.side)

    def gather(self) -> None:
        """Make every rank's signature table complete: a barrier in peer mode (the rows were
        already stored by the BFS kernels), else the in-place NCCL all-gather."""
        if self.world == 1 or self.ring_mode == "cols":
            return      # cols: the all-reduce left the complete table on every rank
        if self.sig_peer_ptrs is not None:
            # the rows were already stored into every rank's table by the BFS kernel: only wait
            if self.sig_symm is not None:
                self.sig_symm.barrier()
            return
        import torch.distributed as dist
        chunk = self.sig_all[self.rank * self.per:(self.rank + 1) * self.per]
        dist.all_gather_into_tensor(self.sig_all, chunk, group=self.group)

    def distances(self, ev_before=None, ev_after=None) -> torch.Tensor:
        """Transpose the gathered table to K-major and run the pairwise kernel; the optional
        CUDA events bracket the pairwise launch alone (bench.py's roofline timing)."""
        out = self._distances(ev_before)
        if ev_after is not None:
            ev_after.record()
        if self.peer:
            self.peer_barrier()
        return out

    def _distances(self, ev_before) -> torch.Tensor:
        n = self.dg.n
        engine.signature_transpose(self.sig_all, self.k_used, self.sigT, 0,
                                   src_rows=None if self.world == 1 else self.table_row)
        if ev_before is not None:
            ev_before.record()
        if self.peer:
            from ._lib import check, lib
            if self.tile_list is not None:
                check(lib.hsd_pairwise_l1_tile_list(engine._ptr(self.sigT), self.k_used, self.sigT.stride(0), n,
                                                    engine._ptr(self.tile_list), int(self.tile_list.shape[0]),
                                                    self.tile_n, self.per, engine._ptr(self.ptrs), self.ld_out,
                                                    engine._stream()))
            else:
                check(lib.hsd_pairwise_l1_sharded(engine._ptr(self.sigT), self.k_used, self.sigT.stride(0),
                                                  n, self.rank, self.world, self.per, engine._ptr(self.ptrs),
                                                  self.ld_out, engine._stream()))
            return self.out[:self.n_rows]
        if self.n_rows == 0:
            return self.out[:0]
        if self.world == 1:
            return engine.pairwise_l1(self.sigT, n, symmetric=True, out=self.out, k_used=self.k_used)
        return engine.pairwise_l1(self.sigT, n, self.row0, self.n_rows, 0, n, symmetric=False, out=self.out,
                                  k_used=self.k_used)

    def peer_barrier(self) -> None:
        """A block is complete only when every rank's launch has stored its tiles into it."""
        if self.symm is not None:
            self.symm.barrier()
        elif self.world > 1 and not hasattr(self, "blocks"):
            import torch.distributed as dist
            dist.barrier(group=self.group)

    # ------------------------------------------------------------------
    # incremental update after edge insertions (BASELINE config 5; SURVEY.md §8 e "Dynamic")
    # ------------------------------------------------------------------
    def update(self, dg_new: engine.DeviceGraph) -> Tuple[torch.Tensor, torch.Tensor]:
        """This rank's row block of the distance matrix of `dg_new` (same node set, edges inserted),
        recomputing only what changed; returns (block, affected node ids).  See update_finish()."""
        self.update_begin(dg_new)
        self.gather()
        return self.update_finish()

    def update_begin(self, dg_new: engine.DeviceGraph) -> None:
        """Keep a copy of the gathered signature table, then rebuild this rank's dealt signatures on
        the edited graph (the BFS kernel stores them into every rank's table in peer mode)."""
        import numpy as np
        if dg_new.n != self.dg.n or not np.array_equal(dg_new.support, self.dg.support):
            raise ValueError("update() needs the same node set and the same set of distinct degrees: every "
                             "signature changes representation otherwise; build a new plan and step() it")
        self.sig_prev = self.sig_all.clone()
        if self.sig_symm is not None:
            self.sig_symm.barrier()     # no peer stores new rows into a table that is still being copied
        self.dg = dg_new
        self._plan_sources(dg_new)
        self.signatures()

    def update_finish(self) -> Tuple[torch.Tensor, torch.Tensor]:
        """After gather(): the exact affected set A = nodes whose signature row differs bit for bit
        from the previous table (identical on every rank: the tables are replicated), then

        * peer mode, update_mode "rows" (default) — every rank recomputes the COLUMNS A of its own row
          block locally; the ROWS of A are dealt round-robin (A[rank::world]), computed against all N
          columns and stored whole into their owners' blocks through NVLink peer memory (contiguous
          rows: coalesced stores).  2·|A|·N distances in the job, balanced even when A falls into one
          rank's row block;
        * peer mode, update_mode "mirror" (HSD_DYN_PEER_MODE=mirror; also the one-GPU case) — dealt
          rows only, each also stored mirrored as a column into every rank's block: |A|·N distances,
          but the mirrored half is a scatter of 4-byte peer stores;
        * fallback (peer=False) — each rank recomputes own rows x A columns and (A ∩ own rows) x all
          columns locally: no traffic, 2·|A|·N distances, unbalanced if A is concentrated.

        2|A| >= N falls back to the symmetric full matrix.  Bit-equal to a from-scratch step(): every
        entry comes from the same kernel and the same signature rows, and |a - b| == |b - a|."""
        n, dev = self.dg.n, self.sig_all.device
        changed = (self.sig_all != self.sig_prev).any(dim=1)
        self.sig_prev = None
        aff = torch.nonzero(changed[self.table_row.long()], as_tuple=False).reshape(-1)   # node ids, ascending
        self.last_affected = aff
        m = int(aff.numel())
        if m == 0:
            if self.peer:
                self.peer_barrier()
            return self.out[:self.n_rows], aff
        if 2 * m >= n:
            return self.distances(), aff
        n4 = engine.roundup(n, 4)
        mode = "local"
        if self.world == 1:
            mode = "mirror"                       # one GPU: its own block is the only "peer"
        elif self.peer:
            mode = self.update_mode               # "rows" (default) or "mirror"
        k = self.k_used
        tbl_all = self.table_row

        def direct_rows(dealt, segments, blk):
            """Full rows (contiguous, coalesced peer stores) of the dealt affected nodes -> their owners."""
            views = self._block_views()
            for r, lo, hi, r0 in segments:
                views[r][:, :n].index_copy_(0, dealt[lo:hi] - r0, blk[lo:hi])

        if mode == "mirror":
            # table = [all nodes | dealt affected nodes]; each distance computed once in the job; the
            # mirrored half is a 4-byte scatter into every block (peer stores when world > 1)
            dealt, segments = deal_affected(aff, n, self.world, self.rank)
            mq = int(dealt.numel())
            if mq:
                sigT = engine.alloc_signature_table(k, n4 + mq, dev)
                engine.signature_transpose(self.sig_all, k, sigT, 0, src_rows=tbl_all)
                engine.signature_transpose(self.sig_all, k, sigT, n4, src_rows=tbl_all[dealt].contiguous())
                blk = engine.pairwise_l1(sigT, n4 + mq, row0=n4, n_rows=mq, col0=0, n_cols=n, symmetric=False, k_used=k)
                if self.world == 1:
                    engine.scatter_symmetric(blk, dealt, self.out)
                else:
                    for r, Dr in enumerate(self._block_views()):
                        r0, nr, _ = shard_rows(n, self.world, r)
                        if nr:
                            Dr[:nr].index_copy_(1, dealt, blk[:, r0:r0 + nr].t())
                    direct_rows(dealt, segments, blk)
        elif mode == "rows":
            # table = [all nodes | all affected nodes | pad | dealt affected nodes]: the COLUMNS of the
            # affected nodes are recomputed by every rank for its own rows (local scatter); their ROWS are
            # dealt round-robin and stored whole into the owners' blocks (coalesced peer stores)
            dealt, segments = deal_affected(aff, n, self.world, self.rank)
            mq = int(dealt.numel())
            m4 = engine.roundup(m, 4)
            sigT = engine.alloc_signature_table(k, n4 + m4 + max(mq, 1), dev)
            engine.signature_transpose(self.sig_all, k, sigT, 0, src_rows=tbl_all)
            engine.signature_transpose(self.sig_all, k, sigT, n4, src_rows=tbl_all[aff].contiguous())
            n_tab = sigT.shape[1]
            if self.n_rows:
                rect = engine.pairwise_l1(sigT, n_tab, row0=self.row0, n_rows=self.n_rows, col0=n4, n_cols=m,
                                          symmetric=False, k_used=k)
                self.out[:self.n_rows].index_copy_(1, aff, rect)
            if mq:
                engine.signature_transpose(self.sig_all, k, sigT, n4 + m4, src_rows=tbl_all[dealt].contiguous())
                blk = engine.pairwise_l1(sigT, n_tab, row0=n4 + m4, n_rows=mq, col0=0, n_cols=n, symmetric=False,
                                         k_used=k)
                direct_rows(dealt, segments, blk)
        elif self.n_rows:
            # no peer memory: own rows x affected columns, then (affected ∩ own rows) x all columns
            sigT = engine.alloc_signature_table(k, n4 + m, dev)
            engine.signature_transpose(self.sig_all, k, sigT, 0, src_rows=tbl_all)
            engine.signature_transpose(self.sig_all, k, sigT, n4, src_rows=tbl_all[aff].contiguous())
            rect = engine.pairwise_l1(sigT, n4 + m, row0=self.row0, n_rows=self.n_rows, col0=n4, n_cols=m,
                                      symmetric=False, k_used=k)
            self.out[:self.n_rows].index_copy_(1, aff, rect)
            lo, hi = (int(x) for x in torch.searchsorted(aff, torch.tensor([self.row0, self.row0 + self.n_rows],
                                                                            device=dev)))
            if hi > lo:
                lo4 = lo // 4 * 4       # TMA tile origins are 16-byte aligned
                rows = engine.pairwise_l1(sigT, n4 + m, row0=n4 + lo4, n_rows=hi - lo4, col0=0, n_cols=n,
                                          symmetric=False, k_used=k)
                self.out.index_copy_(0, aff[lo:hi] - self.row0, rows[lo - lo4:])
        if self.peer:
            self.peer_barrier()
        return self.out[:self.n_rows], aff

    def _block_views(self):
        """Every rank's result block as a tensor on this device (peer mode)."""
        if hasattr(self, "blocks"):
            return self.blocks
        if self.world == 1:
            return [self.out]
        if getattr(self, "_views", None) is None:
            self._views = [self.out_full if r == self.rank else
                           self.symm.get_buffer(r, (self.per, self.ld_out), torch.float32)
                           for r in range(self.world)]
        return self._views

    def step(self) -> torch.Tensor:
        self.signatures()
        self.gather()
        return self.distances()

    def check(self) -> None:
        """Raise where scipy would (an empty ring under empty='raise') — on EVERY rank: the BFS
        kernel flags only the sources dealt to this rank, so the flags are OR-ed over the ranks
        first; otherwise the ranks that own no such source would carry on with a block built from
        all-zero signature rows and hang at the next barrier once the raising rank is gone."""
        if self.empty != "raise":
            return
        flags = agree_status(self.status, self.world if not hasattr(self, "blocks") else 1, self.group)
        if flags & 1:
            raise engine.EmptyRingError("Distribution can't be empty.")
