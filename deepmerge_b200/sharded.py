"""Row-tile sharding of one scene across the GPUs of a box (SURVEY.md section 8(e)).

Rank g owns rows [g*H/G, (g+1)*H/G) of labels / image plus ONE halo row below: the vertical
pixel pair (y, y+1) belongs to the tile that owns y, so nothing is counted twice.  Region ids
are global.  torch.distributed is the plumbing (NCCL on the GPUs; the same code runs against the
in-process stand-in of the tests).

`ShardedMergeEngine.run` -- distributed merge loop, no rank ever holds the whole graph:
  * every rank keeps ITS TILE's edge list (the edges physically inside the tile) and scores,
    selects, re-keys and uniques only those;
  * per-region small state is replicated: the parent array (int32 [R]), point counts, the alive /
    changed flags and a rank-visibility bit mask (bit g = rank g sees the region: it has pixels
    or an edge of it).  A component can span two tiles only through a region both ranks see, so
    after its local unions a rank publishes (shared region, local root) pairs -- the frontier --
    and every rank unites all ranks' pairs into its own forest; one all-reduce(MIN) of the parent
    array then fills in the regions a rank does not see.  No iteration, no convergence test;
  * embedding sums [R, D] are NOT replicated: a rank holds the rows of the regions it sees.  Rows
    travel sparsely: once for the regions seen by two ranks (their per-tile partial sums are
    added in rank order), and per round for the members of components that grew across a tile
    border (shipped by the lowest rank that held the row), as fixed-capacity slots with
    device-side counts (dm_rows_pack / exchange / dm_rows_unpack);
  * area / border / perimeter / band sums stay per-tile partials through the loop (every update
    is linear) and are all-reduced once at the end together with the gathered final edge list.
Integer outputs are bit-identical to the single-GPU result; the fp32 sums of regions whose points
lie in two tiles are added in rank order instead of point order (last-bit differences).

Transport: under torch.distributed over NCCL, when the symmetric-memory rendezvous succeeds, the
slots are exchanged by peer stores of this library's kernels (PeerSlots) and the two replicated
R-sized arrays are all-reduced by its peer kernels (PeerArray), so a step calls no collective and
the round body is one CUDA graph launch.  Otherwise (gloo, the tests' in-process stand-in, a box
without peer access) slots travel by all_gather_into_tensor and the arrays by all_reduce.
"""
from __future__ import annotations

import json
import time
from typing import Optional

import torch


def tile_bounds(H: int, world: int, rank: int):
    """Rows [y0, y1) owned by `rank`; tiles differ by at most one row."""
    base, extra = divmod(H, world)
    y0 = rank * base + min(rank, extra)
    y1 = y0 + base + (1 if rank < extra else 0)
    return y0, y1


def gather_edge_lists(keys: torch.Tensor, lens: torch.Tensor, dist, group=None):
    """all_gather of variable-length per-tile edge lists -> (keys_cat, lens_cat) with the valid
    entries of every rank in rank order.  Lengths are exchanged first, payloads are padded."""
    world = dist.get_world_size(group)
    n = torch.tensor([keys.shape[0]], dtype=torch.int64, device=keys.device)
    counts = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(counts, n, group=group)
    counts = [int(c.item()) for c in counts]
    m = max(max(counts), 1)
    pk = torch.zeros(m, dtype=keys.dtype, device=keys.device)
    pl = torch.zeros(m, dtype=lens.dtype, device=lens.device)
    pk[: keys.shape[0]] = keys
    pl[: lens.shape[0]] = lens
    gk = [torch.empty_like(pk) for _ in range(world)]
    gl = [torch.empty_like(pl) for _ in range(world)]
    dist.all_gather(gk, pk, group=group)
    dist.all_gather(gl, pl, group=group)
    return torch.cat([g[:c] for g, c in zip(gk, counts)]), torch.cat([g[:c] for g, c in zip(gl, counts)])


def allreduce_sum_(t: torch.Tensor, dist, group=None):
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


def points_in_tile(ys: torch.Tensor, y0: int, y1: int):
    """Indices of the sample points whose row falls in [y0, y1): they go with that tile."""
    return torch.nonzero((ys >= y0) & (ys < y1)).flatten()


def all_gather_slots(t: torch.Tensor, dist, group=None):
    """all_gather of equal-sized slots into one tensor [world * len(t)] (one NCCL call, no host sync)."""
    world = dist.get_world_size(group)
    out = torch.empty(world * t.shape[0], dtype=t.dtype, device=t.device)
    if hasattr(dist, "all_gather_into_tensor"):
        dist.all_gather_into_tensor(out, t.contiguous(), group=group)
    else:                                             # minimal stand-ins used by tests
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t.contiguous(), group=group)
        out.copy_(torch.cat(parts))
    return out


class PeerSlots:
    """Gathered slot buffers [world x slot_bytes] in torch symmetric memory: every rank's buffer is mapped into every
    process, so an exchange is ONE kernel of this library storing the rank's slot into all peers over NVLink
    (dm_peer_put_slot) plus a signal-pad barrier -- no collective call.  Two buffers alternate: a buffer is rewritten
    only after every rank has passed the barrier that follows its last read."""

    def __init__(self, dist, group, slot_bytes, device):
        import torch.distributed._symmetric_memory as symm
        world = dist.get_world_size(group)
        name = (group if group is not None else dist.group.WORLD).group_name
        self.slot_bytes, self.world = slot_bytes, world
        self.bufs = []
        for _ in range(2):
            t = symm.empty(world * slot_bytes, dtype=torch.uint8, device=device)
            h = symm.rendezvous(t, name)
            bases = torch.tensor([int(p) for p in h.buffer_ptrs], dtype=torch.int64, device=device)
            t.zero_()
            self.bufs.append((t, h, bases))
        torch.cuda.synchronize(device)
        self.bufs[0][1].barrier()
        self.k = 0

    def exchange(self, L, slot, rank, header_bytes, seg0, seg1, capacity, stream, buf):
        """slot -> every rank's gathered buffer `buf` (0 / 1); returns this rank's gathered view [world, slot_bytes].
        The caller names the buffer (the loop's head uses 0, its round body 1), so that a captured round body replays
        on the same addresses; two uses of one buffer are always separated by a barrier of the other exchange."""
        from .raster import _p
        t, h, bases = self.bufs[buf]
        L.check(L.dm_peer_put_slot(_p(slot), _p(bases), self.world, rank, self.slot_bytes, header_bytes, seg0[0], seg0[1],
                                   seg1[0], seg1[1], capacity, stream), "dm_peer_put_slot")
        h.barrier()
        return t.view(self.world, self.slot_bytes)


class PeerArray:
    """An int32 array in torch symmetric memory (every rank's copy is mapped into every process) with an in-place
    all-reduce made of this library's kernel over NVLink peer loads / stores (dm_peer_allreduce_i32: rank g reduces
    slice g of all copies and stores it into all of them) between two signal-pad barriers -- no NCCL call."""

    def __init__(self, dist, group, n, device):
        import torch.distributed._symmetric_memory as symm
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        name = (group if group is not None else dist.group.WORLD).group_name
        self.n_pad = n + (-n) % 4
        self.buf = symm.empty(self.n_pad, dtype=torch.int32, device=device)
        self.hdl = symm.rendezvous(self.buf, name)
        self.bases = torch.tensor([int(p) for p in self.hdl.buffer_ptrs], dtype=torch.int64, device=device)
        self.buf.zero_()
        self.tensor = self.buf[:n]
        torch.cuda.synchronize(device)
        self.hdl.barrier()

    def all_reduce(self, L, op, stream):
        """op 0 = sum, 1 = min; in place, on the current stream."""
        from .raster import _p
        self.hdl.barrier()                 # every rank's copy is complete (its producers precede the barrier in stream order)
        L.check(L.dm_peer_allreduce_i32(_p(self.bases), self.world, self.rank, 0, self.n_pad, op, stream),
                "dm_peer_allreduce_i32")
        self.hdl.barrier()                 # every slice has landed everywhere


def _peer_exchange_possible(dist):
    """Symmetric memory needs the real torch.distributed over NCCL (one process per GPU)."""
    try:
        import torch.distributed as td
        return dist is td and td.is_initialized() and td.get_backend() == "nccl"
    except Exception:
        return False


class ShardedMergeEngine:
    """One rank's share of a scene sharded by rows.  Wraps a MergeEngine sized for the tile.

    A step makes no host round trip before the merge loop's own read-back: rows and frontier pairs
    travel as fixed-capacity slots together with their device-side counts, and overflow / bad-label
    flags of the tile pass are checked with that first read-back."""

    def __init__(self, H, W, n_regions, D, C, n_points_local, dist, device, group=None, row_capacity=None,
                 edge_capacity=None):
        from .raster import MergeEngine, default_edge_capacity
        self.dist, self.group = dist, group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        if self.world > 31:          # every rank checks alike: the rank-visibility masks are 31 bits of an int32
            raise ValueError("ShardedMergeEngine supports at most 31 ranks (got %d)" % self.world)
        self.H, self.W = H, W
        self.row_capacity = row_capacity
        self.y0, self.y1 = tile_bounds(H, self.world, self.rank)
        self.rows_own = self.y1 - self.y0
        self.has_halo = self.rank < self.world - 1
        # capacity: the raw per-tile entries of THIS tile must fit (an even share of the regions plus 50 %; a scene
        # whose regions crowd into one tile needs edge_capacity=...).  Kernel grids of the graph stages are sized by it.
        cap = int(edge_capacity) if edge_capacity else min(
            default_edge_capacity(n_regions, H, W),
            default_edge_capacity(int(1.5 * n_regions / self.world) + 1024, self.rows_own + 1, W))
        self.eng = MergeEngine(self.rows_own, W, n_regions, D, C=C, n_points=n_points_local, edge_capacity=cap,
                               device=device)
        self.cat_counts = torch.zeros(2, dtype=torch.int64, device=self.eng.dev)

    # ------------------------------------------------------------------------------------------------
    # distributed merge loop
    # ------------------------------------------------------------------------------------------------
    def _alloc_dist(self):
        e = self.eng
        dev, R, D = e.dev, e.R, e.D
        # frontier / cross-component rows per rank and exchange (overflow is detected and reported)
        self.row_cap = int(self.row_capacity) if self.row_capacity else int(min(R, max(4096, self.W // 2)))
        self.row_cap += (-self.row_cap) % 4                        # 16-byte aligned segments inside the slots
        z = lambda *sh, dt: torch.zeros(*sh, dtype=dt, device=dev)
        self.seen, self.grew, self.send, self.seen_comp = (z(R, dt=torch.uint8) for _ in range(4))
        self.mask_old = z(R, dt=torch.int32)
        self.cnt_local = z(R, dt=torch.int32)
        self.mask_cnt = z(2 * R, dt=torch.int32)                   # [mask | cnt]: one all-reduce
        self.mask = self.mask_cnt[:R]
        self.agreed = z(R, dt=torch.int32)
        # one exchange slot = [count (16 B) | ids | rows] in ONE byte buffer: a single all_gather per exchange
        self.slot_bytes = 16 + 4 * self.row_cap + 4 * self.row_cap * D
        self.slot_bytes += (-self.slot_bytes) % 16
        self.slot = z(self.slot_bytes, dt=torch.uint8)
        self.slot_n = self.slot[:8].view(torch.int64)
        self.slot_ids = self.slot[16:16 + 4 * self.row_cap].view(torch.int32)
        self.slot_rows = self.slot[16 + 4 * self.row_cap:16 + 4 * self.row_cap * (D + 1)].view(torch.float32).view(self.row_cap, D)
        # [0] selected, [1] parent changed, [2] row-slot overflow, [3] tile edge-list overflow, [4] bad label, [5] internal
        # error, [6] raw entries needed -- [0] and [2:7] are all-reduced with MAX once per round, so that every rank raises
        # (or goes on) together: a rank that left the loop alone would leave its peers hanging in the next collective
        # frontier pairs of the distributed union-find: [count | pad | pairs] per rank, one all_gather per round
        # [count | pad | 8 flag words | pairs]: the round's flags travel with the pairs
        self.fslot_bytes = 80 + 8 * self.row_cap
        self.fslot_bytes += (-self.fslot_bytes) % 16
        self.fslot = z(self.fslot_bytes, dt=torch.uint8)
        self.fslot_flags = self.fslot[16:80].view(torch.int64)
        self.flags = z(8, dt=torch.int64)
        # peer transport: both slot exchanges, and the two replicated R-sized arrays in symmetric memory so that their
        # all-reduces are peer kernels -- all four or none
        self.peer_rows = self.peer_pairs = self.peer_mask_cnt = self.peer_parent = None
        if _peer_exchange_possible(self.dist):
            try:
                rows = PeerSlots(self.dist, self.group, self.slot_bytes, dev)
                pairs = PeerSlots(self.dist, self.group, self.fslot_bytes, dev)
                pm, pp = PeerArray(self.dist, self.group, 2 * R, dev), PeerArray(self.dist, self.group, R, dev)
            except Exception as ex:                                # no NVLink peer access / symmetric memory on this box
                self.peer_error = repr(ex)
            else:
                self.peer_rows, self.peer_pairs, self.peer_mask_cnt, self.peer_parent = rows, pairs, pm, pp
                self.mask_cnt, self.mask = pm.tensor, pm.tensor[:R]
                e.parent = pp.tensor
        e.sum.zero_()                                              # rows the pooling pass never writes start as zeros
        self._last_fg = None
        self.any_selected = z(1, dt=torch.int64)
        self.host_fflags = torch.zeros((self.world, 10), dtype=torch.int64).pin_memory()
        self.hdr_dev = z(self.world, 80, dt=torch.uint8)
        self.host_flags = torch.zeros(8, dtype=torch.int64).pin_memory()

    def _exchange_rows(self, flag, add, buf):
        """Ship the embedding sums of the flagged regions to every rank: pack -> all_gather (fixed slots + device
        counts) -> unpack slot by slot in rank order (add: partial sums are accumulated in that order)."""
        from .raster import _p, _stream
        e, L, dist, s = self.eng, self.eng.L, self.dist, _stream()
        L.check(L.dm_rows_pack(_p(flag), _p(e.sum), e.R, e.D, _p(self.slot_ids), _p(self.slot_rows), self.row_cap,
                               _p(self.slot_n), s), "dm_rows_pack")
        rc = self.row_cap
        if self.peer_rows is not None:     # one kernel storing the used part of the slot into every peer + a barrier
            g = self.peer_rows.exchange(L, self.slot, self.rank, 16, (16, 4), (16 + 4 * rc, 4 * e.D), rc, s, buf)
        else:
            g = all_gather_slots(self.slot, dist, self.group).view(self.world, self.slot_bytes)
        # a slot that overflowed on ANY rank is seen by every rank in the gathered counts: all of them flag it
        L.check(L.dm_slots_overflow(_p(g), self.world, self.slot_bytes, rc, self.flags[2:3].data_ptr(), s), "dm_slots_overflow")
        g_n = [g[r, :8].view(torch.int64) for r in range(self.world)]
        g_ids = [g[r, 16:16 + 4 * rc].view(torch.int32) for r in range(self.world)]
        g_rows = [g[r, 16 + 4 * rc:16 + 4 * rc * (e.D + 1)].view(torch.float32) for r in range(self.world)]
        if add:       # partial sums: clear every row that receives one, then add slot by slot (= in rank order)
            L.check(L.dm_rows_unpack_slots(_p(g), self.world, self.slot_bytes, rc, e.R, e.D, _p(e.sum), 1, s), "dm_rows_unpack_slots")
            for r in range(self.world):
                L.check(L.dm_rows_unpack(_p(g_ids[r]), _p(g_rows[r]), _p(g_n[r]), rc, e.R, e.D, _p(e.sum), 1, s),
                        "dm_rows_unpack")
        else:         # whole rows from their single sender: one launch for all slots
            L.check(L.dm_rows_unpack_slots(_p(g), self.world, self.slot_bytes, rc, e.R, e.D, _p(e.sum), 0, s), "dm_rows_unpack_slots")

    def _read_headers(self, gathered, after_enqueue=None):
        """The round's one host read-back: the slot headers of all ranks ([count, pad, 8 flags] each) and this rank's
        engine counters.  after_enqueue() runs between the enqueue of the copies and the wait for them."""
        self.hdr_dev.copy_(gathered[:, :80])                       # one strided copy of the headers, then one to the host
        self.host_fflags.copy_(self.hdr_dev.view(torch.int64).view(self.world, 10), non_blocking=True)
        c = self.eng._read_counts(after_enqueue)
        return self.host_fflags.tolist(), c

    def _pre_exchange(self, rule, do_unions, first_round, buf):
        """Selection of the round, its local unions and the ONE exchange of the round -> gathered frontier slots.

        The union-find of the round is prepared BEFORE anyone knows whether the round takes place: local unions, then the
        frontier pairs (shared component, its local root).  The pairs of all ranks carry the whole cross-tile connectivity
        -- no iteration, no convergence test -- and the round's flags ("edges selected", errors) travel in the same slot.
        (Nothing selected anywhere: no unions, no pairs.)"""
        from .raster import _p, _stream
        e, L, s = self.eng, self.eng.L, _stream()
        R, cap = e.R, e.cap
        rule.select(e)
        if do_unions:
            L.check(L.dm_uf_union(_p(e.parent), _p(e.keys), _p(e.selected), _p(e.n_edges), cap, s), "dm_uf_union")
            L.check(L.dm_uf_compress(_p(e.parent), R, s), "dm_uf_compress")
            L.check(L.dm_shard_frontier_pairs(_p(e.parent), _p(e.alive), _p(self.mask), self.rank, R, _p(self.fslot),
                                              self.row_cap, s), "dm_shard_frontier_pairs")
        else:
            self.fslot[:16].zero_()
        # the round's flags (edges selected; first round: this rank's tile-pass conditions) -> the slot header
        L.check(L.dm_shard_round_flags(_p(e.counts), _p(self.flags), int(first_round), _p(self.fslot_flags), s),
                "dm_shard_round_flags")
        if self.peer_pairs is not None:                     # one kernel of NVLink peer stores + a barrier
            fg = self.peer_pairs.exchange(L, self.fslot, self.rank, 80, (80, 8), (80, 0), self.row_cap, s, buf)
        else:
            fg = all_gather_slots(self.fslot, self.dist, self.group).view(self.world, self.fslot_bytes)
        # "did any rank select an edge" on the device: the gate of the relabel that follows the read-back's copy
        L.check(L.dm_slots_word_max(_p(fg), self.world, self.fslot_bytes, 16, _p(self.any_selected), s), "dm_slots_word_max")
        return fg

    def _dist_round_body(self, rule, do_unions, fg):
        """One round between two read-backs: unions from everybody's frontier pairs, rows of the components that grew
        across a tile border, merged statistics, re-keyed tile edge list, means / scores of what changed, and the next
        round's selection + exchange."""
        from .raster import _p, _stream
        e, L, dist, grp, s = self.eng, self.eng.L, self.dist, self.group, _stream()
        R = e.R
        L.check(L.dm_uf_union_slots(_p(e.parent), _p(fg), self.world, self.fslot_bytes, self.row_cap, R, s),
                "dm_uf_union_slots")
        L.check(L.dm_uf_compress(_p(e.parent), R, s), "dm_uf_compress")
        if self.peer_parent is not None:                   # fills in the regions this rank does not see
            self.peer_parent.all_reduce(L, 1, s)
        else:
            dist.all_reduce(e.parent, op=dist.ReduceOp.MIN, group=grp)
        # rows of components that grew across a tile border go to every rank that now sees them
        self.mask_old.copy_(self.mask)
        L.check(L.dm_shard_propagate(_p(e.parent), _p(e.alive), _p(self.mask), _p(self.grew), R, s), "dm_shard_propagate")
        L.check(L.dm_shard_plan(_p(e.parent), _p(e.alive), _p(self.mask_old), _p(self.mask), _p(self.grew), self.rank, R,
                                _p(self.send), _p(self.seen_comp), s), "dm_shard_plan")
        self._exchange_rows(self.send, add=False, buf=1)
        rule.merge_and_rescore(e, self.seen_comp)          # embedding sums only of the components this rank sees
        return self._pre_exchange(rule, do_unions, False, 1)

    def _dist_round(self, rule, do_unions):
        """The round body; one CUDA graph launch when every exchange in it is a kernel of this library (peer stores /
        peer all-reduce over symmetric memory + signal-pad barriers): collective calls cannot be captured."""
        # the body reads the gathered pairs of the previous exchange: buffer 0 after the head, buffer 1 after a body
        src = self._last_fg
        body = lambda: self._dist_round_body(rule, do_unions, src)
        if self.peer_rows is None:
            self._last_fg = body()
        else:
            self._last_fg = self.eng._graph_launch(body, rule, bool(do_unions), src.data_ptr())
        return self._last_fg

    def run(self, labels_tile, feats_local, tau, *, image_tile=None, xs_local=None, ys_local_rel=None, max_rounds=64,
            gather_outputs=True, mlp=None):
        """labels_tile: int32 [rows_own (+1 halo), W]; ys_local_rel are rows relative to the tile.

        The result is DISTRIBUTED unless gather_outputs: labels = this tile's label map, root / cnt replicated,
        edge_keys / boundary_len = this tile's final edge list (the global list is the union, lengths add up),
        area / perimeter (and the engine's band sums) = this tile's partials (they add up over ranks), sum = rows of
        the regions this rank sees.  gather_outputs=True all-reduces the statistics and gathers + uniques the edge
        lists so that every rank holds the same MergeResult a single GPU would produce.

        mlp (a PackedMLP, replicated on every rank): the tcgen05 pair-MLP scores every live tile edge every round and an edge
        is selected when argmax(o) == 1 (Nets.py:28-35) instead of L2 distance < tau -- as MergeEngine.run(mlp=...) does."""
        from .raster import _EDGES, _MERGED, MergeResult, _EmbeddingRule, _p, _stream
        e, L, dist, grp = self.eng, self.eng.L, self.dist, self.group
        rule = _EmbeddingRule(tau, mlp)
        R, D, cap = e.R, e.D, e.cap
        if not hasattr(self, "mask"):
            self._alloc_dist()
        MIN, MAX, SUM = dist.ReduceOp.MIN, dist.ReduceOp.MAX, dist.ReduceOp.SUM
        # ids are global: most regions have no point in this tile.  Their sum rows are never read here (a row is read only
        # for a region with points of its own, a received partial / shipped row, or a merge -- and a region without sample
        # points never merges), so the pooling pass visits only the id interval that holds the tile's points instead of
        # zero-filling R x D floats per step.
        e.pool_id_range = True
        with torch.cuda.device(e.dev):
            s = _stream()
            # (1) tile pass: fused RAG + band pooling; e.keys / e.blen = the tile's own edge list,
            #     e.perim = border + incident boundary lengths of THIS tile (a partial, like area and the band sums)
            #     (the tile's point pooling only needs the labels: it runs beside the raster pass on the engine's side stream)
            cur = torch.cuda.current_stream(e.dev)
            e.side.wait_stream(cur)
            with torch.cuda.stream(e.side):
                e._pool(labels_tile, xs_local, ys_local_rel, None, feats_local)
            e._rag(labels_tile, image_tile, self.rows_own, self.rank == 0, self.rank == self.world - 1)
            # (2) which ranks see which region
            self.seen.zero_()
            L.check(L.dm_mark_endpoints(_p(e.keys), _p(e.n_edges), cap, R, _p(self.seen), s), "dm_mark_endpoints")
            # (3) pooled embeddings: per-tile partial sums; counts replicated, rows of regions seen by two ranks exchanged
            cur.wait_stream(e.side)
            L.check(L.dm_shard_seen(_p(e.area), _p(self.seen), _p(e.cnt), self.rank, R, _p(self.mask_cnt), _p(self.cnt_local), s),
                    "dm_shard_seen")
            if self.peer_mask_cnt is not None:                      # masks: distinct bits, the sum is the OR; counts add up
                self.peer_mask_cnt.all_reduce(L, 0, s)
            else:
                dist.all_reduce(self.mask_cnt, op=SUM, group=grp)
            self.flags.zero_()
            L.check(L.dm_shard_frontier(_p(self.mask_cnt), _p(self.cnt_local), R, _p(e.cnt), _p(self.send), s), "dm_shard_frontier")
            self._exchange_rows(self.send, add=True, buf=0)
            # (4) merge loop on the tile's edges with the replicated parent array
            rule.prepare(e)
            e._merge_init()
            L.check(L.dm_region_mean(_p(e.sum), _p(e.cnt), R, D, _p(e.mean), _p(e.norm2), _p(self.seen), s), "dm_region_mean")
            rule.score(e, None)
            rounds = merges = 0
            fg = self._last_fg = self._pre_exchange(rule, max_rounds > 0, True, 0)
            # (5) tile-local relabel with the replicated root LUT: enqueued behind every exchange, right after the copies the
            #     host waits for, and gated on the device by "no rank selected an edge" -- when the loop ends it is already
            #     running, when it goes on the kernel returns at once
            gated_relabel = lambda: e._relabel_gated(labels_tile, self.rows_own,
                                                     None if rounds == max_rounds else self.any_selected)
            while True:
                hf, c = self._read_headers(fg, gated_relabel)
                f = [max(int(h[2 + k]) for h in hf) for k in range(8)]     # every rank sees every rank's flags: all act alike
                if f[4] != 0:
                    raise ValueError("labels contain ids >= n_regions")
                if f[5] != 0 or f[3] != 0:
                    raise RuntimeError("tile edge list overflow / pipeline error (capacity %d, needed %d)" % (cap, f[6]))
                if f[2] != 0 or any(int(h[0]) > self.row_cap for h in hf):
                    raise RuntimeError("row exchange slot overflow (row_cap %d)" % self.row_cap)
                merges += int(c[_MERGED])
                if f[0] == 0 or rounds == max_rounds:
                    break
                rounds += 1
                fg = self._dist_round(rule, rounds < max_rounds)
            Ef = int(e.host_counts[_EDGES])
            if gather_outputs:
                # per-tile partials -> global statistics; tile edge lists -> the global final edge list
                allreduce_sum_(e.stats, dist, grp)                  # area | border | band sums | perimeter in one buffer
                nmax = e.n_edges.clone()
                dist.all_reduce(nmax, op=MAX, group=grp)
                m = max(1, int(nmax.item()))                        # (the gathered form may afford this host round trip)
                gk = all_gather_slots(e.keys[:m], dist, grp)
                gl = all_gather_slots(e.blen[:m], dist, grp)
                gc = all_gather_slots(e.n_edges, dist, grp)
                tot = self.world * m
                out_k = torch.empty(tot, dtype=torch.int64, device=e.dev)
                out_l = torch.empty(tot, dtype=torch.int32, device=e.dev)
                n_out = torch.zeros(2, dtype=torch.int64, device=e.dev)
                L.check(L.dm_edges_concat(_p(gk), _p(gl), _p(gc), self.world, m, _p(out_k), _p(out_l), tot, _p(self.cat_counts), s),
                        "dm_edges_concat")
                wsb = L.dm_edges_unique_workspace_bytes(tot)
                ws = torch.empty(wsb, dtype=torch.uint8, device=e.dev)
                L.check(L.dm_edges_sort_unique(_p(out_k), _p(out_l), _p(self.cat_counts), tot, R, _p(n_out), _p(ws), wsb, s),
                        "dm_edges_sort_unique")
                Ef = int(n_out[0].item())
                return MergeResult(e.out[: self.rows_own], e.parent, rounds, merges, out_k[:Ef], out_l[:Ef], None, e.area,
                                   e.perim, e.sum, e.cnt)
        return MergeResult(e.out[: self.rows_own], e.parent, rounds, merges, e.keys[:Ef], e.blen[:Ef], None, e.area,
                           e.perim, e.sum, e.cnt)


# ----------------------------------------------------------------------------------------------
# bench leg for N > 1 (launched by torchrun, one rank per GPU)
# ----------------------------------------------------------------------------------------------
SHARDED_CFG = dict(H=40000, W=40000, R=1000000, C=4, P=4, D=100, tau=0.5, seed=1234)
SHARDED_WORKLOAD = "configs[2]: 40k x 40k scene, ~1M segments, row-tile sharded across N B200 (frontier exchange and peer all-reduce over NVLink symmetric memory)"


def position_checksum(t, first=0, chunk=1 << 24):
    """64-bit position-weighted checksum of an integer tensor (wraps mod 2^64): sum over i of (t[i] + 2) * w(first + i),
    w a fixed odd-multiplier hash of the global position -- so that equal checksums of a tile and of the same rows of a
    whole map mean equal contents in equal places.  Device tensor in, Python int out."""
    flat = t.reshape(-1)
    acc = torch.zeros((), dtype=torch.int64, device=t.device)
    for a in range(0, flat.numel(), chunk):
        v = flat[a:a + chunk].to(torch.int64)
        idx = torch.arange(first + a, first + a + v.numel(), dtype=torch.int64, device=t.device)
        w = ((idx * 0x9E3779B1 + 0x7F4A7C15) & 0xFFFFFFFF) | 1
        acc += ((v + 2) * w).sum()
    return int(acc.item())


def bench_sharded(args, cfg1, workload1, dist, dev, ClockSampler, measured_peaks, emit=True):
    """Weak scaling: every rank owns a tile of H_1 x W_1 / ... -- the N-GPU scene is the single-GPU
    workload's height times N (same tile per GPU), so per-GPU work is fixed as N grows."""
    import numpy as np
    from . import _lib
    from .synth import grid_pitch, synth_scene
    from .raster import _p, _stream, points_region

    world, rank = dist.get_world_size(), dist.get_rank()
    L = _lib.lib()
    cfg = dict(cfg1)
    if args.side:
        cfg.update(H=args.side, W=args.side, R=max(4, int(round(cfg1["R"] * args.side * args.side / (cfg1["H"] * cfg1["W"])))))
    # weak scaling: N tiles of the single-GPU scene stacked vertically
    H, W, C, D, P = cfg["H"] * world, cfg["W"], cfg["C"], cfg["D"], cfg["P"]
    R_target = cfg["R"] * world
    fixed_scene = bool(getattr(args, "config2", False))
    if fixed_scene:                       # BASELINE.json configs[2]: ONE 40k x 40k scene split over the ranks (strong scaling)
        cfg = dict(SHARDED_CFG)
        H, W, C, D, P, R_target = cfg["H"], cfg["W"], cfg["C"], cfg["D"], cfg["P"], cfg["R"]
    y0, y1 = tile_bounds(H, world, rank)
    has_halo = rank < world - 1
    sc = synth_scene(H, W, R_target, C=C, P=P, D=D, seed=cfg["seed"], device=dev, rows=(y0, y1 + (1 if has_halo else 0)))
    R = sc.n_regions
    mine = points_in_tile(sc.ys, y0, y1)
    xs, ys_rel = sc.xs[mine].contiguous(), (sc.ys[mine] - y0).contiguous()
    # embeddings of the tile's points (region_of_point from the tile's own labels)
    rop = points_region(sc.labels[: y1 - y0], xs, ys_rel)
    feats = torch.empty((xs.shape[0], D), dtype=torch.float32, device=dev)
    # feats are hashed per GLOBAL point id so that the scene does not depend on the sharding
    SL = _lib.synth_lib()
    SL.check(SL.dm_synth_feats(_p(feats), _p(rop), _p(sc.region_obj), _p(mine.contiguous()), xs.shape[0], D, cfg["seed"],
                               _stream()), "dm_synth_feats")
    image = sc.image[: y1 - y0] if sc.image is not None else None
    eng = ShardedMergeEngine(H, W, R, D, C, xs.shape[0], dist, dev)

    def step(gather=False):
        return eng.run(sc.labels, feats, cfg["tau"], image_tile=image, xs_local=xs, ys_local_rel=ys_rel, gather_outputs=gather)

    for _ in range(max(args.warmup, 3)):
        res = step()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = L.dm_launch_count()
    with ClockSampler(dev.index) as clocks:
        dist.barrier()
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(args.steps):
            res = step()
        ev1.record()
        torch.cuda.synchronize()
        dist.barrier()
    ms_local = ev0.elapsed_time(ev1) / args.steps
    launches = L.dm_launch_count() - launches0
    # the same with the statistics all-reduced and the final edge list gathered on every rank
    k_g = max(1, args.steps // 2)
    step(True)
    dist.barrier()
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(k_g):
        step(True)
    ev1.record()
    torch.cuda.synchronize()
    t = torch.tensor([ms_local, ev0.elapsed_time(ev1) / k_g], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_gathered = float(t[0].item()), float(t[1].item())

    # end to end with HOST buffers on every rank (tile H2D, label-map tile D2H inside the timed region)
    host = {"labels": sc.labels.cpu().pin_memory(), "image": image.cpu().pin_memory(), "feats": feats.cpu().pin_memory(),
            "xs": xs.cpu().pin_memory(), "ys": ys_rel.cpu().pin_memory()}
    out_host = torch.empty((y1 - y0, W), dtype=torch.int32).pin_memory()
    h2d = sum(v.numel() * v.element_size() for v in host.values())

    # every rank pipelines its own tile: the H2D of step k+1 and the D2H of step k-1 overlap step k (ScenePipeline)
    from .raster import ScenePipeline
    pipe = ScenePipeline(eng.eng, run_fn=lambda d, tau, **kw: eng.run(d["labels"], d["feats"], tau, image_tile=d["image"],
                                                                       xs_local=d["xs"], ys_local_rel=d["ys"],
                                                                       gather_outputs=False))
    n_e2e = max(3, args.steps // 2)
    for _ in pipe.run((host for _ in range(2)), cfg["tau"]):
        pass
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in pipe.run((host for _ in range(n_e2e)), cfg["tau"]):
        pass
    torch.cuda.synchronize()
    dist.barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / n_e2e
    eng.eng.out = pipe.dev_out[0]
    # what the host side can deliver when all ranks copy at once (copies only, no compute): the ceiling of the e2e figure
    def link_gbs(fn, nbytes, reps=3):
        fn()
        torch.cuda.synchronize()
        dist.barrier()
        t1 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        return nbytes * reps / (time.perf_counter() - t1) / 1e9
    dev_in = {k: torch.empty_like(v, device=dev) for k, v in host.items()}
    dev_lab = torch.empty((y1 - y0, W), dtype=torch.int32, device=dev)
    link_h2d = link_gbs(lambda: [dev_in[k].copy_(host[k], non_blocking=True) for k in host], h2d)
    link_d2h = link_gbs(lambda: out_host.copy_(dev_lab, non_blocking=True), out_host.numel() * 4)
    del dev_in, dev_lab
    t = torch.tensor([e2e_ms, float(h2d), float(out_host.numel() * 4)], dtype=torch.float64, device=dev)
    lk = torch.tensor([link_h2d, link_d2h], dtype=torch.float64, device=dev)
    lk_min = lk.clone()
    dist.all_reduce(lk_min, op=dist.ReduceOp.MIN)
    tmax = t.clone()
    dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    # the dominant kernel (fused raster pass over this rank's tile) alone, CUDA events
    rows_t = y1 - y0
    rk0 = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    rk1 = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    e = eng.eng
    for i in range(5):
        e.stats.zero_()
        rk0[i].record()
        L.check(L.dm_rag_scan(_p(sc.labels), rows_t, sc.labels.shape[0], W, W, _p(image), C, W * C, R, int(rank == 0),
                              int(rank == world - 1), _p(e.area), _p(e.border), _p(e.bsum), _p(e.bsq), e.cap, _p(e.counts),
                              _p(e.ws), e.ws_bytes, _stream()), "scan")
        rk1[i].record()
    torch.cuda.synchronize()
    rag_ms = float(np.mean([a.elapsed_time(b) for a, b in zip(rk0[1:], rk1[1:])]))
    res = step()
    # ---- parity of the multi-process answer (outside every timed region): position-weighted checksums of every
    # rank's label tile and root table against ONE GPU running the single-GPU engine over the whole scene
    mine_cs = torch.tensor([position_checksum(res.labels, y0 * W), position_checksum(res.root), res.rounds, res.merges],
                           dtype=torch.int64, device=dev)
    all_cs = [torch.zeros_like(mine_cs) for _ in range(world)]
    dist.all_gather(all_cs, mine_cs)
    parity_ok, parity_note = None, "skipped (--no-parity)"
    if rank == 0 and not getattr(args, "no_parity", False):
        from .raster import MergeEngine
        try:
            whole = synth_scene(H, W, R_target, C=C, P=P, D=D, seed=cfg["seed"], device=dev)
            eng1 = MergeEngine(H, W, R, D, C=C, n_points=whole.feats.shape[0], device=dev)
            one = eng1.run(whole.labels, whole.feats, cfg["tau"], image=whole.image, xs=whole.xs, ys=whole.ys)
            root_cs = position_checksum(one.root)
            bad = []
            for r in range(world):
                a, b = tile_bounds(H, world, r)
                want = [position_checksum(one.labels[a:b], a * W), root_cs, one.rounds, one.merges]
                if [int(x) for x in all_cs[r].tolist()] != want:
                    bad.append(r)
            parity_ok = not bad
            parity_note = ("label tiles, root table, rounds and merges of all %d ranks equal the single-GPU engine's on the "
                           "whole %dx%d scene (64-bit position-weighted checksums)" % (world, H, W)) if parity_ok else \
                          "MISMATCH on ranks %s" % bad
            del whole, eng1, one
            torch.cuda.empty_cache()
        except torch.OutOfMemoryError:
            parity_note = "skipped: the whole scene does not fit one GPU beside this rank's tile"
    line = None
    if rank == 0:
        peak, kind = measured_peaks()
        alg = (4 + C) * rows_t * W + 12 * (3 * R // world) + 16 * (R // world) * C
        n_roots = int((res.root == torch.arange(R, device=dev, dtype=torch.int32)).sum())
        line = {
            "metric": "megapixels/sec end-to-end (RAG+pool+score+merge+relabel)", "value": H * W / ms / 1e3, "unit": "Mpx/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong" if fixed_scene else "weak", "vs_baseline": None, "dtype": "int32/u8 index + fp32 scores",
            "data": "synthetic",
            "config": {"workload": (SHARDED_WORKLOAD if fixed_scene else
                                    f"{workload1} -- one such tile per GPU, stacked by rows ({H}x{W}), row-tile sharded: frontier "
                                    "exchange, peer-store slots and peer all-reduce over NVLink symmetric memory"),
                       "H": H, "W": W, "bands": C, "segments": R,
                       "points": int(sc.xs.shape[0]), "embed_dim": D, "tau": cfg["tau"], "parallelism": f"row-tiles x{world}",
                       "result_form": "distributed (tile label maps, replicated root LUT, per-rank partial region statistics and "
                                      "tile edge lists); ms_per_step_gathered = with the statistics all-reduced and the final "
                                      "edge list gathered on every rank",
                       "l2_policy": "inputs larger than L2, no flush needed"},
            "merged_edges_per_s": res.merges / (ms * 1e-3), "segments_after": n_roots, "rounds": res.rounds,
            "parity_ok": parity_ok, "parity": parity_note,
            "ms_per_step_gathered": ms_gathered,
            "e2e": {"value": H * W / float(tmax[0]) / 1e3, "unit": "Mpx/s", "ms_per_step": float(tmax[0]),
                    "h2d_bytes_per_step": int(t[1]), "d2h_bytes_per_step": int(t[2]),
                    "api": "ScenePipeline over ShardedMergeEngine.run: every rank overlaps its tile's H2D / compute / D2H",
                    "per_gpu_h2d_gbs": h2d / (float(tmax[0]) * 1e-3) / 1e9, "per_gpu_d2h_gbs": out_host.numel() * 4 / (float(tmax[0]) * 1e-3) / 1e9,
                    "copy_only_h2d_gbs_per_gpu_all_ranks_at_once": float(lk_min[0]),
                    "copy_only_d2h_gbs_per_gpu_all_ranks_at_once": float(lk_min[1]),
                    "note": "copy_only_* = pinned host <-> device copies of the same buffers with every rank copying at the same "
                            "time and nothing else running (slowest rank): the host side's ceiling for this step"},
            "gpu_launches": int(launches),
            "roofline": {"kernel": "rag_blocks_kernel (fused RAG + band pooling raster pass), rank 0's tile", "bound": "hbm",
                         "achieved": alg / (rag_ms * 1e-3) / 1e9, "peak": peak, "peak_kind": kind, "unit": "GB/s",
                         "frac": alg / (rag_ms * 1e-3) / 1e9 / peak, "ms": rag_ms, "algorithmic_bytes": alg, "traffic": None},
            "cpu_baseline": None, "clocks": clocks.summary(),
        }
        if emit:
            print(json.dumps(line), flush=True)
    dist.barrier()
    if emit:
        dist.destroy_process_group()
    return line if rank == 0 else None
