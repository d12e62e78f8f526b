"""Row-range sharded execution of the operator path over N GPUs of one box (SURVEY.md 8e).

One process per GPU (torchrun).  Every table is split into contiguous row ranges, all columns
of a table co-partitioned, so select / fetch / add / sub / shared scan run shard-locally with
no data-path collective.  `torch.distributed` is plumbing only:

* aggregates     each rank reduces its rows on the device, then ONE exchange step: after
                 ``EngineOps.connect_peers`` a single kernel folds the local partials and
                 swaps them with every peer over NVLink peer memory
                 (``adb_agg_combine_allreduce``); without it, {sum, count} (int64, SUM) and
                 {max, ~min} (int32, MAX) NCCL all-reduces.  avg is the fp64 divide of the
                 reduced sum and count on the host (/root/reference/src/query.c:314);
* position lists stay shard-resident as (shard base row, local int32 positions); an all-gather
                 of the hit counts gives every shard its offset in the concatenated list, which
                 is only materialised for print / verification;
* hash join      both (value, position) pair lists are hash-routed by value and joined
                 locally; equal keys always meet on one rank, output pairs carry global
                 positions.  The exchange is either the routing kernel itself writing every
                 destination's run into that rank's receive region over NVLink peer memory
                 (``adb_peer_exchange_pairs``, after ``connect_peers(dist, join_cap_pairs)``) or
                 ``adb_route_pairs`` + an NCCL all-to-all-v.

The local operators come from an ``ops`` object: ``EngineOps`` (below) drives the CUDA engine
through its C-ABI on torch CUDA tensors; the CPU tests pass an oracle-backed stand-in to check
this module's partitioning and exchange logic under gloo.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import torch

I32 = torch.int32


def shard_range(n_rows: int, rank: int, world: int) -> tuple[int, int]:
    """Rows [begin, end) of shard `rank`: [g*N/G, (g+1)*N/G)."""
    return (n_rows * rank) // world, (n_rows * (rank + 1)) // world


@dataclass
class Positions:
    """A shard-resident position list: global row = base + local[i]."""
    local: torch.Tensor          # int32, ascending for scans
    base: int
    offset: int = 0              # where this shard's list starts in the concatenation
    total: int = 0               # hits over all shards


class EngineOps:
    """Local operators on torch CUDA tensors through the engine's C-ABI."""

    def __init__(self, engine, device):
        self.eng, self.lib, self.device = engine, engine.lib, device
        # engine kernels, torch's allocator and NCCL share one stream: no cross-stream hazards
        engine.set_stream(torch.cuda.current_stream(device).cuda_stream)
        self._cnt = torch.zeros(1, dtype=torch.int64, device=device)
        self._agg = torch.zeros(4, dtype=torch.int64, device=device)        # >= sizeof(adb_agg)

    @staticmethod
    def _p(t, ctype=C.c_int32):
        return C.cast(C.c_void_p(t.data_ptr()), C.POINTER(ctype))

    @staticmethod
    def _b(x):
        return None if x is None else C.pointer(C.c_int32(int(x)))

    def empty(self, n):
        return torch.empty(max(int(n), 0), dtype=I32, device=self.device)

    def select_scan(self, col, lo, hi):
        h = C.c_int64(0)
        self.eng._ck(self.lib.adb_select_count(self._p(col), col.numel(), None, self._b(lo),
                                               self._b(hi), self._p(self._cnt, C.c_int64), C.byref(h)))
        out = self.empty(h.value)
        self.eng._ck(self.lib.adb_select_emit(None, 0, self._p(out)))
        return out

    def fetch(self, col, pos):
        out = self.empty(pos.numel())
        self.eng._ck(self.lib.adb_fetch(self._p(col), self._p(pos), pos.numel(), None, 0, self._p(out)))
        return out

    def aggregate_packed(self, vals):
        """-> ({sum, count} int64[2], {max, ~min} int32[2]) on the device, allreduce-ready."""
        from .engine import _AggStruct
        aggp = C.cast(C.c_void_p(self._agg.data_ptr()), C.POINTER(_AggStruct))
        self.eng._ck(self.lib.adb_aggregate(self._p(vals), vals.numel(), None, aggp, None))
        sc = torch.empty(2, dtype=torch.int64, device=self.device)
        mm = torch.empty(2, dtype=I32, device=self.device)
        self.eng._ck(self.lib.adb_agg_export(aggp, C.c_void_p(sc.data_ptr()), C.c_void_p(mm.data_ptr())))
        return sc, mm

    def connect_peers(self, dist, join_cap_pairs: int = 0):
        """Map the peers' aggregate mailboxes (Engine.peer_setup): aggregates then take the
        one-kernel NVLink exchange instead of two NCCL all-reduces.  With join_cap_pairs, also
        reserve and map the receive buffers of the join's pair exchange
        (Engine.peer_join_setup): hash joins then push their routed pairs straight into the
        destination ranks' memory instead of going through six NCCL all-to-alls."""
        self.eng.peer_setup(dist)
        self.peers = True
        if join_cap_pairs:
            self.eng.peer_join_setup(dist, join_cap_pairs)
            self.peer_join = True

    def exchange_pairs_peer(self, side: int, val, pos):
        """adb_peer_exchange_pairs: this rank's share of the routed pairs as views of its
        receive regions (valid until the next exchange of the same side), or None when the
        receive buffers are not mapped."""
        if not getattr(self, "peer_join", False):
            return None
        cnt = C.c_int64(0)
        rv, rp = C.c_void_p(), C.c_void_p()
        self.eng._ck(self.lib.adb_peer_exchange_pairs(side, self._p(val), self._p(pos), val.numel(),
                                                      C.byref(cnt), C.byref(rv), C.byref(rp)))
        return self._view(rv.value, cnt.value), self._view(rp.value, cnt.value)

    def _view(self, ptr: int, n: int):
        if n == 0:
            return self.empty(0)

        class _Dev:                                   # the CUDA array interface of a raw region
            __cuda_array_interface__ = {"shape": (int(n),), "typestr": "<i4", "data": (int(ptr), False),
                                        "version": 3, "strides": None}
        return torch.as_tensor(_Dev(), device=self.device)

    def aggregate_fused(self, vals):
        """Local reduction + exchange with every peer inside adb_agg_combine_allreduce; returns
        the table-wide (sum, count, min, max) or None when the mailboxes are not mapped."""
        if not getattr(self, "peers", False):
            return None
        from .engine import _AggStruct
        aggp = C.cast(C.c_void_p(self._agg.data_ptr()), C.POINTER(_AggStruct))
        self.eng._ck(self.lib.adb_aggregate(self._p(vals), vals.numel(), None, aggp, None))
        h = _AggStruct()
        self.eng._ck(self.lib.adb_agg_combine_allreduce(aggp, 1, aggp, C.byref(h)))
        return h.sum, h.count, h.min, h.max

    def ewise(self, a, b, subtract):
        out = self.empty(a.numel())
        fn = self.lib.adb_sub if subtract else self.lib.adb_add
        self.eng._ck(fn(self._p(a), self._p(b), a.numel(), None, self._p(out)))
        return out

    def shared_select(self, col, lows, highs):
        q = len(lows)
        lo = (C.c_int32 * q)(*[int(x) for x in lows])
        hi = (C.c_int32 * q)(*[int(x) for x in highs])
        counts = (C.c_int64 * q)()
        self.eng._ck(self.lib.adb_shared_select_count(self._p(col), col.numel(), lo, hi, q, counts))
        outs = [self.empty(counts[i]) for i in range(q)]
        ptrs = (C.c_void_p * q)(*[o.data_ptr() for o in outs])
        self.eng._ck(self.lib.adb_shared_select_emit(ptrs, max(list(counts) + [1])))
        return outs

    def index_build(self, col, with_btree=True):
        """(values, positions, handle) of this shard's rows: adb_index_sort + adb_index_create."""
        n = col.numel()
        vals, poss = self.empty(n), self.empty(n)
        self.eng._ck(self.lib.adb_index_sort(self._p(col), n, self._p(vals), self._p(poss)))
        h = C.c_void_p()
        self.eng._ck(self.lib.adb_index_create(self._p(vals), self._p(poss), n, int(with_btree), C.byref(h)))
        return vals, poss, h

    def select_index(self, index, lo, hi, use_btree):
        h = C.c_int64(0)
        self.eng._ck(self.lib.adb_select_index_count(index[2], int(use_btree), self._b(lo), self._b(hi),
                                                     self._p(self._cnt, C.c_int64), C.byref(h)))
        out = self.empty(h.value)
        self.eng._ck(self.lib.adb_select_index_emit(index[2], self._p(out)))
        return out

    def route_pairs(self, val, pos, parts):
        """adb_route_pairs: the pairs grouped by destination rank, stable, and the per-rank
        counts.  A value's rank is its routing hash scaled to [0, parts); parts = the world size,
        any count in [1, 256]."""
        vo, po = self.empty(val.numel()), self.empty(val.numel())
        counts = (C.c_int64 * parts)()
        self.eng._ck(self.lib.adb_route_pairs(self._p(val), self._p(pos), val.numel(), parts,
                                              self._p(vo), self._p(po), counts))
        return vo, po, list(counts)

    def hash_join(self, v1, p1, v2, p2):
        m = C.c_int64(0)
        self.eng._ck(self.lib.adb_hash_join_count(self._p(v1), self._p(p1), v1.numel(), self._p(v2),
                                                  self._p(p2), v2.numel(), C.byref(m)))
        o1, o2 = self.empty(m.value), self.empty(m.value)
        self.eng._ck(self.lib.adb_join_emit(self._p(o1), self._p(o2)))
        return o1, o2


class ShardedTable:
    """This rank's row range of a table plus the cross-shard steps of every operator."""

    def __init__(self, ops, columns: dict, n_rows_global: int, dist=None):
        self.ops, self.cols, self.dist = ops, columns, dist
        self.world = dist.get_world_size() if dist is not None else 1
        self.rank = dist.get_rank() if dist is not None else 0
        self.begin, self.end = shard_range(n_rows_global, self.rank, self.world)
        for name, t in columns.items():
            if t.numel() != self.end - self.begin:
                raise ValueError(f"column {name}: {t.numel()} rows, shard owns {self.end - self.begin}")
        if self.end - self.begin >= 1 << 31:
            raise ValueError("a shard must stay below 2^31 rows (positions are int, query.c:94-95)")

    # ---- shard-local operators + count exchange ------------------------------------------
    def _offsets(self, count: int) -> tuple[int, int]:
        if self.dist is None:
            return 0, count
        t = torch.zeros(self.world, dtype=torch.int64, device=self.ops.device)
        mine = torch.tensor([count], dtype=torch.int64, device=self.ops.device)
        self.dist.all_gather_into_tensor(t, mine)
        c = t.tolist()
        return sum(c[:self.rank]), sum(c)

    def select(self, col: str, lo=None, hi=None) -> Positions:
        local = self.ops.select_scan(self.cols[col], lo, hi)
        off, total = self._offsets(local.numel())
        return Positions(local, self.begin, off, total)

    def shared_select(self, col: str, lows, highs) -> list[Positions]:
        outs = self.ops.shared_select(self.cols[col], lows, highs)
        if self.dist is None:
            return [Positions(o, self.begin, 0, o.numel()) for o in outs]
        q = len(outs)
        mine = torch.tensor([o.numel() for o in outs], dtype=torch.int64, device=self.ops.device)
        allc = torch.zeros(self.world * q, dtype=torch.int64, device=self.ops.device)
        self.dist.all_gather_into_tensor(allc, mine)          # one exchange for the whole batch
        allc = allc.view(self.world, q)
        before = allc[:self.rank].sum(0).tolist()
        totals = allc.sum(0).tolist()
        return [Positions(outs[i], self.begin, before[i], totals[i]) for i in range(q)]

    def build_index(self, col: str, with_btree: bool = True):
        """Per-shard sorted index (+ implicit B+-tree) over this shard's rows of `col`."""
        self.indexes = getattr(self, "indexes", {})
        self.indexes[col] = self.ops.index_build(self.cols[col], with_btree)

    def select_index(self, col: str, lo, hi, use_btree: bool = False) -> Positions:
        """Range select through the shard-local index.  The concatenation over shards is
        shard-major, value order inside a shard (SURVEY.md 8e): equal to the reference's
        single-index result as a set; compare order-insensitively or merge for print."""
        local = self.ops.select_index(self.indexes[col], lo, hi, use_btree)
        off, total = self._offsets(local.numel())
        return Positions(local, self.begin, off, total)

    def fetch(self, col: str, pos: Positions) -> torch.Tensor:
        return self.ops.fetch(self.cols[col], pos.local)       # positions never leave their shard

    def add(self, a, b):
        return self.ops.ewise(a, b, False)

    def sub(self, a, b):
        return self.ops.ewise(a, b, True)

    # ---- aggregates: one exchange step -----------------------------------------------------
    def aggregate(self, vals: torch.Tensor) -> dict:
        fused = self.ops.aggregate_fused(vals) if self.dist is not None and hasattr(self.ops, "aggregate_fused") else None
        if fused is not None:
            s, n, mn, mx = fused
            return {"sum": s, "count": n, "min": mn, "max": mx,
                    "avg": float("nan") if n == 0 else float(s) / float(n)}
        sc, mm = self.ops.aggregate_packed(vals)
        if self.dist is not None:
            self.dist.all_reduce(sc, op=self.dist.ReduceOp.SUM)
            self.dist.all_reduce(mm, op=self.dist.ReduceOp.MAX)
        s, n = sc.tolist()
        mx, notmn = mm.tolist()
        # (double)sum / (double)count: Python's int -> float conversion rounds to nearest even
        # exactly as the C cast does, and the division is the same IEEE operation
        avg = float("nan") if n == 0 else float(s) / float(n)
        return {"sum": s, "count": n, "min": ~notmn, "max": mx, "avg": avg}

    # ---- verification / print: materialise the concatenation -------------------------------
    def gather_global(self, local_i32: torch.Tensor, base: int = 0) -> torch.Tensor:
        """All shards' lists concatenated in shard order, as int64 (+ base) on every rank."""
        mine = local_i32.to(torch.int64) + base
        if self.dist is None:
            return mine
        n = torch.tensor([mine.numel()], dtype=torch.int64, device=self.ops.device)
        alln = torch.zeros(self.world, dtype=torch.int64, device=self.ops.device)
        self.dist.all_gather_into_tensor(alln, n)
        sizes = alln.tolist()
        cap = max(sizes + [1])
        pad = torch.zeros(cap, dtype=torch.int64, device=self.ops.device)
        pad[:mine.numel()] = mine
        buf = torch.zeros(self.world * cap, dtype=torch.int64, device=self.ops.device)
        self.dist.all_gather_into_tensor(buf, pad)
        return torch.cat([buf[r * cap:r * cap + sizes[r]] for r in range(self.world)])

    # ---- hash join: route -> all-to-all-v -> local build + probe ----------------------------
    def exchange_pairs(self, val: torch.Tensor, pos: torch.Tensor, side: int = 0):
        """Hash-route a (value, global position) pair list; returns this rank's share, the
        pieces ordered by source rank and in source order inside a piece.  `side` names the
        receive region when the exchange runs over peer memory (both inputs of a join must
        be resident at once)."""
        if self.dist is None:
            return val, pos
        if hasattr(self.ops, "exchange_pairs_peer"):
            got = self.ops.exchange_pairs_peer(side, val, pos)
            if got is not None:
                return got
        vo, po, counts = self.ops.route_pairs(val, pos, self.world)
        send = torch.tensor(counts, dtype=torch.int64, device=self.ops.device)
        recv = torch.zeros_like(send)
        self.dist.all_to_all_single(recv, send)
        rc = recv.tolist()
        rv = torch.empty(sum(rc), dtype=I32, device=self.ops.device)
        rp = torch.empty(sum(rc), dtype=I32, device=self.ops.device)
        self.dist.all_to_all_single(rv, vo, output_split_sizes=rc, input_split_sizes=counts)
        self.dist.all_to_all_single(rp, po, output_split_sizes=rc, input_split_sizes=counts)
        return rv, rp

    def hash_join(self, v1, p1, v2, p2):
        """Equi-join of two sharded pair lists (hash_join, query.c:652-696).  Positions must be
        global and fit int32 (the reference's own limit).  Returns this rank's (pos1, pos2)
        pairs; the union over ranks is the reference's result as a set of pairs."""
        a_v, a_p = self.exchange_pairs(v1, p1, 0)
        b_v, b_p = self.exchange_pairs(v2, p2, 1)
        return self.ops.hash_join(a_v, a_p, b_v, b_p)
