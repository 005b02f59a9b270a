"""Row-sharded search across the GPUs of one box (SURVEY.md §8e).

One process per GPU.  Rank r owns the contiguous rows [lo_r, hi_r) of the DB; queries are replicated;
every rank scans its shard (K2), the per-shard top-k lists are exchanged with ONE all-gather of a
packed [ids | scores | counts] blob per rank over NCCL/NVLink, and K3 merges them (every rank
computes the same answer).  No other collective is on the data path.

`shard_bounds`, `pack_results`, `unpack_results` and `allgather_packed` are backend-agnostic host
logic (exercised with gloo on CPU in tests/test_sharded_gloo.py); `ShardedIndex.search` is the CUDA
product path.

The self-join of a collection row-sharded over the devices of ONE process (B200VectorDB(devices=[...]).find_near_duplicates) is
here too: `selfjoin_plan` (pure host logic) and `selfjoin_sharded`, which joins the shards where they live and moves only
query blocks.
"""
from __future__ import annotations

import ctypes as C
from typing import NamedTuple

import numpy as np
import torch
import torch.distributed as dist

from . import _lib, ops
from ._lib import check


def shard_bounds(n_rows: int, world: int, rank: int, align: int = 128) -> tuple[int, int]:
    """Contiguous row range of `rank`.  Shards are whole 128-row blocks of the tiled DB storage (so that a shard
    is a slice of it); the first (blocks % world) ranks get one extra block, the last shard ends at n_rows."""
    blocks = (n_rows + align - 1) // align
    base, extra = divmod(blocks, world)
    lo = rank * base + min(rank, extra)
    hi = lo + base + (1 if rank < extra else 0)
    return min(lo * align, n_rows), min(hi * align, n_rows)


def packed_bytes(nq: int, k: int) -> int:
    return (nq * k * 12 + nq * 4 + 7) // 8 * 8


def pack_results(ids: torch.Tensor, scores: torch.Tensor, counts: torch.Tensor) -> torch.Tensor:
    """[ids int64 nq*k | scores f32 nq*k | counts int32 nq] as one uint8 blob (pure byte copies)."""
    nq, k = ids.shape
    blob = torch.zeros(packed_bytes(nq, k), dtype=torch.uint8, device=ids.device)
    blob[: nq * k * 8].copy_(ids.contiguous().view(torch.uint8).flatten())
    blob[nq * k * 8: nq * k * 12].copy_(scores.contiguous().view(torch.uint8).flatten())
    blob[nq * k * 12: nq * k * 12 + nq * 4].copy_(counts.contiguous().view(torch.uint8).flatten())
    return blob


def unpack_results(gathered: torch.Tensor, nq: int, k: int):
    """gathered uint8 [G, packed_bytes] -> (ids [G,nq,k], scores [G,nq,k], counts [G,nq]) (copies)."""
    G = gathered.shape[0]
    ids = gathered[:, : nq * k * 8].contiguous().view(torch.int64).view(G, nq, k)
    scores = gathered[:, nq * k * 8: nq * k * 12].contiguous().view(torch.float32).view(G, nq, k)
    counts = gathered[:, nq * k * 12: nq * k * 12 + nq * 4].contiguous().view(torch.int32).view(G, nq)
    return ids, scores, counts


def allgather_packed(blob: torch.Tensor, group=None) -> torch.Tensor:
    world = dist.get_world_size(group)
    out = torch.empty((world, blob.numel()), dtype=torch.uint8, device=blob.device)
    dist.all_gather_into_tensor(out.view(-1), blob, group=group)
    return out


def selfjoin_blocks(n_rows: int, world: int, rank: int, block: int = 4096) -> list[tuple[int, int]]:
    """Query-row ranges of `rank` for the self-join (DB replicated): 4096-row blocks dealt in snake order
    (0..w-1, w-1..0, ...), so that the triangular work (block b scans rows >= b) is balanced across ranks.
    Adjacent blocks are merged."""
    out: list[tuple[int, int]] = []
    nblk = (n_rows + block - 1) // block
    for b in range(nblk):
        rnd, pos = divmod(b, world)
        if (pos if rnd % 2 == 0 else world - 1 - pos) != rank:
            continue
        lo, hi = b * block, min(n_rows, (b + 1) * block)
        if out and out[-1][1] == lo:
            out[-1] = (out[-1][0], hi)
        else:
            out.append((lo, hi))
    return out


class JoinItem(NamedTuple):
    """Query rows [q_lo, q_hi) of shard q_shard against target rows [t_lo, t_hi) of shard t_shard (local rows); it runs on the
    target shard's device.  q_shard == t_shard: a block of that shard's triangle (pairs i < j only, t_lo = q_lo, t_hi = the
    shard's size); otherwise a rectangle (every pair)."""
    q_shard: int
    q_lo: int
    q_hi: int
    t_shard: int
    t_lo: int
    t_hi: int


def selfjoin_plan(sizes: list[int], block: int = 4096) -> list[list[JoinItem]]:
    """Work of the self-join of a collection row-sharded into shards of `sizes` rows: list g holds the items that run on shard
    g's device.  Every unordered pair of rows is examined by exactly one item, and no shard leaves its device: only query
    blocks of `block` rows (a multiple of 128) move.

    The triangle of a shard runs on its own device.  The rectangle of shards a < b is split at s, a multiple of `block`: query
    blocks [0, s) of a run on b against all of b, and every query block of b runs on a against rows [s, n_a) of a (a target
    sub-range that starts on a 128-row block).  s is chosen so that the devices' loads, in row pairs, are as even as the
    triangles allow: the fractional shares are balanced pairwise until they settle (each step equalises the loads of the two
    devices of one rectangle, which minimises the sum of squared loads and with it the largest), then rounded to whole
    blocks one rectangle at a time."""
    G = len(sizes)
    n = [int(x) for x in sizes]
    load = [x * (x - 1) / 2 for x in n]
    rects = [(a, b) for a in range(G) for b in range(a + 1, G) if n[a] and n[b]]
    share = {}                                   # share of rectangle (a, b) that runs on b
    for a, b in rects:
        share[a, b] = 0.5
        load[a] += n[a] * n[b] / 2
        load[b] += n[a] * n[b] / 2
    for _ in range(200):
        moved = 0.0
        for a, b in rects:
            r, x = n[a] * n[b], share[a, b]
            la, lb = load[a] - (1 - x) * r, load[b] - x * r
            v = min(1.0, max(0.0, (la - lb + r) / (2 * r)))
            share[a, b] = v
            load[a], load[b] = la + (1 - v) * r, lb + v * r
            moved = max(moved, abs(v - x) * r)
        if moved < 1.0:
            break
    split = {}
    for a, b in rects:
        r, x = n[a] * n[b], share[a, b]
        la, lb = load[a] - (1 - x) * r, load[b] - x * r
        lo = int(x * n[a]) // block * block
        s = min((min(c, n[a]) for c in (lo, lo + block)), key=lambda c: (max(la + (n[a] - c) * n[b], lb + c * n[b]), c))
        split[a, b] = s
        load[a], load[b] = la + (n[a] - s) * n[b], lb + s * n[b]
    plan: list[list[JoinItem]] = [[] for _ in range(G)]
    for g in range(G):
        plan[g] += [JoinItem(g, lo, min(lo + block, n[g]), g, lo, n[g]) for lo in range(0, n[g], block)]
    for a, b in rects:
        s = split[a, b]
        plan[b] += [JoinItem(a, lo, min(lo + block, s), b, 0, n[b]) for lo in range(0, s, block)]
        if s < n[a]:
            plan[a] += [JoinItem(b, lo, min(lo + block, n[b]), a, s, n[a]) for lo in range(0, n[b], block)]
    return plan


def selfjoin_sharded(shards: list, d: int, threshold: float, max_pairs: int = 1 << 22, cand_cap: int = 32768,
                     block: int = 4096, device_ms: dict | None = None):
    """Self-join of a collection row-sharded over the devices of one process: all pairs of rows with cos >= threshold.
    shards: [(tiled storage, rows, first global row)], each tensor on its shard's device (several shards may share a device).
    Returns host arrays (pairs int64 [m, 2] of global rows, lower first; scores f32 [m]) — the same pairs and bit-identical
    scores as the single-device join of the same rows.

    Every item of `selfjoin_plan` is enqueued, round-robin over the devices, before any synchronisation: one host sync per
    device.  A query block of another device is copied (a peer copy) into one of two staging blocks on the target device,
    ordered after the source device's current stream; the joins run on each device's current stream and append to one pair
    buffer per device.  Overflow protocol of `ops.selfjoin_exact`, judged per device: overflowed candidate lists re-run that
    device's items with 8x the capacity (exact once it covers the rows scanned + 4096), a pair count above the buffer re-runs
    them with a buffer of that count.  `device_ms`: filled with each device's busy time (CUDA events, ms) of the last attempt."""
    sizes = [int(n) for _, n, _ in shards]
    plan = selfjoin_plan(sizes, block)
    items: dict[int, list[JoinItem]] = {}
    for g, its in enumerate(plan):
        items.setdefault(shards[g][0].device.index, []).extend(its)
    cap = {dv: int(cand_cap) for dv in items}
    out_cap = {dv: int(max_pairs) for dv in items}
    rows_scanned = {dv: max(it.t_hi - it.t_lo for it in its) for dv, its in items.items() if its}
    todo = sorted(rows_scanned)
    done: dict[int, tuple] = {}
    while todo:
        ready = {}           # copies read a shard after what its device's current stream had queued before the join
        for v, _, _ in shards:
            if v.device.index not in ready:
                ready[v.device.index] = torch.cuda.Event()
                ready[v.device.index].record(torch.cuda.current_stream(v.device))
        runs = {dv: _join_runs(items[dv], shards, dv) for dv in todo}
        st = {dv: _JoinState(torch.device("cuda", dv), out_cap[dv], d, block, ready) for dv in todo}
        for k in range(max(len(r) for r in runs.values())):
            for dv in todo:
                if k < len(runs[dv]):
                    st[dv].run(runs[dv][k], shards, d, threshold, cap[dv])
        retry = []
        for dv in todo:
            s = st[dv]
            s.stop.record(torch.cuda.current_stream(s.dev))
            torch.cuda.current_stream(s.dev).synchronize()
            if device_ms is not None:
                device_ms[dv] = s.start.elapsed_time(s.stop)
            pairs, scores, count, over = s.out
            m, ov = int(count.item()), int(over.item())
            if ov > 0 and cap[dv] < rows_scanned[dv] + 4096:
                cap[dv] = min(cap[dv] * 8, rows_scanned[dv] + 4096 + ops.TILE_ROWS * 16)
                retry.append(dv)
            elif m > out_cap[dv]:
                out_cap[dv] = m
                retry.append(dv)
            elif ov > 0:
                raise _lib.RvoError(f"self-join candidate lists overflowed at capacity {cap[dv]} on cuda:{dv}")
            else:
                done[dv] = (pairs[:m].cpu().numpy(), scores[:m].cpu().numpy())
        todo = retry
    if not done:
        return np.zeros((0, 2), np.int64), np.zeros(0, np.float32)
    return np.concatenate([done[dv][0] for dv in sorted(done)]), np.concatenate([done[dv][1] for dv in sorted(done)])


def _join_runs(its: list[JoinItem], shards: list, dv: int) -> list[JoinItem]:
    """The items of one device as calls: consecutive items that read their query rows in place (same device) and share a
    target merge into one call (the C entry walks the query blocks itself); a query block of another device stays one call."""
    runs: list[JoinItem] = []
    for it in its:
        local = shards[it.q_shard][0].device.index == dv
        p = runs[-1] if runs else None
        if (local and p is not None and shards[p.q_shard][0].device.index == dv and p.q_shard == it.q_shard
                and p.t_shard == it.t_shard and p.q_hi == it.q_lo and p.t_hi == it.t_hi
                and (p.t_lo == it.t_lo or it.q_shard == it.t_shard)):
            runs[-1] = p._replace(q_hi=it.q_hi)
        else:
            runs.append(it)
    return runs


class _JoinState:
    """Pair buffer, staging blocks and streams of one device during `selfjoin_sharded`."""

    def __init__(self, dev: torch.device, out_cap: int, d: int, block: int, ready: dict):
        self.dev, self.ready = dev, ready
        self.out = ops.join_out(out_cap, dev)
        self.d, self.block = d, block
        self.slots: list = []                    # two staging blocks: the copy of one overlaps the join of the other
        self.free: list = []                     # event per slot: the join that last read it has finished
        self.next = 0
        self.copy_stream = None
        self.src_streams: dict = {}
        self.start, self.stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.start.record(torch.cuda.current_stream(dev))

    def run(self, it: JoinItem, shards: list, d: int, threshold: float, cand_cap: int) -> None:
        qv, _, q_row0 = shards[it.q_shard]
        tv, _, t_row0 = shards[it.t_shard]
        cur = torch.cuda.current_stream(self.dev)
        if it.q_shard == it.t_shard:
            with torch.cuda.device(self.dev):
                ops.join_threshold(tv, it.q_lo, it.q_hi, t_row0, tv, it.t_hi, d, threshold, t_row0, cand_cap, self.out)
            return
        target = tv[it.t_lo // ops.TILE_ROWS:]
        if qv.device == self.dev:
            qdb, q_lo, q_hi, q_off = qv, it.q_lo, it.q_hi, q_row0
        else:
            b0, b1 = it.q_lo // ops.TILE_ROWS, (it.q_hi + ops.TILE_ROWS - 1) // ops.TILE_ROWS
            if not self.slots:
                self.slots = [ops.db_alloc(self.block, d, self.dev) for _ in range(2)]
                self.free = [None, None]
                self.copy_stream = torch.cuda.Stream(self.dev)
            k = self.next % 2
            self.next += 1
            src = self.src_streams.get(qv.device.index)
            if src is None:
                src = self.src_streams[qv.device.index] = torch.cuda.Stream(qv.device)
                src.wait_event(self.ready[qv.device.index])
            if self.free[k] is not None:
                self.copy_stream.wait_event(self.free[k])
            # a cross-device copy_ runs on the source device's current stream, after the destination device's current stream
            with torch.cuda.stream(src), torch.cuda.stream(self.copy_stream):
                self.slots[k][: b1 - b0].copy_(qv[b0:b1], non_blocking=True)
            cur.wait_stream(self.copy_stream)
            qdb, q_lo, q_hi, q_off = self.slots[k], it.q_lo - b0 * ops.TILE_ROWS, it.q_hi - b0 * ops.TILE_ROWS, q_row0 + b0 * ops.TILE_ROWS
        with torch.cuda.device(self.dev):
            ops.join_threshold(qdb, q_lo, q_hi, q_off, target, it.t_hi - it.t_lo, d, threshold, t_row0 + it.t_lo, cand_cap,
                               self.out)
        if qdb is not qv:
            ev = torch.cuda.Event()
            ev.record(cur)
            self.free[k] = ev


class ShardedIndex:
    """The local shard of a row-sharded bf16 DB plus the exchange/merge step."""

    def __init__(self, local_db: torch.Tensor, n_local: int, d: int, id_offset: int, group=None):
        """local_db: tiled bf16 storage (ops.db_alloc) of this rank's rows; id_offset: its first global row."""
        ops.require_cuda(local_db, "local_db")
        self.db, self.n_local, self.d, self.id_offset, self.group = local_db, int(n_local), int(d), int(id_offset), group
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        self._bufs: dict = {}
        self._pipe = None          # submit / collect state
        self._xchg = None          # peer-memory exchange state (enable_peer_exchange)

    # ---- peer-memory exchange: K2's last kernel pushes the result into every peer's region over NVLink ----------------
    def enable_peer_exchange(self, nq_max: int, k_max: int) -> bool:
        """Collective (every rank of the group calls it).  Allocates this rank's exchange region, swaps CUDA IPC handles with
        the peers and maps theirs.  Afterwards `search` replaces the NCCL all-gather by stores into peer memory fused into
        the last kernel of the shard search, and K3 waits on epoch flags (include/revers_o_b200.h, "Peer-memory exchange").
        Returns False (and changes nothing) when the box/topology does not allow it; all ranks get the same answer."""
        if self.world < 2 or self.world > 8:
            return False
        lib = _lib.load()
        dev = self.db.device
        ok, region, peers = 1, C.c_void_p(), []
        nbytes = lib.rvo_exchange_bytes(self.world, int(nq_max), int(k_max))
        handle = (C.c_ubyte * 64)()
        with torch.cuda.device(dev):
            if nbytes == 0 or self.n_local == 0 or lib.rvo_exchange_alloc(nbytes, C.byref(region)) != 0 \
                    or lib.rvo_exchange_export(region, handle) != 0:
                ok = 0
        gathered = [None] * self.world
        dist.all_gather_object(gathered, (ok, bytes(handle)), group=self.group)
        ok = int(all(g[0] for g in gathered))
        table = (C.c_void_p * self.world)()
        if ok:
            with torch.cuda.device(dev):
                for g, (_, h) in enumerate(gathered):
                    if g == self.rank:
                        table[g] = region.value
                        continue
                    p = C.c_void_p()
                    if lib.rvo_exchange_import((C.c_ubyte * 64).from_buffer_copy(h), C.byref(p)) != 0:
                        ok = 0
                        break
                    table[g] = p.value
                    peers.append(p)
        flags = [None] * self.world
        dist.all_gather_object(flags, ok, group=self.group)       # every mapping must have worked on every rank
        if not all(flags):
            with torch.cuda.device(dev):
                for p in peers:
                    lib.rvo_exchange_unimport(p)
                if region.value:
                    lib.rvo_exchange_free(region)
            return False
        self._xchg = {"region": region, "peers": peers, "table": table, "nq_max": int(nq_max), "k_max": int(k_max), "epoch": 0}
        return True

    def _use_fused(self, k: int) -> bool:
        import os
        return self.world * k <= 2048 and os.environ.get("RVO_FUSED", "1") != "0"

    def disable_peer_exchange(self) -> None:
        """Collective.  Unmaps the peers' regions and frees the local one (after every rank has stopped using them)."""
        if self._xchg is None:
            return
        torch.cuda.synchronize(self.db.device)
        dist.barrier(group=self.group)
        lib = _lib.load()
        with torch.cuda.device(self.db.device):
            for p in self._xchg["peers"]:
                lib.rvo_exchange_unimport(p)
            dist.barrier(group=self.group)
            lib.rvo_exchange_free(self._xchg["region"])
        self._xchg = None

    def _search_push(self, queries: torch.Tensor, k: int, score_threshold, out=None):
        import math
        x = self._xchg
        nq = queries.shape[0]
        dev = self.db.device
        lib = _lib.load()
        key = ("x", nq, k)
        if self._bufs.get("key") != key:
            self._bufs = {"key": key, "oi": torch.empty((nq, k), dtype=torch.int64, device=dev),
                          "os": torch.empty((nq, k), dtype=torch.float32, device=dev),
                          "oc": torch.empty((nq,), dtype=torch.int32, device=dev)}
        b = self._bufs
        epoch = x["epoch"] + 1      # committed only after BOTH launches succeeded: a failed call must not desynchronise the ranks
        nbytes = lib.rvo_search_workspace_bytes(self.n_local, self.d, nq, k)
        ws = ops.workspace(dev, nbytes)
        thr = -math.inf if score_threshold is None else float(score_threshold)
        stream = torch.cuda.current_stream(dev).cuda_stream
        if self._use_fused(k):
            # exchange AND merge inside the last search kernel: the outputs are the merged lists, no second launch
            oi, os_, oc = out if out is not None else (b["oi"], b["os"], b["oc"])
            check(lib.rvo_search_topk_fused(self.db.data_ptr(), self.n_local, self.d, ops.d_pad_of(self.d), queries.data_ptr(), nq, k,
                                            thr, self.id_offset, x["table"], self.world, self.rank, x["nq_max"], x["k_max"], epoch,
                                            oi.data_ptr(), os_.data_ptr(), oc.data_ptr(), ws.data_ptr(), nbytes, stream),
                  "rvo_search_topk_fused")
            x["epoch"] = epoch
            return oi, os_, oc
        check(lib.rvo_search_topk_push(self.db.data_ptr(), self.n_local, self.d, ops.d_pad_of(self.d), queries.data_ptr(), nq, k,
                                       thr, self.id_offset, x["table"], self.world, self.rank, x["nq_max"], x["k_max"],
                                       epoch, ws.data_ptr(), nbytes, stream), "rvo_search_topk_push")
        oi, os_, oc = out if out is not None else (b["oi"], b["os"], b["oc"])
        check(lib.rvo_merge_topk_exchange(x["region"], self.world, nq, k, x["nq_max"], x["k_max"], epoch,
                                          oi.data_ptr(), os_.data_ptr(), oc.data_ptr(), stream),
              "rvo_merge_topk_exchange")
        x["epoch"] = epoch
        return oi, os_, oc

    @classmethod
    def from_disk(cls, path: str, collection_name: str, device, rank: int | None = None, world: int | None = None,
                  group=None, chunk_blocks: int = 4096):
        """Load this rank's row shard of a saved collection (`B200VectorDB.save`) straight to its GPU: the tiled file is
        memory-mapped and only the rank's 128-row blocks are read, `chunk_blocks` blocks at a time through a pinned
        staging buffer (SURVEY.md §8f row 3; replaces qdrant's sqlite + pickle load behind core_system.py:90-119)."""
        from .vector_db import read_shard_blocks
        if world is None:
            world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        if rank is None:
            rank = dist.get_rank(group) if dist.is_available() and dist.is_initialized() else 0
        view, n_local, row0, dim = read_shard_blocks(path, collection_name, world, rank)
        dev = torch.device(device)
        db = ops.db_alloc(max(n_local, 1) if view.shape[0] == 0 else view.shape[0] * ops.TILE_ROWS, dim, dev)
        if view.shape[0]:
            stage = torch.empty((min(chunk_blocks, view.shape[0]),) + tuple(view.shape[1:]), dtype=torch.int16).pin_memory()
            for b0 in range(0, view.shape[0], chunk_blocks):
                b1 = min(view.shape[0], b0 + chunk_blocks)
                stage[: b1 - b0].numpy()[...] = view[b0:b1]
                db[b0:b1].copy_(stage[: b1 - b0].view(torch.bfloat16), non_blocking=True)
                torch.cuda.current_stream(dev).synchronize()      # the staging buffer is reused by the next chunk
        idx = cls(db, n_local, dim, row0, group)
        idx.attach_tables(path, collection_name)
        return idx

    # ---- host-side tables indexed by GLOBAL row (SURVEY.md §8e: "uuid strings / payloads stay in a host-side table") -----
    def attach_tables(self, path: str, collection_name: str) -> None:
        """Map the collection's id column and payload log (vector_db.py on-disk format 2): `<collection>.ids` is memory-mapped
        (fixed-width records: no parse, pages touched on demand), payloads are parsed per hit.  Every rank maps the same files."""
        import json
        import os

        import numpy as np

        from .tables import IdTable, PayloadStore
        self.ids = self.payloads = None
        try:
            with open(os.path.join(path, "meta.json")) as f:
                m = json.load(f)["collections"][collection_name]
        except (OSError, KeyError):
            return
        n = int(m["n"])
        if m.get("ids_dtype") and n:
            arr = np.memmap(os.path.join(path, f"{collection_name}.ids"), dtype=np.dtype(m["ids_dtype"]), mode="r", shape=(n,))
            self.ids = IdTable.from_array(arr)
        if "idx_bytes" in m:
            self.payloads = PayloadStore.open(os.path.join(path, f"{collection_name}.payload.jsonl"),
                                              os.path.join(path, f"{collection_name}.payload.idx"), n, int(m["idx_bytes"]))

    def hits(self, ids_row, scores_row, count: int) -> list:
        """One query's merged result as the `ScoredPoint`s core_system.py:671-676 consumes (id, score, payload)."""
        from .vector_db import ScoredPoint
        out = []
        for i, s in zip(ids_row[:count].tolist(), scores_row[:count].tolist()):
            out.append(ScoredPoint(id=self.ids[i] if getattr(self, "ids", None) is not None else i, version=0, score=float(s),
                                   payload=self.payloads[i] if getattr(self, "payloads", None) is not None else None))
        return out

    def search_local(self, queries: torch.Tensor, k: int, score_threshold=None):
        return ops.search_topk(self.db, self.n_local, self.d, queries, k, score_threshold, self.id_offset)

    def search(self, queries: torch.Tensor, k: int, score_threshold=None, out=None):
        """queries: f32 [Q, d] on this rank's GPU (replicated).  Returns merged (ids, scores, counts) — views of buffers the
        index reuses on its next call with the same (Q, k): copy them if they must outlive it.  Asynchronous on the current
        stream; every rank of the group must call it (same Q, k) in the same order.  `queries` may be a pinned host tensor and
        `out` = (ids int64 [Q,k], scores f32 [Q,k], counts int32 [Q]) pinned host tensors: the first kernel then reads and K3
        writes over PCIe, with no copy launches around the search."""
        if self.world == 1:
            return ops.search_topk(self.db, self.n_local, self.d, queries, k, score_threshold, self.id_offset, out=out)
        nq = queries.shape[0]
        x = self._xchg
        if x is not None and _lib.RVO_SMALL_Q < nq <= x["nq_max"] and k <= x["k_max"]:
            return self._search_push(queries, k, score_threshold, out)
        dev = self.db.device
        # K2 writes straight into the packed [ids | scores | counts] blob that the all-gather ships (no pack kernels)
        key = (nq, k)
        if self._bufs.get("key") != key:
            nb = packed_bytes(nq, k)
            self._bufs = {"key": key, "blob": torch.zeros(nb, dtype=torch.uint8, device=dev),
                          "gathered": torch.empty((self.world, nb), dtype=torch.uint8, device=dev),
                          "oi": torch.empty((nq, k), dtype=torch.int64, device=dev),
                          "os": torch.empty((nq, k), dtype=torch.float32, device=dev),
                          "oc": torch.empty((nq,), dtype=torch.int32, device=dev)}
        b = self._bufs
        blob = b["blob"]
        ids = blob[: nq * k * 8].view(torch.int64).view(nq, k)
        scores = blob[nq * k * 8: nq * k * 12].view(torch.float32).view(nq, k)
        counts = blob[nq * k * 12: nq * k * 12 + nq * 4].view(torch.int32)
        ops.search_topk(self.db, self.n_local, self.d, queries, k, score_threshold, self.id_offset, out=(ids, scores, counts))
        dist.all_gather_into_tensor(b["gathered"].view(-1), blob, group=self.group)   # the ONE collective of the path
        oi, os_, oc = out if out is not None else (b["oi"], b["os"], b["oc"])
        check(_lib.load().rvo_merge_topk_packed(b["gathered"].data_ptr(), b["gathered"].stride(0), self.world, nq, k,
                                                oi.data_ptr(), os_.data_ptr(), oc.data_ptr(),
                                                torch.cuda.current_stream(dev).cuda_stream), "rvo_merge_topk_packed")
        return oi, os_, oc

    # ---- pipelined serving: the scan of batch i+1 is enqueued BEFORE the exchange + merge of batch i ---------------------------
    def submit(self, queries: torch.Tensor, k: int, score_threshold=None):
        """Enqueue K2 of one batch (and, with the peer exchange, its push) and return a ticket for `collect`.  At most TWO
        tickets may be outstanding; every rank of the group must submit / collect in the same order.  A serving loop calls
        `t1 = submit(q1); t2 = submit(q2); r1 = collect(t1); t3 = submit(q3); r2 = collect(t2); ...`: while a rank waits for
        the slowest peer's lists of batch i it is already scanning batch i+1 (the synchronous `search` makes every step as slow
        as the slowest rank plus the rendezvous).  One GPU: the two batches run on two streams with their own scratch, so the
        threshold-seeding kernels and the select of one batch fill the ramp and tail of the other's scan."""
        import math
        nq = queries.shape[0]
        dev = self.db.device
        lib = _lib.load()
        p = self._pipe
        if p is None or p["key"] != (nq, k):
            p = self._pipe = {"key": (nq, k), "n": 0, "out": [None, None], "pending": [],
                              "streams": [torch.cuda.Stream(dev), torch.cuda.Stream(dev)] if self.world == 1 else None,
                              "events": [torch.cuda.Event(), torch.cuda.Event()]}
            nb = packed_bytes(nq, k)
            for j in range(2):
                p["out"][j] = {"oi": torch.empty((nq, k), dtype=torch.int64, device=dev),
                               "os": torch.empty((nq, k), dtype=torch.float32, device=dev),
                               "oc": torch.empty((nq,), dtype=torch.int32, device=dev),
                               "blob": torch.zeros(nb, dtype=torch.uint8, device=dev),
                               "gathered": torch.empty((self.world, nb), dtype=torch.uint8, device=dev) if self.world > 1 else None}
        if len(p["pending"]) >= 2:
            raise _lib.RvoError("two batches are already in flight: collect one first")
        j = p["n"] & 1
        p["n"] += 1
        o = p["out"][j]
        thr = -math.inf if score_threshold is None else float(score_threshold)
        x = self._xchg
        ticket = {"j": j, "nq": nq, "k": k, "mode": "local", "epoch": 0}
        if self.world == 1:
            st = p["streams"][j]
            st.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(st):
                ops.search_topk(self.db, self.n_local, self.d, queries, k, score_threshold, self.id_offset,
                                out=(o["oi"], o["os"], o["oc"]), ws_key=("pipe", id(self), j))
                p["events"][j].record(st)
        elif x is not None and _lib.RVO_SMALL_Q < nq <= x["nq_max"] and k <= x["k_max"] and self._use_fused(k):
            # the fused exchange has no separate merge to defer: the whole search is one chain of launches
            epoch = x["epoch"] + 1
            nbytes = lib.rvo_search_workspace_bytes(self.n_local, self.d, nq, k)
            ws = ops.workspace(dev, nbytes)
            check(lib.rvo_search_topk_fused(self.db.data_ptr(), self.n_local, self.d, ops.d_pad_of(self.d), queries.data_ptr(), nq, k,
                                            thr, self.id_offset, x["table"], self.world, self.rank, x["nq_max"], x["k_max"], epoch,
                                            o["oi"].data_ptr(), o["os"].data_ptr(), o["oc"].data_ptr(), ws.data_ptr(), nbytes,
                                            torch.cuda.current_stream(dev).cuda_stream), "rvo_search_topk_fused")
            x["epoch"] = epoch
            ticket.update(mode="fused", epoch=epoch)
        elif x is not None and _lib.RVO_SMALL_Q < nq <= x["nq_max"] and k <= x["k_max"]:
            epoch = x["epoch"] + 1
            nbytes = lib.rvo_search_workspace_bytes(self.n_local, self.d, nq, k)
            ws = ops.workspace(dev, nbytes)
            check(lib.rvo_search_topk_push(self.db.data_ptr(), self.n_local, self.d, ops.d_pad_of(self.d), queries.data_ptr(), nq, k,
                                           thr, self.id_offset, x["table"], self.world, self.rank, x["nq_max"], x["k_max"], epoch,
                                           ws.data_ptr(), nbytes, torch.cuda.current_stream(dev).cuda_stream), "rvo_search_topk_push")
            x["epoch"] = epoch
            ticket.update(mode="push", epoch=epoch)
        else:
            blob = o["blob"]
            views = (blob[: nq * k * 8].view(torch.int64).view(nq, k), blob[nq * k * 8: nq * k * 12].view(torch.float32).view(nq, k),
                     blob[nq * k * 12: nq * k * 12 + nq * 4].view(torch.int32))
            ops.search_topk(self.db, self.n_local, self.d, queries, k, score_threshold, self.id_offset, out=views)
            ticket.update(mode="nccl")
        p["pending"].append(ticket)
        return ticket

    def collect(self, ticket):
        """Exchange + merge of a submitted batch (tickets in submission order).  Returns (ids, scores, counts): views of buffers
        that are reused two submissions later."""
        p = self._pipe
        if not p or not p["pending"] or p["pending"][0] is not ticket:
            raise _lib.RvoError("collect() takes the oldest outstanding ticket")
        p["pending"].pop(0)
        o = p["out"][ticket["j"]]
        dev = self.db.device
        nq, k = ticket["nq"], ticket["k"]
        lib = _lib.load()
        if ticket["mode"] == "local":
            torch.cuda.current_stream(dev).wait_event(p["events"][ticket["j"]])
        elif ticket["mode"] == "fused":
            pass
        elif ticket["mode"] == "push":
            x = self._xchg
            check(lib.rvo_merge_topk_exchange(x["region"], self.world, nq, k, x["nq_max"], x["k_max"], ticket["epoch"],
                                              o["oi"].data_ptr(), o["os"].data_ptr(), o["oc"].data_ptr(),
                                              torch.cuda.current_stream(dev).cuda_stream), "rvo_merge_topk_exchange")
        else:
            dist.all_gather_into_tensor(o["gathered"].view(-1), o["blob"], group=self.group)
            check(lib.rvo_merge_topk_packed(o["gathered"].data_ptr(), o["gathered"].stride(0), self.world, nq, k,
                                            o["oi"].data_ptr(), o["os"].data_ptr(), o["oc"].data_ptr(),
                                            torch.cuda.current_stream(dev).cuda_stream), "rvo_merge_topk_packed")
        return o["oi"], o["os"], o["oc"]

    def search_exact(self, queries: torch.Tensor, k: int, score_threshold=None):
        ids, scores, counts = self._search_exact(queries, k, score_threshold)
        if bool((counts == -2).any().item()):
            raise _lib.RvoError("peer exchange timed out (option exchange_timeout_ms): a rank did not publish its lists; "
                                "re-run with disable_peer_exchange() (NCCL all-gather)")
        return ids, scores, counts

    def _search_exact(self, queries: torch.Tensor, k: int, score_threshold=None):
        """`search` plus the overflow protocol of rvo_search_topk: queries whose merged count is -1 (more than 2048
        candidates inside the bf16 admission margin on some shard) are re-run on every rank through the exact fp32 scan
        (`ops.search_topk_exact`) and merged again.  Every rank computes the same merged counts, so all ranks take the
        same branch without an extra collective; reading the counts is one host sync."""
        ids, scores, counts = self.search(queries, k, score_threshold)
        bad = (counts < 0).nonzero().flatten()
        if bad.numel() == 0:
            return ids, scores, counts
        ids, scores, counts = ids.clone(), scores.clone(), counts.clone()
        sub = queries[bad].contiguous()
        a, b_, c = ops.search_topk_exact(self.db, self.n_local, self.d, sub, k, score_threshold, self.id_offset)
        if self.world > 1:
            blob = pack_results(a, b_, c)
            g = allgather_packed(blob, self.group)
            gi, gs, gc = unpack_results(g, sub.shape[0], k)
            a, b_, c = ops.merge_topk(gi, gs, gc, k)
        ids[bad], scores[bad], counts[bad] = a, b_, c
        return ids, scores, counts
