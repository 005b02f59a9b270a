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
query blocks.  So is the join between two such collections (B200VectorDB.join_collections): `crossjoin_plan` and
`crossjoin_sharded`, run by the same device loop, and the duplicate groups of a row-sharded collection
(B200VectorDB.find_duplicate_groups): `components_sharded`, the self-join's items unioned into one forest per device.  The
k-nearest-neighbour join of two such collections, or of one with itself (B200VectorDB.knn_join), is `knn_plan` and `knn_sharded`:
per-shard lists merged by K3 on the left shard's device, sharing the staging code (`_Staging`) of the joins.  Spherical k-means of
such a collection (B200VectorDB.cluster) is `kmeans_sharded`: every shard assigned and summed on its own device, the integer sums
added on the first device.
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


def _split_rectangles(load, rects: list, block: int) -> dict:
    """Split points of rectangles whose two sides live on two different devices.  rects: [(key, u, v, n_a, n_b)]: query blocks
    [0, s) of side a run on v against all of side b, every query block of b runs on u against rows [s, n_a) of a.  `load`
    (indexable by u and v) holds the loads, in row pairs, that are already fixed, and is updated with the rectangles' shares.
    The fractional shares are balanced pairwise until they settle (each step equalises the loads of the two devices of one
    rectangle, which minimises the sum of squared loads and with it the largest), then rounded to multiples of `block` one
    rectangle at a time.  Returns {key: s}."""
    share = {}                                   # share of each rectangle that runs on v
    for key, u, v, na, nb in rects:
        share[key] = 0.5
        load[u] += na * nb / 2
        load[v] += na * nb / 2
    for _ in range(200):
        moved = 0.0
        for key, u, v, na, nb in rects:
            r, x = na * nb, share[key]
            lu, lv = load[u] - (1 - x) * r, load[v] - x * r
            w = min(1.0, max(0.0, (lu - lv + r) / (2 * r)))
            share[key] = w
            load[u], load[v] = lu + (1 - w) * r, lv + w * r
            moved = max(moved, abs(w - x) * r)
        if moved < 1.0:
            break
    split = {}
    for key, u, v, na, nb in rects:
        r, x = na * nb, share[key]
        lu, lv = load[u] - (1 - x) * r, load[v] - x * r
        lo = int(x * na) // block * block
        s = min((min(c, na) for c in (lo, lo + block)), key=lambda c: (max(lu + (na - c) * nb, lv + c * nb), c))
        split[key] = s
        load[u], load[v] = lu + (na - s) * nb, lv + s * nb
    return split


def selfjoin_plan(sizes: list[int], block: int = 4096) -> list[list[JoinItem]]:
    """Work of the self-join of a collection row-sharded into shards of `sizes` rows: list g holds the items that run on shard
    g's device.  Every unordered pair of rows is examined by exactly one item, and no shard leaves its device: only query
    blocks of `block` rows (a multiple of 128) move.

    The triangle of a shard runs on its own device.  The rectangle of shards a < b is split at s, a multiple of `block`: query
    blocks [0, s) of a run on b against all of b, and every query block of b runs on a against rows [s, n_a) of a (a target
    sub-range that starts on a 128-row block).  s is chosen so that the devices' loads, in row pairs, are as even as the
    triangles allow (`_split_rectangles`, with one load per shard)."""
    G = len(sizes)
    n = [int(x) for x in sizes]
    load = [x * (x - 1) / 2 for x in n]
    rects = [(a, b) for a in range(G) for b in range(a + 1, G) if n[a] and n[b]]
    split = _split_rectangles(load, [((a, b), a, b, n[a], n[b]) for a, b in rects], block)
    plan: list[list[JoinItem]] = [[] for _ in range(G)]
    for g in range(G):
        plan[g] += [JoinItem(g, lo, min(lo + block, n[g]), g, lo, n[g]) for lo in range(0, n[g], block)]
    for a, b in rects:
        s = split[a, b]
        plan[b] += [JoinItem(a, lo, min(lo + block, s), b, 0, n[b]) for lo in range(0, s, block)]
        if s < n[a]:
            plan[a] += [JoinItem(b, lo, min(lo + block, n[b]), a, s, n[a]) for lo in range(0, n[b], block)]
    return plan


def crossjoin_plan(left: list, right: list, block: int = 4096) -> dict[int, list[JoinItem]]:
    """Work of the join between two row-sharded collections: left and right are [(device index, rows)], one entry per shard
    (several shards may share a device, and the two sides may list different devices).  Returns {device index: items that
    run there} for every device listed.  An item's shard index counts the left shards first: shard a of the left side is
    a, shard b of the right side is len(left) + b.  Every (left row, right row) pair is examined by exactly one item, and
    only query blocks of `block` rows (a multiple of 128) move.

    The rectangle of left shard a and right shard b runs whole on their device when they share one (left query blocks
    against all of b).  Otherwise it is split at s, a multiple of `block`: left query blocks [0, s) of a run on b's device
    against all of b, and every query block of b runs on a's device against left rows [s, n_a) (a target sub-range that
    starts on a 128-row block).  The loads are the devices' (`_split_rectangles`, one load per device)."""
    L = [(int(dv), int(n)) for dv, n in left]
    R = [(int(dv), int(n)) for dv, n in right]
    nl = len(L)
    plan: dict[int, list[JoinItem]] = {}
    for dv, _ in L + R:
        plan.setdefault(dv, [])
    load = {dv: 0.0 for dv in plan}
    rects = []
    for a, (da, na) in enumerate(L):
        for b, (db, nb) in enumerate(R):
            if not na or not nb:
                continue
            if da == db:
                load[da] += na * nb
                plan[da] += [JoinItem(a, lo, min(lo + block, na), nl + b, 0, nb) for lo in range(0, na, block)]
            else:
                rects.append(((a, b), da, db, na, nb))
    split = _split_rectangles(load, rects, block)
    for (a, b), da, db, na, nb in rects:
        s = split[a, b]
        plan[db] += [JoinItem(a, lo, min(lo + block, s), nl + b, 0, nb) for lo in range(0, s, block)]
        if s < na:
            plan[da] += [JoinItem(nl + b, lo, min(lo + block, nb), a, s, na) for lo in range(0, nb, block)]
    return plan


def selfjoin_sharded(shards: list, d: int, threshold: float, max_pairs: int = 1 << 22, cand_cap: int = 32768,
                     block: int = 4096, device_ms: dict | None = None):
    """Self-join of a collection row-sharded over the devices of one process: all pairs of rows with cos >= threshold.
    shards: [(tiled storage, rows, first global row)], each tensor on its shard's device (several shards may share a device).
    Returns host arrays (pairs int64 [m, 2] of global rows, lower first; scores f32 [m]) — the same pairs and bit-identical
    scores as the single-device join of the same rows.  Runs the items of `selfjoin_plan` through `_join_on_devices`."""
    sizes = [int(n) for _, n, _ in shards]
    plan = selfjoin_plan(sizes, block)
    items: dict[int, list[JoinItem]] = {}
    for g, its in enumerate(plan):
        items.setdefault(shards[g][0].device.index, []).extend(its)
    return _join_on_devices(shards, items, d, threshold, max_pairs, cand_cap, block, device_ms, None)


def crossjoin_sharded(left: list, right: list, d: int, threshold: float, max_pairs: int = 1 << 22, cand_cap: int = 32768,
                      block: int = 4096, device_ms: dict | None = None):
    """Join of two collections, each row-sharded over devices of one process (one shard on one device is the plain case):
    all (left row, right row) pairs with cos >= threshold.  left, right: [(tiled storage, rows, first global row)].  Returns
    host arrays (pairs int64 [m, 2] = (left global row, right global row); scores f32 [m], the fp32 dot of the two stored
    rows, bit-identical to the self-join's score of the same rows).  Runs the items of `crossjoin_plan` through
    `_join_on_devices`."""
    items = crossjoin_plan([(v.device.index, n) for v, n, _ in left], [(v.device.index, n) for v, n, _ in right], block)
    return _join_on_devices(list(left) + list(right), items, d, threshold, max_pairs, cand_cap, block, device_ms, len(left))


def components_sharded(shards: list, d: int, threshold: float, cand_cap: int = 32768, block: int = 4096,
                       device_ms: dict | None = None):
    """Single-linkage groups of a collection row-sharded over the devices of one process: the connected components of exactly
    the pairs `selfjoin_sharded` returns.  shards as there.  Each device runs its `selfjoin_plan` items into a union-find forest
    over all the global rows (`rvo_join_components`); then every other device's forest is flattened, copied to the first device
    and merged there (`rvo_components_merge`), so every edge any device found is in the result.  Returns (labels int64 [N] host
    array over the global rows [0, N), N = the end of the last shard, each the smallest global row of its component; n_pairs) —
    the same as `ops.components_exact` on one device."""
    sizes = [int(n) for _, n, _ in shards]
    plan = selfjoin_plan(sizes, block)
    items: dict[int, list[JoinItem]] = {}
    for g, its in enumerate(plan):
        items.setdefault(shards[g][0].device.index, []).extend(its)
    n_labels = max(int(r0) + int(n) for _, n, r0 in shards)
    done = _join_on_devices(shards, items, d, threshold, 0, cand_cap, block, device_ms, None, n_labels)
    devs = sorted(done)
    root = done[devs[0]][0]
    for dv in devs[1:]:
        labels = ops.components_flatten(done[dv][0])
        with torch.cuda.device(root.device):
            ops.components_merge(root, labels.to(root.device))    # a peer copy, ordered after the flatten and before the merge
    labels = ops.components_flatten(root).cpu().numpy().astype(np.int64)
    return labels, sum(m for _, m in done.values())


def _join_on_devices(shards: list, items: dict, d: int, threshold: float, max_pairs: int, cand_cap: int, block: int,
                     device_ms: dict | None, n_left: int | None, n_labels: int | None = None):
    """Run {device index: [JoinItem]} over shards [(tiled storage, rows, first global row)].  n_left None: the items are a
    self-join's (triangles and rectangles, `rvo_join_threshold`); otherwise shards [0, n_left) are the left collection and
    the rest the right one, and every item is a cross join (`rvo_cross_join_threshold`).  n_labels given (a self-join only): the
    pairs are not stored but unioned into one forest per device over the n_labels global rows (`rvo_join_components`), and
    {device index: (parent int32 [n_labels] on that device, pairs found there)} is returned.

    Every item is enqueued, round-robin over the devices, before any synchronisation: one host sync per device.  A query
    block of another device is copied (a peer copy) into one of two staging blocks on the target device, ordered after the
    source device's current stream; the joins run on each device's current stream and append to one pair buffer per device.
    Overflow protocol of `ops.selfjoin_exact`, judged per device: overflowed candidate lists re-run that device's items with
    8x the capacity (exact once it covers the rows scanned + 4096), a pair count above the buffer re-runs them with a buffer
    of that count (pair buffers only: a forest keeps its edges across a re-run, since re-applying an edge changes nothing).
    `device_ms`: filled with each device's busy time (CUDA events, ms) of the last attempt."""
    cap = {dv: int(cand_cap) for dv in items}
    out_cap = {dv: int(max_pairs) for dv in items}
    rows_scanned = {dv: max(it.t_hi - it.t_lo for it in its) for dv, its in items.items() if its}
    todo = sorted(rows_scanned)
    done: dict[int, tuple] = {}
    forests = {dv: ops.components_out(n_labels, torch.device("cuda", dv))[0] for dv in todo} if n_labels else {}
    while todo:
        ready = {}           # copies read a shard after what its device's current stream had queued before the join
        for v, _, _ in shards:
            if v.device.index not in ready:
                ready[v.device.index] = torch.cuda.Event()
                ready[v.device.index].record(torch.cuda.current_stream(v.device))
        runs = {dv: _join_runs(items[dv], shards, dv) for dv in todo}
        st = {dv: _JoinState(torch.device("cuda", dv), out_cap[dv], d, block, ready, n_left, forests.get(dv)) for dv in todo}
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
            count, over = s.out[-2:]
            m, ov = int(count.item()), int(over.item())
            if ov > 0 and cap[dv] < rows_scanned[dv] + 4096:
                cap[dv] = min(cap[dv] * 8, rows_scanned[dv] + 4096 + ops.TILE_ROWS * 16)
                retry.append(dv)
            elif not n_labels and m > out_cap[dv]:
                out_cap[dv] = m
                retry.append(dv)
            elif ov > 0:
                what = "self-join" if n_left is None else "cross join"
                raise _lib.RvoError(f"{what} candidate lists overflowed at capacity {cap[dv]} on cuda:{dv}")
            elif n_labels:
                done[dv] = (s.out[0], m)
            else:
                done[dv] = (s.out[0][:m].cpu().numpy(), s.out[1][:m].cpu().numpy())
        todo = retry
    if n_labels:
        return done
    if not done:
        return np.zeros((0, 2), np.int64), np.zeros(0, np.float32)
    return np.concatenate([done[dv][0] for dv in sorted(done)]), np.concatenate([done[dv][1] for dv in sorted(done)])


class KnnItem(NamedTuple):
    """Query rows [q_lo, q_hi) of left shard q_shard against every row of right shard t_shard, on the right shard's device."""
    q_shard: int
    q_lo: int
    q_hi: int
    t_shard: int


def knn_plan(left: list, right: list, block: int = 8192) -> dict[int, list[KnnItem]]:
    """Work of the kNN join of two row-sharded collections: left and right are [(device index, rows)].  Returns {device index of
    a right shard: items that run there}.  Every left shard is cut into query blocks of `block` rows (a multiple of 128, so a
    block is whole tiles), and every (query block, right shard) pair is one item on the right shard's device: right shards never
    move, query blocks do.  Each device's items come block by block in left row order."""
    if block <= 0 or block % ops.TILE_ROWS:
        raise _lib.RvoError(f"kNN join query blocks must be a positive multiple of {ops.TILE_ROWS} rows, got {block}")
    plan: dict[int, list[KnnItem]] = {int(dv): [] for dv, _ in right}
    for a, (_, na) in enumerate(left):
        for lo in range(0, int(na), block):
            for b, (dv, nb) in enumerate(right):
                if int(nb):
                    plan[int(dv)].append(KnnItem(a, lo, min(lo + block, int(na)), b))
    return plan


def knn_sharded(left: list, right: list, d: int, k: int, score_threshold: float | None, exclude_self: bool,
                device_ms: dict | None = None, block: int = 8192, chunk: int = 1 << 18):
    """kNN join of two collections, each row-sharded over devices of one process: for every left row, in row order, the k
    right rows with the highest fp32 dot of the two stored rows.  left, right: [(tiled storage, rows, first global row)], the
    left shards in row order; `exclude_self` (left and right are one collection): a row's own match is left out.  Returns host
    arrays (rows int64 [N_L, k] of global right rows, -1 pad; scores f32 [N_L, k], -inf pad; counts int32 [N_L]); a count of -1
    remains only for rows wider than 2048 that overflowed (`ops.knn_exact`).  Equal to the single-device result: ids identical,
    scores equal up to the last bits where one layout took the fp32 route for a row and the other did not.

    Results go to pinned host memory as they are made, so device memory does not grow with the left collection.  One shard
    on one device: one `rvo_knn_join` call per `chunk` left rows into one reusable device buffer (12 * chunk * k bytes).
    Otherwise `knn_plan`'s items run with k' = k + 1 (self mode) or k lists each, one query block (`block` rows, a multiple of
    128) at a time, enqueued before any synchronisation: for each block, every right shard's device joins it (a block of another
    device is peer-copied into that device's staging blocks, `_Staging`) into that shard's reusable list buffer [block, k']; the
    lists are peer-copied into the block's home device's gather buffer [shards, block, k'], merged there (`rvo_merge_topk`: at
    most 64 right shards, shards * k' <= 4096), stripped of the row itself (self mode) and copied to pinned host memory.
    Per device that is 12 * block * k' bytes per right shard it holds, 12 * shards * block * k' bytes of gather buffer if it
    holds left rows, two staging blocks and one search workspace.  A cross-device copy orders both devices' current streams
    around it, so a buffer is rewritten only after its previous contents have been copied or merged.  Rows the merge flags -1
    are then re-run through the exact fp32 routes (`ops.knn_fp32`) on every right shard and merged again, as the sharded search
    does.  `device_ms`: each device's busy time (CUDA events, ms) of the enqueued work."""
    if block <= 0 or block % ops.TILE_ROWS:
        raise _lib.RvoError(f"kNN join query blocks must be a positive multiple of {ops.TILE_ROWS} rows, got {block}")
    kk = k + 1 if exclude_self else k
    G = len(right)
    n_left = sum(int(n) for _, n, _ in left)
    out_i = torch.full((n_left, k), -1, dtype=torch.int64).pin_memory()
    out_s = torch.full((n_left, k), -float("inf"), dtype=torch.float32).pin_memory()
    out_c = torch.zeros((n_left,), dtype=torch.int32).pin_memory()
    if n_left == 0 or G == 0:
        return out_i.numpy(), out_s.numpy(), out_c.numpy()
    single = len(left) == 1 and G == 1 and left[0][0].device == right[0][0].device
    if not single and (G > 64 or G * kk > 4096):
        raise _lib.RvoError(f"kNN join over {G} right shards with {kk} candidates each: the merge takes at most 64 shards and "
                            "4096 candidates per row")
    offs = [0]
    for _, n, _ in left:
        offs.append(offs[-1] + int(n))
    ready = {}                     # copies read a shard after what its device's current stream had queued before the join
    for v, _, _ in list(left) + list(right):
        if v.device.index not in ready:
            ready[v.device.index] = torch.cuda.Event()
            ready[v.device.index].record(torch.cuda.current_stream(v.device))
    st = {dv: _Staging(torch.device("cuda", dv), d, block, ready) for dv in ready}
    if single:
        (qv, nl, q0), (tv, nr, t0) = left[0], right[0]
        m = min(chunk, nl)
        buf = (torch.empty((m, k), dtype=torch.int64, device=tv.device), torch.empty((m, k), dtype=torch.float32, device=tv.device),
               torch.empty((m,), dtype=torch.int32, device=tv.device))
        with torch.cuda.device(tv.device):
            for lo in range(0, nl, m):
                hi = min(nl, lo + m)
                res = ops.knn_join(qv, lo, hi, q0, tv, nr, d, k, score_threshold, t0, exclude_self,
                                   out=tuple(x[: hi - lo] for x in buf))
                for dst, src in zip((out_i, out_s, out_c), res):      # stream-ordered before the next call rewrites buf
                    dst[lo:hi].copy_(src, non_blocking=True)
    else:
        _knn_blocks(left, right, offs, d, k, kk, score_threshold, exclude_self, block, st, (out_i, out_s, out_c))
    for s in st.values():
        s.stop.record(torch.cuda.current_stream(s.dev))
    for dv in sorted(st):
        torch.cuda.current_stream(torch.device("cuda", dv)).synchronize()
    if device_ms is not None:
        for dv, s in st.items():
            device_ms[dv] = s.start.elapsed_time(s.stop)
    for a, (qv, nl, q0) in enumerate(left):
        bad = (out_c[offs[a]: offs[a] + int(nl)] < 0).nonzero().flatten()
        if bad.numel():
            _knn_overflow(left[a], offs[a], bad, right, d, k, kk, score_threshold, exclude_self, (out_i, out_s, out_c))
    return out_i.numpy(), out_s.numpy(), out_c.numpy()


def _knn_blocks(left: list, right: list, offs: list, d: int, k: int, kk: int, score_threshold, exclude_self: bool, block: int,
                st: dict, out: tuple) -> None:
    """The block pipeline of `knn_sharded` (several shards): enqueues, for every query block of `knn_plan` in left row order,
    the joins on the right shards' devices, the peer copies of their lists to the block's home device, the merge, the exclusion
    and the copy into the pinned host outputs `out`.  Nothing synchronises."""
    G = len(right)
    parts = [(torch.empty((block, kk), dtype=torch.int64, device=tv.device),
              torch.empty((block, kk), dtype=torch.float32, device=tv.device),
              torch.empty((block,), dtype=torch.int32, device=tv.device)) for tv, _, _ in right]
    gather = {}
    for qv, nl, _ in left:
        if nl and qv.device.index not in gather:
            dev = qv.device
            gather[dev.index] = (torch.empty(G * block * kk, dtype=torch.int64, device=dev),
                                 torch.empty(G * block * kk, dtype=torch.float32, device=dev),
                                 torch.empty(G * block, dtype=torch.int32, device=dev))
    plan = knn_plan([(v.device.index, n) for v, n, _ in left], [(v.device.index, n) for v, n, _ in right], block)
    blocks: dict = {}                                  # (left shard, q_lo) -> (q_hi, [items]) in left row order
    for dv, its in plan.items():
        for it in its:
            blocks.setdefault((it.q_shard, it.q_lo), (it.q_hi, []))[1].append(it)
    for (a, lo), (hi, its) in sorted(blocks.items()):
        qv, _, q0 = left[a]
        nb = hi - lo
        for it in its:
            tv, nr, t0 = right[it.t_shard]
            s = st[tv.device.index]
            qdb, q_lo, q_hi, q_off, slot = s.stage(qv, lo, hi, q0)
            pi, ps, pc = parts[it.t_shard]
            with torch.cuda.device(s.dev):
                ops.knn_join(qdb, q_lo, q_hi, q_off, tv, nr, d, kk, score_threshold, t0, False, out=(pi[:nb], ps[:nb], pc[:nb]))
            s.release(slot)
        home = qv.device
        fi, fs, fc = gather[home.index]
        gi, gs, gc = fi[: G * nb * kk].view(G, nb, kk), fs[: G * nb * kk].view(G, nb, kk), fc[: G * nb].view(G, nb)
        with torch.cuda.device(home):
            for it in its:                             # peer copies: after the join on its device, before the merge here
                pi, ps, pc = parts[it.t_shard]
                gi[it.t_shard].copy_(pi[:nb], non_blocking=True)
                gs[it.t_shard].copy_(ps[:nb], non_blocking=True)
                gc[it.t_shard].copy_(pc[:nb], non_blocking=True)
            res = ops.merge_topk(gi, gs, gc, kk)
            if exclude_self:
                res = ops.knn_exclude_self(*res, lo, q0)
            o0 = offs[a] + lo
            for dst, src in zip(out, res):
                dst[o0:o0 + nb].copy_(src, non_blocking=True)


def _knn_overflow(left_shard, off: int, bad: torch.Tensor, right: list, d: int, k: int, kk: int, score_threshold,
                  exclude_self: bool, out: tuple) -> None:
    """Overflow protocol of `knn_sharded` for the flagged local rows `bad` of one left shard: their tiles are copied to every
    right shard's device, the exact fp32 routes (`ops.knn_fp32`) run them there as a q_rows list, and the lists are merged on
    the left shard's device (then the row itself is left out) into rows off + bad of the host outputs.  Every shard scores such
    a row with the same fp32 arithmetic, as the single-device protocol does over all the rows.  Rows wider than 2048 have no
    fp32 route and stay flagged.  Synchronises."""
    qv, _, q0 = left_shard
    if ops.d_pad_of(d) > 2048:
        return
    home = qv.device
    rows = bad.to(home)
    tiles, slot = torch.unique(rows // ops.TILE_ROWS, return_inverse=True)
    stage = qv[tiles]                                          # the tiles holding the flagged rows
    local = slot * ops.TILE_ROWS + rows % ops.TILE_ROWS        # their rows inside the staged tiles
    parts = []
    for tv, nr, t0 in right:
        with torch.cuda.device(tv.device):
            qd, qr = stage.to(tv.device), local.to(tv.device)
            parts.append(ops.knn_fp32(qd, qr, 0, tv, nr, d, kk, score_threshold, t0, False))
    with torch.cuda.device(home):
        res = ops.merge_topk(torch.stack([p[0].to(home) for p in parts]), torch.stack([p[1].to(home) for p in parts]),
                             torch.stack([p[2].to(home) for p in parts]), kk)
        if exclude_self:
            res = ops.knn_exclude_self(*res, 0, q0, rows)
        idx = bad + off
        for dst, src in zip(out, res):
            dst[idx] = src.cpu()


class KMeansResult(NamedTuple):
    """Spherical k-means in the clusters' own numbering.  labels int32 [N] and scores float32 [N] (host, global row order):
    every row's assignment to `centroids`; centroids: the tiled bf16 storage of the C centroids (on the first device);
    sizes int64 [C] (host): members per cluster; iterations: updates run; converged: the last assignment equals the previous."""
    labels: np.ndarray
    scores: np.ndarray
    centroids: torch.Tensor
    sizes: np.ndarray
    iterations: int
    converged: bool


def gather_rows(shards: list, rows, d: int, device: torch.device) -> torch.Tensor:
    """The stored bf16 rows `rows` (global rows of shards [(tiled storage, rows, first global row)]) copied bit for bit into
    rows [0, len(rows)) of a new tiled storage on `device`."""
    rows = torch.as_tensor(np.asarray(rows, dtype=np.int64))
    out = ops.db_alloc(max(len(rows), 1), d, device)
    dst = torch.arange(len(rows), dtype=torch.int64)
    for v, n, r0 in shards:
        sel = ((rows >= r0) & (rows < r0 + n)).nonzero().flatten()
        if sel.numel():
            lr = (rows[sel] - r0).to(v.device)
            o = dst[sel].to(device)
            out[o // ops.TILE_ROWS, :, o % ops.TILE_ROWS, :] = v[lr // ops.TILE_ROWS, :, lr % ops.TILE_ROWS, :].to(device)
    return out


def reseed_rows(scores: list, row0s: list, n_empty: int) -> list:
    """The rows that re-seed `n_empty` empty clusters: the rows with the lowest assignment scores, ties by the lower row, in that
    order (cluster j of the empty ones, in index order, takes entry j).  scores: one 1-d tensor per shard, the scores of its rows
    in row order; row0s: each shard's first global row.  Each shard offers its n_empty lowest, so only those are compared."""
    dev = scores[0].device
    cand_s, cand_r = [], []
    for sc, r0 in zip(scores, row0s):
        o = torch.sort(sc, stable=True).indices[:n_empty]             # ascending, equal scores in row order
        cand_s.append(sc[o].to(dev))
        cand_r.append((o + int(r0)).to(dev))
    s, r = torch.cat(cand_s), torch.cat(cand_r)
    o = torch.argsort(r)
    s, r = s[o], r[o]
    return r[torch.sort(s, stable=True).indices[:n_empty]].tolist()


def kmeans_sharded(shards: list, d: int, centroids: torch.Tensor, n_clusters: int, max_iter: int = 50) -> KMeansResult:
    """Spherical k-means of a collection row-sharded over the devices of one process; no row moves.  shards: [(tiled storage,
    rows, first global row)] in row order, covering the global rows [0, N) with N < 2^31; `centroids`: tiled storage holding the
    C = n_clusters initial centroids on the first device (not modified).

    Assign, then, while fewer than max_iter updates have run, update and assign again; stop at the first assignment equal to
    the previous one (the centroids are then a fixed point).  Each iteration:
      - the centroid buffer (2 C d_pad bytes) is peer-copied from the first device to every other shard device;
      - every shard runs `ops.knn_join` (k = 1) of its rows against it on its own device, all enqueued before the overflow
        check, and rows the fused path flags go through the exact fp32 routes (`ops.knn_fp32`): `ops.knn_exact`'s protocol;
      - `ops.kmeans_update` turns each shard's assignment into labels and adds its members to its device's int64 sums and
        counts; the other devices' sums, counts and change counts are peer-copied to the first device and added there.  The
        sums are integers, so the result does not depend on the shard layout;
      - `ops.kmeans_finalize` normalises the sums into the next centroid buffer, and one host synchronisation reads the
        change count and the number of empty clusters;
      - each empty cluster (no member, or an all-zero sum), in index order, takes the stored row `reseed_rows` gives.
    Memory per device: sums 8 C d and counts 8 C bytes, the centroid buffer(s), the assignment (21 bytes per row of its shards)
    and the workspaces of `knn_join` and `kmeans_update`."""
    C, max_iter = int(n_clusters), int(max_iter)
    n_total = sum(int(n) for _, n, _ in shards)
    if not 0 < n_total < (1 << 31):
        raise _lib.RvoError(f"k-means needs 1 to 2^31 - 1 rows, got {n_total}")
    if not 1 <= C <= min(n_total, _lib.RVO_KMEANS_MAX_CLUSTERS):
        raise _lib.RvoError(f"k-means: n_clusters={C} outside 1..{min(n_total, _lib.RVO_KMEANS_MAX_CLUSTERS)}")
    if max_iter < 0:
        raise _lib.RvoError(f"k-means: max_iter={max_iter} < 0")
    home = centroids.device
    devs = list(dict.fromkeys([home] + [v.device for v, _, _ in shards]))
    acc = {dv: (torch.zeros((C, d), dtype=torch.int64, device=dv), torch.zeros((C,), dtype=torch.int64, device=dv),
                torch.zeros((2,), dtype=torch.int64, device=dv)) for dv in devs}          # sums, counts, (changed, empty)
    cent = [ops.db_alloc(C, d, home), ops.db_alloc(C, d, home)]
    cent[0].copy_(centroids[: cent[0].shape[0]])
    local = {dv: ops.db_alloc(C, d, dv) for dv in devs if dv != home}
    empty = torch.zeros((C,), dtype=torch.int32, device=home)
    assign = [(torch.empty((n, 1), dtype=torch.int64, device=v.device), torch.empty((n, 1), dtype=torch.float32, device=v.device),
               torch.empty((n,), dtype=torch.int32, device=v.device)) for v, n, _ in shards]
    labels = [[torch.empty((n,), dtype=torch.int32, device=v.device) for v, n, _ in shards] for _ in range(2)]
    it, cur, converged = 0, 0, False
    while True:
        for dv, buf in local.items():
            with torch.cuda.device(dv):
                buf.copy_(cent[0], non_blocking=True)          # a peer copy, after the home stream's finalise, before the joins
        for (v, n, r0), out in zip(shards, assign):
            with torch.cuda.device(v.device):
                ops.knn_join(v, 0, n, r0, local.get(v.device, cent[0]), C, d, 1, None, 0, False, out=out)
        for (v, n, r0), (ids, sc, cnt) in zip(shards, assign):
            bad = (cnt < 0).nonzero().flatten()                # host sync; pathological inputs only take the branch
            if bad.numel() and ops.d_pad_of(d) > 2048:
                raise _lib.RvoError(f"k-means: rows {(bad + r0).tolist()[:20]} overflowed the candidate lists and rows of {d} "
                                    "dims (> 2048) have no exact fp32 route")
            if bad.numel():
                with torch.cuda.device(v.device):
                    ids[bad], sc[bad], cnt[bad] = ops.knn_fp32(v, bad, r0, local.get(v.device, cent[0]), C, d, 1, None, 0, False)
        for g, ((v, n, _), (ids, _, _)) in enumerate(zip(shards, assign)):
            sums, counts, stats = acc[v.device]
            with torch.cuda.device(v.device):
                ops.kmeans_update(v, 0, n, d, ids, C, labels[1 - cur][g] if it else None, labels[cur][g], sums, counts, stats[:1])
        sums, counts, stats = acc[home]
        with torch.cuda.device(home):
            for dv in devs[1:]:                                  # integer additions: any order gives the same sums
                sums += acc[dv][0].to(home)
                counts += acc[dv][1].to(home)
                stats[:1] += acc[dv][2][:1].to(home)
            if it < max_iter:
                ops.kmeans_finalize(sums, counts, d, cent[1], empty, stats[1:])
        changed, n_empty = stats.tolist()
        if it and changed == 0:
            converged = True
            break
        if it == max_iter:
            break
        if n_empty:
            which = empty.nonzero().flatten().tolist()
            rows = reseed_rows([a[1].view(-1) for a in assign], [r0 for _, _, r0 in shards], len(which))
            seeds = gather_rows(shards, rows, d, home)
            w = torch.tensor(which, dtype=torch.int64, device=home)
            j = torch.arange(len(which), dtype=torch.int64, device=home)
            cent[1][w // ops.TILE_ROWS, :, w % ops.TILE_ROWS, :] = seeds[j // ops.TILE_ROWS, :, j % ops.TILE_ROWS, :]
        cent.reverse()
        cur = 1 - cur
        it += 1
        for a in acc.values():
            for t in a:
                t.zero_()
    lab = np.concatenate([x.cpu().numpy() for x in labels[cur]])
    sc = np.concatenate([a[1].view(-1).cpu().numpy() for a in assign])
    return KMeansResult(lab, sc, cent[0], acc[home][1].cpu().numpy(), it, converged)


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


class _Staging:
    """Staging blocks, copy streams and busy-time events of one device: query blocks of shards on other devices are peer-copied
    into one of two staging blocks here, so the copy of one block overlaps the work on the other (`_JoinState`, `knn_sharded`)."""

    def __init__(self, dev: torch.device, d: int, block: int, ready: dict):
        self.dev, self.ready = dev, ready
        self.d, self.block = d, block
        self.slots: list = []                    # two staging blocks: the copy of one overlaps the join of the other
        self.free: list = []                     # event per slot: the join that last read it has finished
        self.next = 0
        self.copy_stream = None
        self.src_streams: dict = {}
        self.start, self.stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.start.record(torch.cuda.current_stream(dev))

    def stage(self, qv: torch.Tensor, q_lo: int, q_hi: int, q_row0: int):
        """Query rows [q_lo, q_hi) (at most `block`) of the tiled storage qv, whose first global row is q_row0, as seen from this
        device: (tiled storage, lo, hi, first global row of that storage, staging slot or None).  Rows of this device are read
        in place; others are copied, ordered after the source device's current stream as it was when `ready` was recorded and
        before this device's current stream.  Pass the slot to `release` after the work that reads it is enqueued."""
        if qv.device == self.dev:
            return qv, q_lo, q_hi, q_row0, None
        b0, b1 = q_lo // ops.TILE_ROWS, (q_hi + ops.TILE_ROWS - 1) // ops.TILE_ROWS
        if not self.slots:
            self.slots = [ops.db_alloc(self.block, self.d, self.dev) for _ in range(2)]
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
        torch.cuda.current_stream(self.dev).wait_stream(self.copy_stream)
        return self.slots[k], q_lo - b0 * ops.TILE_ROWS, q_hi - b0 * ops.TILE_ROWS, q_row0 + b0 * ops.TILE_ROWS, k

    def release(self, slot) -> None:
        if slot is not None:
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(self.dev))
            self.free[slot] = ev


class _JoinState(_Staging):
    """Output (a pair buffer, or a union-find forest), staging blocks and streams of one device during `_join_on_devices`."""

    def __init__(self, dev: torch.device, out_cap: int, d: int, block: int, ready: dict, n_left: int | None = None,
                 parent: torch.Tensor | None = None):
        super().__init__(dev, d, block, ready)
        self.n_left = n_left
        if parent is None:
            self.out, self.join = ops.join_out(out_cap, dev), ops.join_threshold
        else:       # the forest of earlier attempts is kept; the hit count and overflow counter start at 0
            self.out = (parent, torch.zeros((1,), dtype=torch.int64, device=dev), torch.zeros((1,), dtype=torch.int32, device=dev))
            self.join = ops.join_components

    def run(self, it: JoinItem, shards: list, d: int, threshold: float, cand_cap: int) -> None:
        qv, _, q_row0 = shards[it.q_shard]
        tv, _, t_row0 = shards[it.t_shard]
        if it.q_shard == it.t_shard:
            with torch.cuda.device(self.dev):
                self.join(tv, it.q_lo, it.q_hi, t_row0, tv, it.t_hi, d, threshold, t_row0, cand_cap, self.out)
            return
        target = tv[it.t_lo // ops.TILE_ROWS:]
        qdb, q_lo, q_hi, q_off, slot = self.stage(qv, it.q_lo, it.q_hi, q_row0)
        with torch.cuda.device(self.dev):
            if self.n_left is None:
                self.join(qdb, q_lo, q_hi, q_off, target, it.t_hi - it.t_lo, d, threshold, t_row0 + it.t_lo, cand_cap, self.out)
            else:
                ops.cross_join_threshold(qdb, q_lo, q_hi, q_off, target, it.t_hi - it.t_lo, d, threshold, t_row0 + it.t_lo,
                                         it.q_shard >= self.n_left, cand_cap, self.out)
        self.release(slot)


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
