"""B200VectorDB — the object `SimpleReverso.vector_db` holds instead of `QdrantClient(path=...)`.

It duck-types exactly the five qdrant-client methods core_system.py uses (SURVEY.md §8b):
  QdrantClient(path=str)                         core_system.py:100,521
  .get_collections().collections[i].name         core_system.py:104-107
  .recreate_collection(collection_name, vectors_config=VectorParams(size, distance=COSINE))   :600-603
  .upsert(collection_name, points=[PointStruct(id, vector, payload)])                          :621
  .search(collection_name, query_vector, limit, score_threshold) -> [obj(.score,.payload)]     :659-664
plus the batched entry point `search_batch` (new; reduces to `search` row by row, SURVEY.md F7).

Vectors live on the GPU(s) as L2-normalised bf16 rows in the TILED storage of include/revers_o_b200.h
([row/128][col/64][128][64]: one contiguous 16 KiB TMA box per tile; the DB is DEFINED as its bf16 values).  All arithmetic
(normalise, scan, select, re-score, merge) runs in the CUDA library; there is no CPU fallback.

ONE PROCESS, SEVERAL GPUS (SURVEY.md §8e behind the reference's own entry points): `B200VectorDB(path, devices=[0, 1, ...])`
row-shards every collection over the listed devices in whole 128-row blocks — global row = shard.row0 + local row, the id the
kernels emit directly (`id_offset`).  A search enqueues K2 on every shard's device (each on that device's stream), the packed
per-shard lists are copied to the first device and K3 merges them: `SimpleReverso.search_similar` needs nothing else to hit a
100M-row collection on 8 GPUs.  A device may be listed twice (virtual shards: exercises the path on a 1-GPU box).

Host side (tables.py): ids in one numpy array, payloads in an append-only JSONL log read lazily per hit.

PERSISTENCE is implicit, like qdrant-local's: with a `path`, `recreate_collection` / `upsert` / `upsert_batch` /
`ingest_regions` write through — only the touched 128-row blocks, the new id records and the new payload lines are appended,
then meta.json is replaced atomically (it vouches for the valid length of every file, so a crash mid-write loses at most the
last batch).  `save(other_path)` writes a full copy.  On-disk format (SURVEY.md §8f row 3): <path>/meta.json +
<collection>.bf16 (the tiled storage as is, mmap-able, loadable shard-wise by 128-row block) + <collection>.ids (fixed-width
records) + <collection>.payload.jsonl / .payload.idx.
"""
from __future__ import annotations

import json
import os
import threading
import weakref
from contextlib import contextmanager
from dataclasses import dataclass
from types import SimpleNamespace
from typing import Any, Iterable

import numpy as np
import torch

from . import _lib, ops
from ._lib import RVO_MAX_K, RvoError, check
from .tables import IdTable, PayloadStore

FORMAT = "revers_o_b200/2"


class Distance:
    COSINE = "Cosine"


@dataclass
class VectorParams:
    size: int
    distance: str = Distance.COSINE


@dataclass
class PointStruct:
    id: Any
    vector: Any
    payload: dict | None = None


@dataclass
class ScoredPoint:
    """What core_system.py:671-676 consumes: `.payload` (dict) and `.score` (float)."""
    id: Any
    version: int
    score: float
    payload: dict | None
    vector: Any = None


# `from qdrant_client.http import models` replacement: models.VectorParams / Distance / PointStruct
models = SimpleNamespace(Distance=Distance, VectorParams=VectorParams, PointStruct=PointStruct,
                         ScoredPoint=ScoredPoint)


class _RWLock:
    """Searches (readers) overlap each other; upsert / recreate / load (writers) are exclusive — a search never scans rows
    that an in-place upsert is half-way through writing (Gradio callbacks share one instance across threads, ui.py:20)."""

    def __init__(self):
        self._cond = threading.Condition(threading.Lock())
        self._readers = 0
        self._by_thread: dict = {}   # reader holds per thread: a thread that still holds one must not ask for the write side
        self._writer = None      # owning thread id (re-entrant for the writer)
        self._depth = 0

    @contextmanager
    def read(self):
        me = threading.get_ident()
        with self._cond:
            if self._writer == me:          # the writer may read its own state
                self._depth += 1
                mode = "w"
            else:
                while self._writer is not None:
                    self._cond.wait()
                self._readers += 1
                self._by_thread[me] = self._by_thread.get(me, 0) + 1
                mode = "r"
        try:
            yield
        finally:
            with self._cond:
                if mode == "w":
                    self._depth -= 1
                else:
                    self._readers -= 1
                    left = self._by_thread.get(me, 1) - 1
                    if left:
                        self._by_thread[me] = left
                    else:
                        self._by_thread.pop(me, None)
                    if self._readers == 0:
                        self._cond.notify_all()

    @contextmanager
    def write(self):
        me = threading.get_ident()
        with self._cond:
            if self._writer == me:
                self._depth += 1
            else:
                if self._by_thread.get(me):
                    # e.g. an upsert between search_batch_async() and result() on the same thread: it would wait for itself
                    raise RvoError("this thread still has searches in flight on the database: collect their results before writing")
                while self._writer is not None or self._readers > 0:
                    self._cond.wait()
                self._writer, self._depth = me, 1
        try:
            yield
        finally:
            with self._cond:
                self._depth -= 1
                if self._depth == 0:
                    self._writer = None
                    self._cond.notify_all()


class _Shard:
    """Rows [row0, row0 + n) of a collection on one device."""

    def __init__(self, device: torch.device, dim: int, row0: int = 0):
        self.device, self.dim, self.row0, self.n = device, dim, row0, 0
        self.vectors = ops.db_alloc(0, dim, device)   # tiled bf16 storage [blocks, d_pad/64, 128, 64]

    def reserve(self, rows: int) -> None:
        have = ops.db_capacity(self.vectors)
        if rows <= have:
            return
        new = ops.db_alloc(max(rows, int(have * 1.5), 1024), self.dim, self.device)
        if self.vectors.shape[0]:
            new[: self.vectors.shape[0]].copy_(self.vectors)  # whole row blocks: device-to-device memcpy
        self.vectors = new


class _Collection:
    def __init__(self, name: str, dim: int, devices: list, shard_rows: int):
        self.name, self.dim = name, int(dim)
        self.d_pad = ops.d_pad_of(self.dim)
        self.devices = devices
        self.shard_rows = max(ops.TILE_ROWS, int(shard_rows) // ops.TILE_ROWS * ops.TILE_ROWS)
        self.shards = [_Shard(dev, self.dim) for dev in devices]
        self.tail = 0                       # shard receiving appends
        self.ids = IdTable()
        self.payloads = PayloadStore()
        # persistence bookkeeping (what meta.json vouches for)
        self.dirty_blocks: set[int] = set()
        self.persisted = {"n": 0, "ids_bytes": 0, "ids_dtype": None, "log_bytes": 0, "idx_bytes": 0}

    # single-shard view used by tests / bench (`c.vectors, c.n = resident_db, rows` adopts a resident shard)
    @property
    def vectors(self) -> torch.Tensor:
        return self.shards[0].vectors

    @vectors.setter
    def vectors(self, t: torch.Tensor) -> None:
        self.shards[0].vectors = t

    @property
    def n(self) -> int:
        return sum(s.n for s in self.shards)

    @n.setter
    def n(self, v: int) -> None:
        if len(self.shards) != 1 and any(s.n for s in self.shards[1:]):
            raise RvoError("cannot set the row count of a multi-shard collection")
        self.shards[0].n = int(v)

    def locate(self, row: int) -> tuple[_Shard, int]:
        for s in self.shards:
            if s.row0 <= row < s.row0 + s.n:
                return s, row - s.row0
        raise RvoError(f"row {row} outside the collection")

    def append_plan(self, count: int) -> list[tuple[_Shard, int, int]]:
        """Where `count` new rows go: [(shard, local_row0, rows)].  A shard closes only at a multiple of 128 rows at or above
        its quota (`shard_rows`), so that every shard but the last stays a whole number of blocks (the on-disk file is the
        concatenation of the shards' blocks); the last device takes whatever is left."""
        plan = []
        while count > 0:
            s = self.shards[self.tail]
            last = self.tail == len(self.shards) - 1
            room = count if last else (self.shard_rows - s.n if s.n < self.shard_rows else (-s.n) % ops.TILE_ROWS)
            if room == 0:
                self.tail += 1
                self.shards[self.tail].row0 = s.row0 + s.n
                continue
            take = min(count, room)
            plan.append((s, s.n, take))
            s.n += take                     # reserved; the caller writes the rows or rolls back
            count -= take
        return plan


class SearchHandle:
    """A batch in flight (B200VectorDB.search_batch_async).  `result()` waits for it and returns (ids, scores, counts) as numpy
    arrays; it must be called exactly once (it also releases the collection for writers)."""

    def __init__(self, db, lock, lane, args, q_src):
        self._db, self._lock, self._lane, self._args, self._q = db, lock, lane, args, q_src

    def result(self):
        lane = self._lane
        if lane is None:
            raise RvoError("result() was already collected")
        try:
            lane.done.synchronize()
            out_i, out_s, out_c = lane.ids_np.copy(), lane.scores_np.copy(), lane.counts_np.copy()
            if out_c.min() < 0:      # overflow protocol (pathological tie mass): exact fp32 scan of the flagged queries
                vectors, n, dim, row0, k, thr = self._args
                bad = np.nonzero(out_c < 0)[0]
                qbad = lane.q_dev[torch.from_numpy(bad).to(lane.q_dev.device)].contiguous()
                a, b, cc = ops.search_topk_exact(vectors, n, dim, qbad, k, thr, row0)
                out_i[bad], out_s[bad], out_c[bad] = a.cpu().numpy(), b.cpu().numpy(), cc.cpu().numpy()
            return out_i, out_s, out_c
        finally:
            lane.busy = None
            self._lane = None
            self._lock.__exit__(None, None, None)

    def __del__(self):      # a handle dropped without result(): the collection must not stay read-locked
        if getattr(self, "_lane", None) is not None:
            try:
                self._lane.done.synchronize()
            except Exception:
                pass
            self._lane.busy = None
            self._lane = None
            try:
                self._lock.__exit__(None, None, None)
            except Exception:
                pass


class B200VectorDB:
    def __init__(self, path: str | None = None, device: str | torch.device | None = None, devices: list | None = None,
                 shard_rows: int = 1 << 22, **_):
        """path: directory to persist to / load from (None: memory only).  device: the GPU holding the vectors; devices: several
        GPUs (ordinals or torch devices) — collections are row-sharded over them; shard_rows: rows a device takes during
        incremental ingest before the next one starts (a collection LOADED from disk is split evenly instead)."""
        if not torch.cuda.is_available():
            raise RvoError("B200VectorDB needs a CUDA (sm_100) device: there is no CPU fallback")
        self.path = path
        if devices:
            self.devices = [torch.device("cuda", d) if isinstance(d, int) else torch.device(d) for d in devices]
        else:
            self.devices = [torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")]
        self.devices = [torch.device("cuda", d.index if d.index is not None else torch.cuda.current_device()) for d in self.devices]
        self.device = self.devices[0]
        self.shard_rows = shard_rows
        self.autosave = True                 # qdrant-local persists implicitly (core_system.py:521,621)
        self._lock = _RWLock()
        self._collections: dict[str, _Collection] = {}
        self._staging: dict = {}
        if path and os.path.exists(os.path.join(path, "meta.json")):
            self._load(path)

    # ---- qdrant-client surface ---------------------------------------------------------------
    def get_collections(self):
        with self._lock.read():
            return SimpleNamespace(collections=[SimpleNamespace(name=n) for n in self._collections])

    def recreate_collection(self, collection_name: str, vectors_config: VectorParams | None = None, **kw):
        size = vectors_config.size if vectors_config is not None else kw["size"]
        distance = getattr(vectors_config, "distance", Distance.COSINE)
        if str(getattr(distance, "value", distance)).lower() != "cosine":
            raise RvoError("only Distance.COSINE is supported (the reference uses no other, core_system.py:602)")
        with self._lock.write():
            self._collections[collection_name] = _Collection(collection_name, size, self.devices, self.shard_rows)
            if self.path and self.autosave:
                self._persist(self._collections[collection_name], fresh=True)
        return True

    def upsert(self, collection_name: str, points: Iterable):
        """Normalise (qdrant COSINE semantics) and append/overwrite rows.  `vector` may be a python list
        (core_system.py:608), a numpy array or a torch tensor."""
        pts = list(points)
        if not pts:
            return SimpleNamespace(status="completed")
        vecs = np.asarray([np.asarray(_get(p, "vector"), dtype=np.float32) for p in pts], dtype=np.float32)
        self._upsert_rows(collection_name, [_get(p, "id") for p in pts], torch.from_numpy(vecs),
                          [_get(p, "payload") for p in pts], assume_new=False)
        return SimpleNamespace(status="completed")

    def search(self, collection_name: str, query_vector, limit: int = 10, score_threshold: float | None = None, **_):
        """core_system.py:659-664.  One query; returns ScoredPoint-like hits, score descending."""
        q = np.asarray(query_vector, dtype=np.float32).reshape(1, -1)
        if not np.isfinite(q).all():
            raise RvoError("Wrong input: query vector has NaN / Inf components")
        ids, scores, counts = self.search_batch(collection_name, q, limit, score_threshold)
        c = self._coll(collection_name)
        n = int(counts[0])
        return [ScoredPoint(id=c.ids[int(i)], version=0, score=float(s), payload=c.payloads[int(i)])
                for i, s in zip(ids[0, :n], scores[0, :n])]

    # ---- batched entry point (new) -------------------------------------------------------------
    def search_batch(self, collection_name: str, queries, limit: int = 10, score_threshold: float | None = None,
                     as_device: bool = False):
        """queries: [Q, D] float32 (numpy / torch, host or device; a PINNED torch CPU tensor is copied to the GPU without
        a staging copy).  Returns (ids [Q,k] int64 row numbers, scores [Q,k] float32, counts [Q] int32); numpy unless
        `as_device`."""
        k = int(limit)
        if k > RVO_MAX_K:
            raise RvoError(f"limit={k} above the supported maximum {RVO_MAX_K}")
        with self._lock.read():         # held until the results are back: an in-place upsert cannot interleave with the scan
            c = self._coll(collection_name)
            active = [(s.device, s.vectors, s.n, s.row0) for s in c.shards if s.n > 0]
            if len(active) <= 1:
                dev, vectors, n, row0 = active[0] if active else (c.shards[0].device, c.shards[0].vectors, 0, 0)
                return self._search_one(c.dim, dev, vectors, n, row0, queries, k, score_threshold, as_device)
            return self._search_sharded(c.dim, active, queries, k, score_threshold, as_device)

    # ---- pipelined serving: overlap the copies / host work of one batch with the scan of another --------------------------
    def search_batch_async(self, collection_name: str, queries, limit: int = 10, score_threshold: float | None = None,
                           depth: int = 2) -> "SearchHandle":
        """Submit a batch and return at once; `handle.result()` gives what `search_batch` would have returned.  Up to `depth`
        batches are in flight per calling thread, each on its own CUDA stream with its own scratch and pinned I/O buffers:
        the host-to-device copy, the threshold-seeding kernels and the device-to-host copy of one batch run under the scan
        of another (a serving loop calls `h2 = db.search_batch_async(...); r1 = h1.result(); ...`).  Single-device collections;
        a sharded collection is served by `search_batch` (its shards already run concurrently).  queries: [Q, D] float32 numpy
        or torch CPU tensor (pinned: no staging copy)."""
        k = int(limit)
        if k > RVO_MAX_K:
            raise RvoError(f"limit={k} above the supported maximum {RVO_MAX_K}")
        if isinstance(queries, torch.Tensor):
            if queries.is_cuda:
                raise RvoError("search_batch_async takes host queries (the pipeline exists to hide their copy)")
            qh = queries.detach()
            if qh.dtype != torch.float32 or not qh.is_contiguous() or qh.dim() != 2:
                qh = qh.to(torch.float32).reshape(-1, qh.shape[-1]).contiguous()
        else:
            qa = np.ascontiguousarray(queries, dtype=np.float32)
            qh = torch.from_numpy(qa.reshape(-1, qa.shape[-1]))
        lock = self._lock.read()
        lock.__enter__()                                # released by handle.result(): no upsert rewrites rows under the scan
        try:
            c = self._coll(collection_name)
            active = [s for s in c.shards if s.n > 0]
            if len(active) > 1:
                raise RvoError("search_batch_async serves single-device collections; use search_batch for sharded ones")
            sh = active[0] if active else c.shards[0]
            self._check_dim(qh.shape[1], c.dim)
            nq = qh.shape[0]
            lanes = self._lanes(sh.device, nq, c.dim, k, depth)
            lane = lanes["ring"][lanes["next"] % depth]
            lanes["next"] += 1
            if lane.busy is not None and lane.busy() is not None:
                raise RvoError(f"more than {depth} batches in flight on this thread: collect a result first")
            lane.stream.wait_stream(torch.cuda.current_stream(sh.device))   # rows upserted on the caller's stream are complete
            with torch.cuda.stream(lane.stream):
                src = qh
                if not qh.is_pinned():
                    lane.q_stage.copy_(qh)
                    src = lane.q_stage
                lane.q_dev.copy_(src, non_blocking=True)
                ops.search_topk(sh.vectors, sh.n, c.dim, lane.q_dev, k, score_threshold, sh.row0,
                                out=(lane.ids, lane.scores, lane.counts), ws_key=("lane", id(lane)))
                lane.res_host.copy_(lane.res_dev, non_blocking=True)
                lane.done.record(lane.stream)
            h = SearchHandle(self, lock, lane, (sh.vectors, sh.n, c.dim, sh.row0, k, score_threshold), src)
            lane.busy = weakref.ref(h)      # weak: a handle dropped without result() must still run its __del__
            return h
        except BaseException:
            lock.__exit__(None, None, None)
            raise

    def _lanes(self, dev: torch.device, nq: int, d: int, k: int, depth: int):
        key = ("lanes", dev.index, nq, d, k, depth, threading.get_ident())
        L = self._staging.get(key)
        if L is None:
            nb_i, nb_s, nb_c = nq * k * 8, nq * k * 4, nq * 4
            nb = (nb_i + nb_s + nb_c + 7) // 8 * 8
            ring = []
            for _ in range(depth):
                res_dev = torch.empty(nb, dtype=torch.uint8, device=dev)
                res_host = torch.empty(nb, dtype=torch.uint8).pin_memory()
                host = res_host.numpy()
                ring.append(SimpleNamespace(
                    stream=torch.cuda.Stream(dev), done=torch.cuda.Event(), busy=None,
                    q_stage=torch.empty((nq, d), dtype=torch.float32).pin_memory(),
                    q_dev=torch.empty((nq, d), dtype=torch.float32, device=dev), res_dev=res_dev, res_host=res_host,
                    ids=res_dev[:nb_i].view(torch.int64).view(nq, k),
                    scores=res_dev[nb_i: nb_i + nb_s].view(torch.float32).view(nq, k),
                    counts=res_dev[nb_i + nb_s: nb_i + nb_s + nb_c].view(torch.int32),
                    ids_np=host[:nb_i].view(np.int64).reshape(nq, k),
                    scores_np=host[nb_i: nb_i + nb_s].view(np.float32).reshape(nq, k),
                    counts_np=host[nb_i + nb_s: nb_i + nb_s + nb_c].view(np.int32)))
            L = {"ring": ring, "next": 0}
            self._staging[key] = L
        return L

    def _check_dim(self, got: int, dim: int) -> None:
        if got != dim:
            raise RvoError(f"Wrong input: Vector dimension error: expected dim: {dim}, got {got}")

    def _search_one(self, dim, dev, vectors, n, row0, queries, k, score_threshold, as_device):
        if isinstance(queries, torch.Tensor) and queries.is_cuda:
            qd = queries.to(device=dev, dtype=torch.float32).contiguous()
            if qd.dim() == 1:
                qd = qd.unsqueeze(0)
            self._check_dim(qd.shape[1], dim)
            if as_device:
                return ops.search_topk_exact(vectors, n, dim, qd, k, score_threshold, row0)
            io = self._io_plan(dev, qd.shape[0], dim, k)
        elif (isinstance(queries, torch.Tensor) and queries.is_pinned() and queries.dtype == torch.float32
              and queries.dim() == 2 and queries.is_contiguous()):
            # caller-owned pinned host memory: DMA straight from it, no staging copy
            self._check_dim(queries.shape[1], dim)
            io = self._io_plan(dev, queries.shape[0], dim, k)
            if as_device:
                io.q_dev.copy_(queries, non_blocking=True)
                return ops.search_topk_exact(vectors, n, dim, io.q_dev, k, score_threshold, row0)
            if os.environ.get("RVO_ZC_IN", "0") == "1":
                qd = queries        # the normalise kernel reads the queries straight from the caller's pinned memory
            else:
                io.q_dev.copy_(queries, non_blocking=True)
                qd = io.q_dev
        else:
            qh = queries.detach().cpu().numpy() if isinstance(queries, torch.Tensor) else queries
            qh = np.ascontiguousarray(qh, dtype=np.float32)
            if qh.ndim == 1:
                qh = qh[None]
            self._check_dim(qh.shape[1], dim)
            # host -> pinned staging -> device, all on the current stream; the views are cached per (Q, D, k) and thread
            io = self._io_plan(dev, qh.shape[0], dim, k)
            np.copyto(io.q_stage_np, qh)
            if as_device:
                io.q_dev.copy_(io.q_stage, non_blocking=True)
                return ops.search_topk_exact(vectors, n, dim, io.q_dev, k, score_threshold, row0)
            if os.environ.get("RVO_ZC_IN", "0") == "1":
                qd = io.q_stage     # pinned staging: the normalise kernel reads it over PCIe, no H2D copy launch
            else:
                io.q_dev.copy_(io.q_stage, non_blocking=True)
                qd = io.q_dev
        # results land in ONE blob [ids int64 | scores f32 | counts i32]: a device blob + one D2H copy by default.  With
        # RVO_ZC_OUT=1 the last kernel stores straight into the pinned host blob (and with RVO_ZC_IN=1 the first kernel reads
        # the queries from pinned host memory): measured equal within noise on one GPU and 30-40 us per step WORSE with two
        # processes on one box, so the copies stay the default
        if qd is io.q_dev:
            # the steady state of a serving loop: same shape, same DB, same threshold -> a prepared call (one ctypes call)
            key = (vectors.data_ptr(), n, row0, score_threshold, _lib.option_epoch)
            if io.prepared_key != key:
                io.prepared = ops.PreparedSearch(vectors, n, dim, io.q_dev, k, score_threshold, row0,
                                                 out=(io.ids, io.scores, io.counts))
                io.prepared_key = key
            io.prepared()
        else:
            ops.search_topk(vectors, n, dim, qd, k, score_threshold, row0, out=(io.ids, io.scores, io.counts))
        if io.res_dev is not io.res_host:
            io.res_host.copy_(io.res_dev, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
        out_i, out_s, out_c = io.ids_np.copy(), io.scores_np.copy(), io.counts_np.copy()
        if out_c.min() < 0:  # overflow protocol of rvo_search_topk: exact fp32 scan in batches of <= RVO_SMALL_Q
            bad = np.nonzero(out_c < 0)[0]
            qbad = qd[torch.from_numpy(bad).to(qd.device)].to(dev).contiguous()
            a, b, cc = ops.search_topk_exact(vectors, n, dim, qbad, k, score_threshold, row0)
            out_i[bad], out_s[bad], out_c[bad] = a.cpu().numpy(), b.cpu().numpy(), cc.cpu().numpy()
        return out_i, out_s, out_c

    def _search_sharded(self, dim, active, queries, k, score_threshold, as_device):
        """Row-sharded search in ONE process (SURVEY.md §8e): K2 on every shard's device, each on its own stream; the packed
        [ids | scores | counts] blobs are copied to the first shard's device (peer copies over NVLink) and K3 merges them."""
        root = active[0][0]
        if isinstance(queries, torch.Tensor):
            q_src = queries.detach().to(dtype=torch.float32)
            if q_src.dim() == 1:
                q_src = q_src.unsqueeze(0)
            q_src = q_src.contiguous()
        else:
            q_src = torch.from_numpy(np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, np.shape(queries)[-1]))
        nq = q_src.shape[0]
        self._check_dim(q_src.shape[1], dim)
        G = len(active)
        plan = self._shard_plan(tuple(d.index for d, _, _, _ in active), nq, dim, k)
        if not q_src.is_cuda and not q_src.is_pinned():
            plan.q_stage.copy_(q_src)
            q_src = plan.q_stage
        lib = _lib.load()
        for g, (dev, vectors, n, row0) in enumerate(active):
            with torch.cuda.device(dev):
                plan.q_dev[g].copy_(q_src, non_blocking=True)
                ops.search_topk(vectors, n, dim, plan.q_dev[g], k, score_threshold, row0, out=plan.views[g])
            # ordered after shard g's search on ITS stream and before the merge on the root's stream
            plan.gathered[g].copy_(plan.blobs[g], non_blocking=True)
        with torch.cuda.device(root):
            check(lib.rvo_merge_topk_packed(plan.gathered.data_ptr(), plan.gathered.stride(0), G, nq, k, plan.out_ids.data_ptr(),
                                            plan.out_scores.data_ptr(), plan.out_counts.data_ptr(),
                                            torch.cuda.current_stream(root).cuda_stream), "rvo_merge_topk_packed")
            bad = (plan.out_counts < 0).nonzero().flatten()           # one host sync: also the end of the search
            if bad.numel():
                # overflow protocol, sharded: the flagged queries go through the exact fp32 scan on every shard, merged again
                parts = []
                for g, (dev, vectors, n, row0) in enumerate(active):
                    with torch.cuda.device(dev):
                        qb = plan.q_dev[g][bad.to(dev)].contiguous()
                        parts.append(ops.search_topk_exact(vectors, n, dim, qb, k, score_threshold, row0))
                gi = torch.stack([p[0].to(root) for p in parts])
                gs = torch.stack([p[1].to(root) for p in parts])
                gc = torch.stack([p[2].to(root) for p in parts])
                a, b, cc = ops.merge_topk(gi, gs, gc, k)
                plan.out_ids[bad], plan.out_scores[bad], plan.out_counts[bad] = a, b, cc
            if as_device:
                return plan.out_ids.clone(), plan.out_scores.clone(), plan.out_counts.clone()
            plan.res_host.copy_(plan.res_dev, non_blocking=True)
            torch.cuda.current_stream(root).synchronize()
            return plan.ids_np.copy(), plan.scores_np.copy(), plan.counts_np.copy()

    def _shard_plan(self, dev_indices: tuple, nq: int, d: int, k: int):
        key = ("shards", dev_indices, nq, d, k, threading.get_ident())
        p = self._staging.get(key)
        if p is None:
            nb_i, nb_s, nb_c = nq * k * 8, nq * k * 4, nq * 4
            nb = (nb_i + nb_s + nb_c + 7) // 8 * 8
            root = torch.device("cuda", dev_indices[0])
            blobs = [torch.zeros(nb, dtype=torch.uint8, device=torch.device("cuda", i)) for i in dev_indices]

            def views(b):
                return (b[:nb_i].view(torch.int64).view(nq, k), b[nb_i: nb_i + nb_s].view(torch.float32).view(nq, k),
                        b[nb_i + nb_s: nb_i + nb_s + nb_c].view(torch.int32))
            res_dev = torch.empty(nb, dtype=torch.uint8, device=root)
            res_host = torch.empty(nb, dtype=torch.uint8).pin_memory()
            host = res_host.numpy()
            oi, os_, oc = views(res_dev)
            p = SimpleNamespace(
                q_stage=torch.empty((nq, d), dtype=torch.float32).pin_memory(),
                q_dev=[torch.empty((nq, d), dtype=torch.float32, device=torch.device("cuda", i)) for i in dev_indices],
                blobs=blobs, views=[views(b) for b in blobs],
                gathered=torch.empty((len(dev_indices), nb), dtype=torch.uint8, device=root),
                res_dev=res_dev, res_host=res_host, out_ids=oi, out_scores=os_, out_counts=oc,
                ids_np=host[:nb_i].view(np.int64).reshape(nq, k),
                scores_np=host[nb_i: nb_i + nb_s].view(np.float32).reshape(nq, k),
                counts_np=host[nb_i + nb_s: nb_i + nb_s + nb_c].view(np.int32))
            if len(self._staging) > 64:
                self._staging.clear()
            self._staging[key] = p
        return p

    def _io_plan(self, dev: torch.device, nq: int, d: int, k: int):
        """Pinned staging + device buffers + every view of them for one (Q, D, k) shape, per calling thread; building the
        ~20 tensor/numpy views costs more host time than the copies they describe, so they are made once."""
        key = ("io", dev.index, nq, d, k, threading.get_ident())
        io = self._staging.get(key)
        if io is None:
            nb_i, nb_s, nb_c = nq * k * 8, nq * k * 4, nq * 4
            nb = (nb_i + nb_s + nb_c + 7) // 8 * 8
            q_stage = torch.empty((nq, d), dtype=torch.float32).pin_memory()
            res_host = torch.empty(nb, dtype=torch.uint8).pin_memory()     # device-addressable (UVA): kernels write into it
            # a small result blob (the UI's Q = 1: 124 bytes) is written by the last kernel straight into the pinned host blob:
            # one copy launch less per search; larger blobs go through a device blob + one D2H copy (measured no worse)
            zc_out = os.environ.get("RVO_ZC_OUT", "auto")
            zero_copy = zc_out == "1" or (zc_out == "auto" and nb <= 16384)
            res_dev = res_host if zero_copy else torch.empty(nb, dtype=torch.uint8, device=dev)
            host = res_host.numpy()
            io = SimpleNamespace(
                q_stage=q_stage, q_stage_np=q_stage.numpy(), prepared=None, prepared_key=None,
                q_dev=torch.empty((nq, d), dtype=torch.float32, device=dev),
                res_dev=res_dev, res_host=res_host,
                ids=res_dev[:nb_i].view(torch.int64).view(nq, k),
                scores=res_dev[nb_i: nb_i + nb_s].view(torch.float32).view(nq, k),
                counts=res_dev[nb_i + nb_s: nb_i + nb_s + nb_c].view(torch.int32),
                ids_np=host[:nb_i].view(np.int64).reshape(nq, k),
                scores_np=host[nb_i: nb_i + nb_s].view(np.float32).reshape(nq, k),
                counts_np=host[nb_i + nb_s: nb_i + nb_s + nb_c].view(np.int32))
            if len(self._staging) > 64:      # shapes come and go (UI: Q = 1; batch jobs: a few sizes): keep the cache bounded
                self._staging.clear()
            self._staging[key] = io
        return io

    # ---- ingest ------------------------------------------------------------------------------------
    def _upsert_rows(self, collection_name: str, ids: list, vectors: torch.Tensor, payloads: list, assume_new: bool,
                     persist: bool | None = None) -> None:
        with self._lock.write():
            c = self._coll(collection_name)
            if vectors.dim() != 2 or vectors.shape[1] != c.dim or vectors.shape[0] != len(ids):
                got = vectors.shape[-1] if vectors.dim() else 0
                if vectors.dim() == 2 and vectors.shape[0] == len(ids):
                    raise RvoError(f"Wrong input: Vector dimension error: expected dim: {c.dim}, got {got}")
                raise RvoError(f"upsert: bad shape {tuple(vectors.shape)} for {len(ids)} ids, dim {c.dim}")
            n_before = c.n
            shard_n = [s.n for s in c.shards]
            tail_before = c.tail
            try:
                rows = c.ids.append(ids, assume_new=assume_new)          # existing ids keep their row (overwrite)
                n_new = len(c.ids) - n_before
                plan = c.append_plan(n_new)
                # destination of every input vector: new rows in plan order, old rows wherever they live
                dst: list[tuple[_Shard, int]] = [None] * len(ids)        # type: ignore[list-item]
                new_dst = [(s, lr + i) for s, lr, cnt in plan for i in range(cnt)]
                last_of_row: dict[int, int] = {}
                for j, r in enumerate(rows.tolist()):
                    last_of_row[r] = j                                   # a row written twice in one batch: the last vector wins
                for r, j in last_of_row.items():
                    dst[j] = new_dst[r - n_before] if r >= n_before else c.locate(r)
                for s, _, _ in plan:
                    s.reserve(s.n)
                self._write_rows(c, dst, vectors)
                c.payloads.append_or_set(rows, payloads)
                for r in set(rows.tolist()):
                    c.dirty_blocks.add(r // ops.TILE_ROWS)
            except BaseException:
                # the host tables must never run ahead of the vectors actually written
                c.ids.truncate(n_before)
                c.payloads.truncate(n_before)
                for s, n0 in zip(c.shards, shard_n):
                    s.n = n0
                c.tail = tail_before
                raise
            if self.path and (self.autosave if persist is None else persist):
                self._persist(c)

    def upsert_batch(self, collection_name: str, ids: list, vectors, payloads: list | None = None, assume_new: bool = False,
                     persist: bool | None = None):
        """Bulk ingest (SURVEY.md §8f row 2): tensors in, no python float lists.  `assume_new` skips the id lookup (freshly
        generated ids); `persist=False` defers the write-through to an explicit `save()`."""
        v = vectors if isinstance(vectors, torch.Tensor) else torch.from_numpy(np.asarray(vectors, np.float32))
        self._upsert_rows(collection_name, list(ids), v, list(payloads) if payloads is not None else [None] * len(ids),
                          assume_new, persist)

    def ingest_regions(self, collection_name: str, feats: torch.Tensor, masks: torch.Tensor, payload_fn=None,
                       max_regions: int = 0, persist: bool | None = None):
        """Batched ingest (SURVEY.md §8f row 2): patch features [B,P,D] bf16 / fp16 + patch-grid masks [B,M,P] uint8 on the GPU ->
        every non-empty region's mask-pooled, L2-normalised embedding appended to the collection by ONE kernel that writes
        bf16 rows straight into the tiled DB (no fp32 embeddings in HBM, no python float lists, core_system.py:363-408 +
        :596-622).  `payload_fn(image_index, region_index) -> (id, payload)`; default: uuid4 id, {"image": b, "region": m}.
        Returns the number of rows appended."""
        import uuid
        with self._lock.write():
            c = self._coll(collection_name)
            B, P, D = feats.shape
            M = masks.shape[1]
            self._check_dim(D, c.dim)
            lim = M if max_regions <= 0 else min(M, max_regions)
            s = c.shards[c.tail]
            if c.tail + 1 < len(c.shards) and s.n >= c.shard_rows and s.n % ops.TILE_ROWS == 0:
                c.tail += 1
                c.shards[c.tail].row0 = s.row0 + s.n
                s = c.shards[c.tail]
            if feats.device != s.device:
                feats, masks = feats.to(s.device), masks.to(s.device)
            s.reserve(s.n + B * lim)
            counts, src, total, _ = ops.mask_pool_to_db(feats, masks, s.vectors, s.n, max_regions)
            m = int(total.item())                      # the one host sync of an ingest batch
            origin = src[:m].cpu().numpy()
            new_ids, pays = [], []
            for o in origin:
                b, r = divmod(int(o), M)
                pid, pay = payload_fn(b, r) if payload_fn else (str(uuid.uuid4()), {"image": b, "region": r})
                new_ids.append(pid)
                pays.append(pay)
            g0 = s.row0 + s.n
            rows = c.ids.append(new_ids, assume_new=True)
            assert len(rows) == 0 or (rows[0] == g0 and rows[-1] == g0 + m - 1), "region ids must be new"
            c.payloads.append_or_set(rows, pays)
            s.n += m
            for blk in range(g0 // ops.TILE_ROWS, (g0 + m + ops.TILE_ROWS - 1) // ops.TILE_ROWS):
                c.dirty_blocks.add(blk)
            if self.path and (self.autosave if persist is None else persist):
                self._persist(c)
            return m

    def find_near_duplicates(self, collection_name: str, threshold: float = 0.95, max_pairs: int = 1 << 22):
        """All pairs of stored points with cosine >= threshold (BASELINE config 4: keyframe near-duplicate self-join;
        generalises `score_threshold`, core_system.py:663).  Returns (list of (id_a, id_b), scores float32 [n]).  A row with more
        near-duplicates than the candidate lists hold (a static scene: thousands of identical frames) is re-joined exactly with
        a larger list instead of failing.  A row-sharded collection is joined where it lives (`sharded.selfjoin_sharded`: each
        shard with itself on its device, every pair of shards split between their two devices, only 4096-row query blocks
        copied), with the same pairs and scores as on one device."""
        with self._lock.read():
            c = self._coll(collection_name)
            active = [s for s in c.shards if s.n]
            if len(active) > 1:
                from .sharded import selfjoin_sharded
                p, sc = selfjoin_sharded([(s.vectors, s.n, s.row0) for s in active], c.dim, threshold, max_pairs=max_pairs)
                return [(c.ids[int(a)], c.ids[int(b)]) for a, b in p], sc
            s = next((s for s in c.shards if s.n), c.shards[0])
            n, vectors = s.n, s.vectors
            if n < 2:
                return [], np.zeros(0, np.float32)
            p, sc = ops.selfjoin_exact(vectors, n, c.dim, threshold, max_pairs=max_pairs, id_offset=s.row0)
            return [(c.ids[int(a)], c.ids[int(b)]) for a, b in p], sc

    def count(self, collection_name: str) -> int:
        return self._coll(collection_name).n

    def rebalance(self, collection_name: str) -> None:
        """Spread the rows evenly over the devices (whole 128-row blocks, `sharded.shard_bounds`): device-to-device copies."""
        from .sharded import shard_bounds
        with self._lock.write():
            c = self._coll(collection_name)
            n, G = c.n, len(c.shards)
            if G == 1 or n == 0:
                return
            old = [(s.row0, s.n, s.vectors) for s in c.shards if s.n]
            new_shards = []
            for g, dev in enumerate(c.devices):
                lo, hi = shard_bounds(n, G, g)
                ns = _Shard(dev, c.dim, lo)
                ns.reserve(max(hi - lo, 1))
                ns.n = hi - lo
                for row0, cnt, vec in old:          # block-aligned overlaps of [lo, hi) with the old shard
                    a, b = max(lo, row0), min(hi, row0 + cnt)
                    if a >= b:
                        continue
                    b_blk = (b + ops.TILE_ROWS - 1) // ops.TILE_ROWS
                    src = vec[(a - row0) // ops.TILE_ROWS: b_blk - row0 // ops.TILE_ROWS]
                    ns.vectors[(a - lo) // ops.TILE_ROWS: (a - lo) // ops.TILE_ROWS + src.shape[0]].copy_(src)
                new_shards.append(ns)
            for dev in {s.device for s in new_shards}:
                torch.cuda.synchronize(dev)
            c.shards = new_shards
            c.tail = max((g for g, s in enumerate(new_shards) if s.n), default=0)

    # ---- persistence -----------------------------------------------------------------------------
    def _files(self, path: str, name: str) -> dict:
        return {k: os.path.join(path, f"{name}.{ext}") for k, ext in
                (("vec", "bf16"), ("ids", "ids"), ("log", "payload.jsonl"), ("idx", "payload.idx"))}

    def _write_blocks(self, c: _Collection, vec_path: str, blocks: list) -> None:
        nk = c.d_pad // ops.TILE_COLS
        blk_bytes = nk * ops.TILE_ROWS * ops.TILE_COLS * 2
        if not blocks:
            return
        if not os.path.exists(vec_path):
            open(vec_path, "wb").close()
        with open(vec_path, "r+b") as fh:
            i = 0
            while i < len(blocks):
                j = i + 1
                while j < len(blocks) and blocks[j] == blocks[j - 1] + 1 and j - i < 4096:
                    j += 1
                b0, b1 = blocks[i], blocks[j - 1] + 1
                for s in c.shards:               # the run may straddle shards (each is whole blocks but the last)
                    s_b0 = s.row0 // ops.TILE_ROWS
                    s_b1 = s_b0 + (s.n + ops.TILE_ROWS - 1) // ops.TILE_ROWS
                    lo, hi = max(b0, s_b0), min(b1, s_b1)
                    if lo < hi:
                        raw = s.vectors[lo - s_b0: hi - s_b0].contiguous().view(torch.int16).cpu().numpy()
                        fh.seek(lo * blk_bytes)
                        fh.write(raw.tobytes())
                i = j

    @staticmethod
    def _write_meta(path: str, c: _Collection, st: dict, drop_others: bool = False) -> None:
        """meta.json is the only file that says how much of the others is valid; replaced atomically, last."""
        meta_path = os.path.join(path, "meta.json")
        meta = {"format": FORMAT, "collections": {}}
        if os.path.exists(meta_path) and not drop_others:
            try:
                with open(meta_path) as fh:
                    old = json.load(fh)
                if old.get("format") == FORMAT:
                    meta["collections"] = old.get("collections", {})
            except Exception:
                pass
        n = st["n"]
        meta["collections"][c.name] = {
            "dim": c.dim, "d_pad": c.d_pad, "n": n, "distance": "Cosine", "layout": "tiled[block][d_pad/64][128][64] bf16",
            "blocks": (n + ops.TILE_ROWS - 1) // ops.TILE_ROWS, "id_kind": c.ids.kind, "ids_dtype": st["ids_dtype"],
            "ids_bytes": st["ids_bytes"], "log_bytes": st["log_bytes"], "idx_bytes": st["idx_bytes"]}
        tmp = meta_path + ".tmp"
        with open(tmp, "w") as fh:
            json.dump(meta, fh)
            fh.flush()
            os.fsync(fh.fileno())
        os.replace(tmp, meta_path)

    def _persist(self, c: _Collection, fresh: bool = False) -> None:
        """Write-through of one collection to self.path: dirty 128-row blocks, new id records, new payload lines; meta.json
        last, atomically.  O(batch), not O(collection)."""
        path = self.path
        os.makedirs(path, exist_ok=True)
        f = self._files(path, c.name)
        if fresh:
            for p in f.values():
                open(p, "wb").close()
            c.persisted = {"n": 0, "ids_bytes": 0, "ids_dtype": None, "log_bytes": 0, "idx_bytes": 0}
        st = dict(c.persisted)
        n = c.n
        self._write_blocks(c, f["vec"], sorted(c.dirty_blocks))
        dt = c.ids.disk_dtype()
        if dt is not None and len(c.ids) >= n:
            arr = c.ids.array()[:n]
            if st["ids_dtype"] != dt or st["n"] > n or not os.path.exists(f["ids"]):
                with open(f["ids"], "wb") as fh:      # first write, or a widened column (longer strings): rewrite
                    fh.write(arr.tobytes())
            else:
                with open(f["ids"], "r+b") as fh:
                    fh.truncate(st["ids_bytes"])
                    fh.seek(st["ids_bytes"])
                    fh.write(arr[st["n"]:].tobytes())
            st["ids_dtype"], st["ids_bytes"] = dt, arr.nbytes
        elif dt is None and st["ids_dtype"] is not None:
            # the ids stopped fitting a typed column (an int id joined uuid strings, or the other way round): from now on they
            # live in the log records, so every row persisted so far gets a fresh record carrying its id, and the stale column
            # is no longer vouched for
            c.payloads.mark_all_dirty(st["n"])
            st["ids_dtype"], st["ids_bytes"] = None, 0
        st["log_bytes"], st["idx_bytes"] = c.payloads.flush(f["log"], f["idx"], st["log_bytes"], st["idx_bytes"], ids=c.ids)
        st["n"] = n
        self._write_meta(path, c, st)
        c.persisted = st
        c.dirty_blocks = set()

    def _export(self, c: _Collection, path: str, first: bool) -> None:
        """Full copy of one collection into another directory; the live collection's own bookkeeping is untouched."""
        os.makedirs(path, exist_ok=True)
        f = self._files(path, c.name)
        for p in f.values():
            open(p, "wb").close()
        n = c.n
        self._write_blocks(c, f["vec"], list(range((n + ops.TILE_ROWS - 1) // ops.TILE_ROWS)))
        st = {"n": n, "ids_bytes": 0, "ids_dtype": None, "log_bytes": 0, "idx_bytes": 0}
        dt = c.ids.disk_dtype()
        have_ids = len(c.ids) >= n
        if dt is not None and have_ids:
            arr = c.ids.array()[:n]
            with open(f["ids"], "wb") as fh:
                fh.write(arr.tobytes())
            st["ids_dtype"], st["ids_bytes"] = dt, arr.nbytes
        rows = min(n, len(c.payloads))
        pairs = np.empty((rows, 2), np.int64)
        pos = 0
        with open(f["log"], "wb") as fh:
            for r in range(rows):
                rec = {"row": r, "payload": c.payloads[r]}
                if dt is None and have_ids:
                    rec["id"] = c.ids[r]
                line = (json.dumps(rec, default=str) + "\n").encode("utf-8")
                fh.write(line)
                pairs[r] = (r, pos)
                pos += len(line)
        with open(f["idx"], "wb") as fh:
            fh.write(pairs.tobytes())
        st["log_bytes"], st["idx_bytes"] = pos, pairs.nbytes
        self._write_meta(path, c, st, drop_others=first)

    def save(self, path: str | None = None) -> None:
        """With no argument (or this DB's own path): flush whatever is not on disk yet.  With another directory: a full copy."""
        path = path or self.path
        if not path:
            raise RvoError("no path to save to")
        with self._lock.write():
            if self.path and os.path.abspath(path) == os.path.abspath(self.path):
                for c in self._collections.values():
                    self._persist(c)
                return
            os.makedirs(path, exist_ok=True)
            for i, c in enumerate(self._collections.values()):
                self._export(c, path, first=(i == 0))
            if not self._collections:
                with open(os.path.join(path, "meta.json"), "w") as fh:
                    json.dump({"format": FORMAT, "collections": {}}, fh)

    def _load(self, path: str) -> None:
        from .sharded import shard_bounds
        with open(os.path.join(path, "meta.json")) as f:
            meta = json.load(f)
        v1 = meta.get("format", "revers_o_b200/1") != FORMAT
        with self._lock.write():
            for name, m in meta.get("collections", {}).items():
                c = _Collection(name, m["dim"], self.devices, self.shard_rows)
                n = int(m["n"])
                files = self._files(path, name)
                G = len(self.devices)
                for g, s in enumerate(c.shards):          # split evenly over the devices, whole blocks
                    lo, hi = shard_bounds(n, G, g)
                    s.row0, s.n = lo, hi - lo
                    if hi > lo:
                        view, _, _, _ = read_shard_blocks(path, name, G, g)
                        s.reserve(hi - lo)
                        _copy_blocks_to_device(view, s.vectors)
                c.tail = max((g for g, s in enumerate(c.shards) if s.n), default=0)
                if v1:      # round-1 files: one JSON line {"id", "payload"} per row
                    ids, pays = [], []
                    with open(files["log"]) as f:
                        for line in f:
                            rec = json.loads(line)
                            ids.append(rec["id"])
                            pays.append(rec["payload"])
                    rows = c.ids.append(ids[:n], assume_new=True)
                    c.payloads.append_or_set(rows, pays[:n])
                    c.dirty_blocks = set(range((n + ops.TILE_ROWS - 1) // ops.TILE_ROWS))
                else:
                    if m.get("ids_dtype"):
                        arr = np.fromfile(files["ids"], dtype=np.dtype(m["ids_dtype"]), count=n)
                        if len(arr) != n:
                            raise RvoError(f"{files['ids']}: {len(arr)} ids on disk, meta.json says {n}")
                        c.ids = IdTable.from_array(arr)
                    c.payloads = PayloadStore.open(files["log"], files["idx"], n, int(m.get("idx_bytes", 0)))
                    if not m.get("ids_dtype") and n:      # object ids live in the log
                        vals = []
                        with open(files["log"], "rb") as f:
                            data = f.read(int(m.get("log_bytes", 0)))
                        byrow = {}
                        for line in data.splitlines():
                            rec = json.loads(line)
                            byrow[rec["row"]] = rec.get("id")
                        vals = [byrow.get(r) for r in range(n)]
                        c.ids = IdTable()
                        c.ids.append(vals, assume_new=True)
                    c.persisted = {"n": n, "ids_bytes": int(m.get("ids_bytes", 0)), "ids_dtype": m.get("ids_dtype"),
                                   "log_bytes": int(m.get("log_bytes", 0)), "idx_bytes": int(m.get("idx_bytes", 0))}
                self._collections[name] = c

    def close(self) -> None:
        for c in self._collections.values():
            c.payloads.close()

    # ---- helpers ---------------------------------------------------------------------------------
    def _coll(self, name: str) -> _Collection:
        c = self._collections.get(name)
        if c is None:
            raise RvoError(f"Collection {name} not found")
        return c

    @staticmethod
    def _to_device_f32(x, device) -> torch.Tensor:
        if isinstance(x, torch.Tensor):
            t = x.to(dtype=torch.float32)
        else:
            t = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
        if t.dim() == 1:
            t = t.unsqueeze(0)
        if not t.is_cuda:
            t = t.pin_memory().to(device, non_blocking=True) if t.numel() > 4096 else t.to(device)
        elif t.device != device:
            t = t.to(device)
        return t.contiguous()

    def _write_rows(self, c: _Collection, dst: list, host_or_dev: torch.Tensor) -> None:
        """Normalise-and-store: one launch per run of consecutive destination rows on the same shard.  `dst[j]` is the
        (shard, local row) of input vector j, or None when a later vector of the batch overwrites the same row."""
        per_dev: dict = {}
        i, n = 0, len(dst)
        while i < n:
            if dst[i] is None:
                i += 1
                continue
            s, r = dst[i]
            j = i + 1
            while j < n and dst[j] is not None and dst[j][0] is s and dst[j][1] == dst[j - 1][1] + 1:
                j += 1
            src = per_dev.get(s.device)
            if src is None:
                src = per_dev[s.device] = self._to_device_f32(host_or_dev, s.device)
            with torch.cuda.device(s.device):
                ops.normalize_rows(src[i:j], db=s.vectors, row0=r)
            i = j


def _copy_blocks_to_device(view: np.ndarray, dst: torch.Tensor, chunk_blocks: int = 4096) -> None:
    """memmap'd tiled blocks -> device, `chunk_blocks` at a time through a pinned staging buffer."""
    if view.shape[0] == 0:
        return
    dev = dst.device
    stage = torch.empty((min(chunk_blocks, view.shape[0]),) + tuple(view.shape[1:]), dtype=torch.int16).pin_memory()
    for b0 in range(0, view.shape[0], chunk_blocks):
        b1 = min(view.shape[0], b0 + chunk_blocks)
        stage[: b1 - b0].numpy()[...] = view[b0:b1]
        dst[b0:b1].copy_(stage[: b1 - b0].view(torch.bfloat16), non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()      # the staging buffer is reused by the next chunk


def read_shard_blocks(path: str, collection_name: str, world: int, rank: int):
    """On-disk format, shard-wise (SURVEY.md §8f row 3): memory-map `<path>/<collection>.bf16` (the tiled storage as is) and
    return (view int16 [blocks_of_this_rank, d_pad/64, 128, 64], n_local, first_global_row, dim) for rank `rank` of `world`
    — whole 128-row blocks, the same split as `sharded.shard_bounds`.  Pure host code (numpy), no copy until the caller
    reads the view; each GPU process of a box maps only its slice of the file."""
    from .sharded import shard_bounds
    with open(os.path.join(path, "meta.json")) as f:
        meta = json.load(f)
    m = meta.get("collections", {}).get(collection_name)
    if m is None:
        raise RvoError(f"Collection {collection_name} not found")
    n, dim, d_pad = int(m["n"]), int(m["dim"]), int(m["d_pad"])
    nk = d_pad // ops.TILE_COLS
    blocks = (n + ops.TILE_ROWS - 1) // ops.TILE_ROWS
    lo, hi = shard_bounds(n, world, rank)
    b0, b1 = lo // ops.TILE_ROWS, (hi + ops.TILE_ROWS - 1) // ops.TILE_ROWS
    if blocks == 0 or hi <= lo:
        return np.zeros((0, nk, ops.TILE_ROWS, ops.TILE_COLS), np.int16), 0, lo, dim
    mm = np.memmap(os.path.join(path, f"{collection_name}.bf16"), dtype=np.int16, mode="r",
                   shape=(blocks, nk, ops.TILE_ROWS, ops.TILE_COLS))
    return mm[b0:b1], hi - lo, lo, dim


def _get(p, name):
    return getattr(p, name) if hasattr(p, name) else p[name]
