"""Tensor-level wrappers over the C ABI.  PyTorch is used for device-memory ownership and streams only;
every arithmetic step runs in the hand-written CUDA library (no torch ops on the data path)."""
from __future__ import annotations

import math
import threading

import torch

from . import _lib
from ._lib import RVO_MAX_K, RVO_SMALL_Q, RvoError, check

_ws_lock = threading.Lock()
_workspaces: dict = {}
_ws_bytes: dict = {}      # (n_rows, d, nq, k) -> rvo_search_workspace_bytes (depends on the tuning options: see set_option)


def _stream(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _ptr(t) -> int:
    return 0 if t is None else t.data_ptr()


def workspace(device: torch.device, nbytes: int, key=None) -> torch.Tensor:
    """Per-(device, thread[, key]) scratch buffer, grown on demand, 1024-byte aligned (torch allocations are 512-byte
    aligned, so one KiB of slack is kept and the view is offset).  Calls that may run CONCURRENTLY on different streams of one
    thread (pipelined searches) pass a `key` so that they do not share scratch."""
    key = (device.index if device.index is not None else torch.cuda.current_device(), threading.get_ident(), key)
    with _ws_lock:
        buf = _workspaces.get(key)
        if buf is None or buf.numel() < nbytes + 1024:
            buf = torch.empty(int(nbytes * 1.25) + 2048, dtype=torch.uint8, device=device)
            _workspaces[key] = buf
    off = (-buf.data_ptr()) % 1024
    return buf[off:off + nbytes]


def _feat_dtype(t: torch.Tensor) -> int:
    return _lib.RVO_DTYPE_F16 if t.dtype == torch.float16 else _lib.RVO_DTYPE_BF16


def require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise RvoError(f"{name} must be a CUDA tensor: the B200 library has no CPU path")


def d_pad_of(d: int) -> int:
    return (d + 63) // 64 * 64


TILE_ROWS, TILE_COLS = 128, 64


def db_alloc(n_rows: int, d: int, device) -> torch.Tensor:
    """Zeroed tiled DB storage for n_rows rows: bf16 [ceil(n/128), d_pad/64, 128, 64] (include/revers_o_b200.h,
    "DB storage layout"): every (row block, k-chunk) tile is one contiguous 16 KiB TMA box."""
    return torch.zeros(((n_rows + TILE_ROWS - 1) // TILE_ROWS, d_pad_of(d) // TILE_COLS, TILE_ROWS, TILE_COLS),
                       dtype=torch.bfloat16, device=device)


def db_capacity(db: torch.Tensor) -> int:
    return db.shape[0] * TILE_ROWS


def tile_rows(x: torch.Tensor) -> torch.Tensor:
    """Row-major bf16 [n, d] -> tiled storage (layout conversion for inputs/IO; a pure permutation)."""
    n, d = x.shape
    out = db_alloc(n, d, x.device)
    nb, nk = out.shape[0], out.shape[1]
    pad = torch.zeros((nb * TILE_ROWS, nk * TILE_COLS), dtype=torch.bfloat16, device=x.device)
    pad[:n, :d] = x
    out.copy_(pad.view(nb, TILE_ROWS, nk, TILE_COLS).permute(0, 2, 1, 3))
    return out


def untile_rows(db: torch.Tensor, n: int, d: int, rows: torch.Tensor | None = None) -> torch.Tensor:
    """Tiled storage -> row-major bf16 [n, d] (or the given rows).  Checker/IO utility, not on the product path."""
    nb, nk = db.shape[0], db.shape[1]
    if rows is not None:
        return db[rows // TILE_ROWS, :, rows % TILE_ROWS, :].reshape(rows.numel(), nk * TILE_COLS)[:, :d]
    return db.permute(0, 2, 1, 3).reshape(nb * TILE_ROWS, nk * TILE_COLS)[:n, :d]


def normalize_rows(src: torch.Tensor, dst_bf16: torch.Tensor | None = None, want_f32: bool = False,
                   db: torch.Tensor | None = None, row0: int = 0):
    """L2-normalise fp32 rows (core_system.py:407,447; qdrant COSINE upsert).
    `db` given: write the rows into the tiled DB at rows row0..row0+n-1 and return (db, f32|None);
    otherwise return (row-major bf16 [n, d_pad], f32|None)."""
    require_cuda(src, "src")
    assert src.dtype == torch.float32 and src.dim() == 2 and src.stride(1) == 1
    n, d = src.shape
    f32 = torch.empty((n, d), dtype=torch.float32, device=src.device) if want_f32 else None
    lib = _lib.load()
    if db is not None:
        assert db.dtype == torch.bfloat16 and db.is_contiguous() and db.dim() == 4 and row0 + n <= db_capacity(db)
        assert db.shape[1] * TILE_COLS == d_pad_of(d)
        check(lib.rvo_normalize_rows(_ptr(src), n, d, src.stride(0), _ptr(db), d_pad_of(d), int(row0), _ptr(f32),
                                     _stream(src.device)), "rvo_normalize_rows")
        return db, f32
    if dst_bf16 is None:
        dst_bf16 = torch.empty((n, d_pad_of(d)), dtype=torch.bfloat16, device=src.device)
    assert dst_bf16.dtype == torch.bfloat16 and dst_bf16.shape[0] >= n and dst_bf16.stride(1) == 1
    check(lib.rvo_normalize_rows(_ptr(src), n, d, src.stride(0), _ptr(dst_bf16), dst_bf16.stride(0), -1, _ptr(f32),
                                 _stream(src.device)), "rvo_normalize_rows")
    return dst_bf16, f32


def mask_pool(feats: torch.Tensor, masks: torch.Tensor, max_regions: int = 0, out=None, ws_key=None):
    """K1.  feats bf16 or fp16 [B,P,D], masks uint8 [B,M,P] -> (out f32 [B*M, D] (first `total` rows valid),
    counts int32 [B], src int32 [B*M], total int32 [1]) — all device tensors, no host sync."""
    require_cuda(feats, "feats")
    require_cuda(masks, "masks")
    assert feats.dtype in (torch.bfloat16, torch.float16) and feats.is_contiguous() and feats.dim() == 3
    assert masks.dtype == torch.uint8 and masks.is_contiguous() and masks.dim() == 3
    B, P, D = feats.shape
    M = masks.shape[1]
    assert masks.shape == (B, M, P)
    dev = feats.device
    if out is None:         # `out`: the four result tensors of a previous call with the same shape, reused (steady-state serving)
        out = (torch.empty((B * M, D), dtype=torch.float32, device=dev), torch.empty((B,), dtype=torch.int32, device=dev),
               torch.empty((B * M,), dtype=torch.int32, device=dev), torch.empty((1,), dtype=torch.int32, device=dev))
    out, counts, src, total = out
    lib = _lib.load()
    nbytes = lib.rvo_mask_pool_workspace_bytes(B, M, P, D)
    ws = workspace(dev, nbytes, ws_key)
    check(lib.rvo_mask_pool(_ptr(feats), _feat_dtype(feats), _ptr(masks), B, M, P, D, int(max_regions), _ptr(out), _ptr(counts), _ptr(src),
                            _ptr(total), _ptr(ws), nbytes, _stream(dev)), "rvo_mask_pool")
    return out, counts, src, total


def mask_pool_to_db(feats: torch.Tensor, masks: torch.Tensor, db: torch.Tensor, row0: int, max_regions: int = 0,
                    want_f32: bool = False):
    """K1 fused with ingest: the kept regions' normalised embeddings go straight into the tiled bf16 DB at rows
    row0, row0+1, ... (compacted, (image, region) order).  Returns (counts int32 [B], src int32 [B*M], total int32 [1],
    f32 [B*M, D] | None) — device tensors, no host sync.  Shapes outside the tensor-core kernel take two CUDA calls
    (rvo_mask_pool + rvo_normalize_rows, one host sync) with the same result."""
    require_cuda(feats, "feats")
    require_cuda(masks, "masks")
    require_cuda(db, "db")
    assert feats.dtype in (torch.bfloat16, torch.float16) and feats.is_contiguous() and feats.dim() == 3
    assert masks.dtype == torch.uint8 and masks.is_contiguous() and masks.dim() == 3
    assert db.dtype == torch.bfloat16 and db.is_contiguous() and db.dim() == 4
    B, P, D = feats.shape
    M = masks.shape[1]
    assert masks.shape == (B, M, P) and db.shape[1] * TILE_COLS == d_pad_of(D)
    lim = M if max_regions <= 0 else min(M, max_regions)
    if row0 + B * lim > db_capacity(db):
        raise RvoError(f"mask_pool_to_db: DB capacity {db_capacity(db)} rows < row0 {row0} + {B * lim}")
    dev = feats.device
    counts = torch.empty((B,), dtype=torch.int32, device=dev)
    src = torch.empty((B * M,), dtype=torch.int32, device=dev)
    total = torch.empty((1,), dtype=torch.int32, device=dev)
    f32 = torch.empty((B * M, D), dtype=torch.float32, device=dev) if want_f32 else None
    lib = _lib.load()
    nbytes = lib.rvo_mask_pool_workspace_bytes(B, M, P, D)
    ws = workspace(dev, nbytes)
    rc = lib.rvo_mask_pool_to_db(_ptr(feats), _feat_dtype(feats), _ptr(masks), B, M, P, D, int(max_regions), _ptr(db), int(row0), _ptr(f32),
                                 _ptr(counts), _ptr(src), _ptr(total), _ptr(ws), nbytes, _stream(dev))
    if rc == _lib.RVO_E_UNSUPPORTED:
        out, counts, src, total = mask_pool(feats, masks, max_regions)
        t = int(total.item())          # this (rare-shape) route synchronises: only the kept rows may be written
        if t:
            normalize_rows(out[:t], db=db, row0=row0)
        return counts, src, total, (out if want_f32 else None)
    check(rc, "rvo_mask_pool_to_db")
    return counts, src, total, f32


def search_topk(db: torch.Tensor, n_rows: int, d: int, queries: torch.Tensor, k: int,
                score_threshold: float | None = None, id_offset: int = 0, out=None, path: int = 0, ws_key=None):
    """K2.  db: tiled bf16 DB storage (`db_alloc`) holding >= n_rows normalised rows, queries f32 [nq, d].
    Returns device tensors (ids int64 [nq,k], scores f32 [nq,k], counts int32 [nq]); async on the current stream.
    counts[q] == -1 marks an overflowed query (see `search_topk_exact`).  `path`: _lib.RVO_PATH_* (0 = by batch size)."""
    require_cuda(db, "db")
    if not (queries.is_cuda or queries.is_pinned()):
        raise RvoError("queries must be a CUDA tensor or a pinned host tensor: the B200 library has no CPU path")
    assert db.dtype == torch.bfloat16 and db.dim() == 4 and db.is_contiguous() and db.shape[2:] == (TILE_ROWS, TILE_COLS)
    assert queries.dtype == torch.float32 and queries.dim() == 2 and queries.is_contiguous()
    nq = queries.shape[0]
    assert queries.shape[1] == d and n_rows <= db_capacity(db) and db.shape[1] * TILE_COLS == d_pad_of(d)
    if not (1 <= k <= RVO_MAX_K):
        raise RvoError(f"k={k} outside 1..{RVO_MAX_K}")
    dev = db.device
    if out is None:
        ids = torch.empty((nq, k), dtype=torch.int64, device=dev)
        scores = torch.empty((nq, k), dtype=torch.float32, device=dev)
        counts = torch.empty((nq,), dtype=torch.int32, device=dev)
    else:
        ids, scores, counts = out
    lib = _lib.load()
    wkey = (n_rows, d, nq, k, path, _lib.option_epoch)
    nbytes = _ws_bytes.get(wkey)
    if nbytes is None:
        nbytes = lib.rvo_search_workspace_bytes_ex(n_rows, d, nq, k, path)
        if nbytes == 0:
            raise RvoError(f"rvo_search_workspace_bytes rejected n_rows={n_rows} d={d} nq={nq} k={k} path={path}: "
                           + lib.rvo_last_error().decode())
        if len(_ws_bytes) > 256:
            _ws_bytes.clear()
        _ws_bytes[wkey] = nbytes
    ws = workspace(dev, nbytes, ws_key)
    thr = -math.inf if score_threshold is None else float(score_threshold)
    check(lib.rvo_search_topk_ex(_ptr(db), n_rows, d, d_pad_of(d), _ptr(queries), nq, k, thr, int(id_offset), int(path), _ptr(ids),
                                 _ptr(scores), _ptr(counts), _ptr(ws), nbytes, _stream(dev)), "rvo_search_topk")
    return ids, scores, counts


class PreparedSearch:
    """`search_topk` with everything but the launch resolved once: argument checks, workspace size and buffer, output tensors and
    the ctypes argument tuple.  Calling it costs one ctypes call plus the current-stream lookup — what a serving loop that repeats
    the same shape (the UI's Q = 1, a batch job's Q = 256) pays per search instead of ~15 us of Python bookkeeping.  The tensors
    it was built from must stay alive and unchanged in address (it holds references)."""

    def __init__(self, db, n_rows, d, queries, k, score_threshold=None, id_offset=0, out=None, path=0, ws_key=None):
        require_cuda(db, "db")
        assert db.dtype == torch.bfloat16 and db.dim() == 4 and db.is_contiguous() and db.shape[2:] == (TILE_ROWS, TILE_COLS)
        assert queries.dtype == torch.float32 and queries.dim() == 2 and queries.is_contiguous()
        assert queries.is_cuda or queries.is_pinned()
        nq = queries.shape[0]
        assert queries.shape[1] == d and n_rows <= db_capacity(db) and db.shape[1] * TILE_COLS == d_pad_of(d)
        if not (1 <= k <= RVO_MAX_K):
            raise RvoError(f"k={k} outside 1..{RVO_MAX_K}")
        self.dev = db.device
        if out is None:
            out = (torch.empty((nq, k), dtype=torch.int64, device=self.dev), torch.empty((nq, k), dtype=torch.float32, device=self.dev),
                   torch.empty((nq,), dtype=torch.int32, device=self.dev))
        self.out = out
        self.lib = _lib.load()
        nbytes = self.lib.rvo_search_workspace_bytes_ex(n_rows, d, nq, k, path)
        if nbytes == 0:
            raise RvoError(f"rvo_search_workspace_bytes rejected n_rows={n_rows} d={d} nq={nq} k={k} path={path}: "
                           + self.lib.rvo_last_error().decode())
        self._keep = (db, queries, workspace(self.dev, nbytes, ws_key))
        thr = -math.inf if score_threshold is None else float(score_threshold)
        self.args = (_ptr(db), n_rows, d, d_pad_of(d), _ptr(queries), nq, k, thr, int(id_offset), int(path), _ptr(out[0]),
                     _ptr(out[1]), _ptr(out[2]), _ptr(self._keep[2]), nbytes)
        self.epoch = _lib.option_epoch
        self._fn = self.lib.rvo_search_topk_ex

    def __call__(self):
        rc = self._fn(*self.args, torch.cuda.current_stream(self.dev).cuda_stream)
        if rc:
            check(rc, "rvo_search_topk")
        return self.out


def search_topk_exact(db, n_rows, d, queries, k, score_threshold=None, id_offset=0):
    """`search_topk` plus the documented overflow protocol: queries flagged -1 by the fused path are re-run in batches of
    <= RVO_SMALL_Q through the exact fp32 scan, and — should its survivor lists overflow as well (adversarial row order) —
    through the dense fp32 route, which cannot overflow whatever the data.  Synchronises (reads counts)."""
    ids, scores, counts = search_topk(db, n_rows, d, queries, k, score_threshold, id_offset)
    bad = (counts < 0).nonzero().flatten().tolist()  # host sync; pathological inputs only take the branch
    small_ok = d_pad_of(d) <= 2048
    for path in ((_lib.RVO_PATH_SMALL, _lib.RVO_PATH_DENSE) if small_ok else ()):
        still = []
        for i in range(0, len(bad), RVO_SMALL_Q):
            sel = bad[i:i + RVO_SMALL_Q]
            sub = queries[sel].contiguous()
            a, b, c = search_topk(db, n_rows, d, sub, k, score_threshold, id_offset, path=path)
            cl = c.tolist()
            for j, q in enumerate(sel):
                if cl[j] < 0:
                    still.append(q)
                    continue
                ids[q].copy_(a[j])
                scores[q].copy_(b[j])
                counts[q] = c[j]
        bad = still
        if not bad:
            break
    return ids, scores, counts


def padded_queries(nq: int, d: int) -> int:
    r = _lib.load().rvo_padded_queries(nq, d)
    if r < 0:
        check(r, "rvo_padded_queries")
    return r


def scan_tile_rows(nq: int, d: int) -> int:
    r = _lib.load().rvo_scan_tile_rows(nq, d)
    if r < 0:
        check(r, "rvo_scan_tile_rows")
    return r


def scores_dense(db: torch.Tensor, n_rows: int, d: int, queries: torch.Tensor, tile_stride: int = 1) -> torch.Tensor:
    """Dense tensor-core score block (tests/diagnostics): [nq, cols] fp32, column c = t*T + i is DB row
    t*tile_stride*T + i with T = scan_tile_rows(nq, d); rows past n_rows hold -inf."""
    require_cuda(db, "db")
    nq = queries.shape[0]
    T = scan_tile_rows(nq, d)
    tiles = (n_rows + T - 1) // T
    cols = (tiles + tile_stride - 1) // tile_stride * T
    nq_pad = padded_queries(nq, d)
    out = torch.zeros((nq_pad, cols), dtype=torch.float32, device=db.device)
    nbytes = nq_pad * d_pad_of(d) * 2 + 4096
    ws = workspace(db.device, nbytes)
    lib = _lib.load()
    check(lib.rvo_scores_dense(_ptr(db), n_rows, d, d_pad_of(d), _ptr(queries), nq, tile_stride, _ptr(out),
                               out.stride(0), _ptr(ws), nbytes, _stream(db.device)), "rvo_scores_dense")
    return out[:nq]


def selfjoin_threshold(db: torch.Tensor, n_rows: int, d: int, threshold: float, row_lo: int = 0, row_hi: int | None = None,
                       out_cap: int = 1 << 22, id_offset: int = 0):
    """Near-duplicate self-join: pairs (i, j), row_lo <= i < row_hi, i < j, cos >= threshold.  Returns device tensors
    (pairs int64 [out_cap, 2], scores f32 [out_cap], count int64 [1], overflowed int32 [1]); async."""
    require_cuda(db, "db")
    assert db.dtype == torch.bfloat16 and db.dim() == 4 and db.is_contiguous()
    row_hi = n_rows if row_hi is None else row_hi
    dev = db.device
    pairs = torch.empty((out_cap, 2), dtype=torch.int64, device=dev)
    scores = torch.empty((out_cap,), dtype=torch.float32, device=dev)
    count = torch.zeros((1,), dtype=torch.int64, device=dev)
    over = torch.zeros((1,), dtype=torch.int32, device=dev)
    lib = _lib.load()
    nbytes = lib.rvo_selfjoin_workspace_bytes(d)
    ws = workspace(dev, nbytes)
    check(lib.rvo_selfjoin_threshold(_ptr(db), n_rows, d, d_pad_of(d), int(row_lo), int(row_hi), float(threshold),
                                     int(id_offset), _ptr(pairs), _ptr(scores), out_cap, _ptr(count), _ptr(over), _ptr(ws),
                                     nbytes, _stream(dev)), "rvo_selfjoin_threshold")
    return pairs, scores, count, over


def selfjoin_exact(db: torch.Tensor, n_rows: int, d: int, threshold: float, row_lo: int = 0, row_hi: int | None = None,
                   max_pairs: int = 1 << 22, id_offset: int = 0, cand_cap: int = 32768):
    """`selfjoin_threshold` that cannot lose pairs: when a query row's candidate sub-list overflows (more near-duplicates
    than `cand_cap` holds — a static video scene) the join is re-run with 8x the capacity (exact once
    cand_cap >= n_rows + 4096), and when more than `max_pairs` pairs exist the output buffers grow to the reported count.
    Returns host arrays (pairs int64 [m, 2], scores f32 [m]).  Synchronises."""
    require_cuda(db, "db")
    row_hi = n_rows if row_hi is None else row_hi
    dev = db.device
    lib = _lib.load()
    cap, out_cap = int(cand_cap), int(max_pairs)
    while True:
        pairs = torch.empty((out_cap, 2), dtype=torch.int64, device=dev)
        scores = torch.empty((out_cap,), dtype=torch.float32, device=dev)
        count = torch.zeros((1,), dtype=torch.int64, device=dev)
        over = torch.zeros((1,), dtype=torch.int32, device=dev)
        nbytes = lib.rvo_selfjoin_workspace_bytes_ex(d, cap)
        ws = workspace(dev, nbytes)
        check(lib.rvo_selfjoin_threshold_ex(_ptr(db), n_rows, d, d_pad_of(d), int(row_lo), int(row_hi), float(threshold),
                                            int(id_offset), cap, _ptr(pairs), _ptr(scores), out_cap, _ptr(count), _ptr(over),
                                            _ptr(ws), nbytes, _stream(dev)), "rvo_selfjoin_threshold_ex")
        m, ov = int(count.item()), int(over.item())
        if ov > 0 and cap < n_rows + 4096:
            cap = min(cap * 8, n_rows + 4096 + TILE_ROWS * 16)
            continue
        if m > out_cap:
            out_cap = m
            continue
        if ov > 0:
            raise RvoError(f"self-join candidate lists overflowed at capacity {cap} for {n_rows} rows")
        return pairs[:m].cpu().numpy(), scores[:m].cpu().numpy()


def join_out(out_cap: int, device) -> tuple:
    """Pair buffer of `join_threshold`: (pairs int64 [out_cap, 2], scores f32 [out_cap], count int64 [1] = 0,
    overflowed int32 [1] = 0)."""
    return (torch.empty((out_cap, 2), dtype=torch.int64, device=device), torch.empty((out_cap,), dtype=torch.float32, device=device),
            torch.zeros((1,), dtype=torch.int64, device=device), torch.zeros((1,), dtype=torch.int32, device=device))


def join_threshold(qdb: torch.Tensor, q_row_lo: int, q_row_hi: int, q_id_offset: int, db: torch.Tensor, n_rows: int, d: int,
                   threshold: float, id_offset: int, cand_cap: int, out: tuple) -> None:
    """rvo_join_threshold: query rows [q_row_lo, q_row_hi) of the tiled storage `qdb` against the first n_rows rows of the tiled
    storage `db`, pairs with cos >= threshold as (lower id, higher id), ids = row + offset.  `qdb is db` with equal offsets is the
    triangle of the self-join (i < j only); otherwise the two row sets must be disjoint and every pair counts.  `out` (`join_out`,
    on db's device) is APPENDED to: its count and overflow counter are never reset.  Async on the current stream of db's device."""
    require_cuda(db, "db")
    require_cuda(qdb, "qdb")
    for t in (qdb, db):
        assert t.dtype == torch.bfloat16 and t.dim() == 4 and t.is_contiguous() and t.shape[1] * TILE_COLS == d_pad_of(d)
    assert n_rows <= db_capacity(db) and q_row_hi <= db_capacity(qdb)
    pairs, scores, count, over = out
    dev = db.device
    lib = _lib.load()
    nbytes = lib.rvo_join_workspace_bytes(d, int(cand_cap))
    ws = workspace(dev, nbytes)
    check(lib.rvo_join_threshold(_ptr(qdb), int(q_row_lo), int(q_row_hi), int(q_id_offset), _ptr(db), int(n_rows), d, d_pad_of(d),
                                 float(threshold), int(id_offset), int(cand_cap), _ptr(pairs), _ptr(scores), pairs.shape[0],
                                 _ptr(count), _ptr(over), _ptr(ws), nbytes, _stream(dev)), "rvo_join_threshold")


def cross_join_threshold(qdb: torch.Tensor, q_row_lo: int, q_row_hi: int, q_id_offset: int, db: torch.Tensor, n_rows: int, d: int,
                         threshold: float, id_offset: int, query_is_right: bool, cand_cap: int, out: tuple) -> None:
    """rvo_cross_join_threshold: query rows [q_row_lo, q_row_hi) of the tiled storage `qdb` against the first n_rows rows of the
    tiled storage `db`, where the two belong to different collections: every pair with cos >= threshold, stored as (left id,
    right id) with ids = row + offset; `query_is_right` says which collection the query rows are.  The ids may overlap and
    `qdb is db` is allowed (the full ordered join, self pairs included).  `out` (`join_out`, on db's device) is APPENDED to, as in
    `join_threshold`.  Async on the current stream of db's device."""
    require_cuda(db, "db")
    require_cuda(qdb, "qdb")
    for t in (qdb, db):
        assert t.dtype == torch.bfloat16 and t.dim() == 4 and t.is_contiguous() and t.shape[1] * TILE_COLS == d_pad_of(d)
    assert n_rows <= db_capacity(db) and q_row_hi <= db_capacity(qdb)
    pairs, scores, count, over = out
    dev = db.device
    lib = _lib.load()
    nbytes = lib.rvo_join_workspace_bytes(d, int(cand_cap))
    ws = workspace(dev, nbytes)
    check(lib.rvo_cross_join_threshold(_ptr(qdb), int(q_row_lo), int(q_row_hi), int(q_id_offset), _ptr(db), int(n_rows), d,
                                       d_pad_of(d), float(threshold), int(id_offset), int(bool(query_is_right)), int(cand_cap),
                                       _ptr(pairs), _ptr(scores), pairs.shape[0], _ptr(count), _ptr(over), _ptr(ws), nbytes,
                                       _stream(dev)), "rvo_cross_join_threshold")


def components_out(n_labels: int, device) -> tuple:
    """Union-find forest of `join_components`: (parent int32 [n_labels] = arange, hit count int64 [1] = 0, overflowed int32 [1]
    = 0).  Refuses 2^31 rows or more (the forest holds int32 rows)."""
    if not 0 < n_labels < (1 << 31):
        raise RvoError(f"duplicate groups need 1 to 2^31 - 1 rows, got {n_labels}")
    return (torch.arange(n_labels, dtype=torch.int32, device=device), torch.zeros((1,), dtype=torch.int64, device=device),
            torch.zeros((1,), dtype=torch.int32, device=device))


def join_components(qdb: torch.Tensor, q_row_lo: int, q_row_hi: int, q_id_offset: int, db: torch.Tensor, n_rows: int, d: int,
                    threshold: float, id_offset: int, cand_cap: int, out: tuple) -> None:
    """rvo_join_components: `join_threshold`'s join (same arguments, same pairs examined), but every pair with cos >= threshold
    unions its two ids in the forest of `out` (`components_out`, on db's device, indexed by id) instead of being stored.  The
    hit count and overflow counter are APPENDED to.  Async on the current stream of db's device."""
    require_cuda(db, "db")
    require_cuda(qdb, "qdb")
    for t in (qdb, db):
        assert t.dtype == torch.bfloat16 and t.dim() == 4 and t.is_contiguous() and t.shape[1] * TILE_COLS == d_pad_of(d)
    assert n_rows <= db_capacity(db) and q_row_hi <= db_capacity(qdb)
    parent, hits, over = out
    assert parent.dtype == torch.int32 and parent.is_contiguous() and parent.device == db.device
    dev = db.device
    lib = _lib.load()
    nbytes = lib.rvo_join_workspace_bytes(d, int(cand_cap))
    ws = workspace(dev, nbytes)
    check(lib.rvo_join_components(_ptr(qdb), int(q_row_lo), int(q_row_hi), int(q_id_offset), _ptr(db), int(n_rows), d,
                                  d_pad_of(d), float(threshold), int(id_offset), int(cand_cap), _ptr(parent), parent.numel(),
                                  _ptr(hits), _ptr(over), _ptr(ws), nbytes, _stream(dev)), "rvo_join_components")


def components_flatten(parent: torch.Tensor) -> torch.Tensor:
    """rvo_components_flatten: int32 labels [n], label[x] = the smallest row of x's component.  Async."""
    require_cuda(parent, "parent")
    assert parent.dtype == torch.int32 and parent.is_contiguous()
    labels = torch.empty_like(parent)
    check(_lib.load().rvo_components_flatten(_ptr(parent), parent.numel(), _ptr(labels), _stream(parent.device)),
          "rvo_components_flatten")
    return labels


def components_merge(parent: torch.Tensor, labels_src: torch.Tensor) -> None:
    """rvo_components_merge: fold the flattened labels of another forest over the same rows (on parent's device) into
    `parent`.  Async."""
    require_cuda(parent, "parent")
    assert parent.dtype == labels_src.dtype == torch.int32 and parent.is_contiguous() and labels_src.is_contiguous()
    assert labels_src.shape == parent.shape and labels_src.device == parent.device
    check(_lib.load().rvo_components_merge(_ptr(parent), _ptr(labels_src), parent.numel(), _stream(parent.device)),
          "rvo_components_merge")


def components_exact(db: torch.Tensor, n_rows: int, d: int, threshold: float, id_offset: int = 0, cand_cap: int = 32768):
    """Single-linkage groups at a threshold: the connected components of the graph whose edges are exactly the pairs
    `selfjoin_exact` returns, unioned on the device while the join runs (no pair is stored: O(n_rows) memory).  Returns
    (labels int64 [n_rows] host array, n_pairs): labels[i] is the smallest id (row + id_offset) of row i's component, and
    n_pairs the number of pairs with cos >= threshold.  Overflow protocol of `selfjoin_exact`: overflowed candidate lists re-run
    the join with 8x the capacity (exact once cand_cap >= n_rows + 4096), keeping the forest (re-applying an edge changes
    nothing) and resetting the hit count.  Synchronises."""
    require_cuda(db, "db")
    assert db.dtype == torch.bfloat16 and db.dim() == 4 and db.is_contiguous()
    parent, hits, over = components_out(n_rows, db.device)
    cap = int(cand_cap)
    while True:
        hits.zero_()
        over.zero_()
        join_components(db, 0, n_rows, 0, db, n_rows, d, threshold, 0, cap, (parent, hits, over))
        m, ov = int(hits.item()), int(over.item())
        if ov > 0 and cap < n_rows + 4096:
            cap = min(cap * 8, n_rows + 4096 + TILE_ROWS * 16)
            continue
        if ov > 0:
            raise RvoError(f"self-join candidate lists overflowed at capacity {cap} for {n_rows} rows")
        labels = components_flatten(parent).cpu().numpy().astype("int64")
        return labels + int(id_offset), m


def knn_join(qdb: torch.Tensor, q_row_lo: int, q_row_hi: int, q_id_offset: int, db: torch.Tensor, n_rows: int, d: int, k: int,
             score_threshold: float | None, id_offset: int, exclude_self: bool, q_rows: torch.Tensor | None = None, path: int = 0,
             out=None):
    """rvo_knn_join: for each query row of the tiled storage `qdb` — rows [q_row_lo, q_row_hi), or q_rows[q_row_lo:q_row_hi]
    when a device int64 list is given — the k rows of the first n_rows rows of `db` with the highest fp32 dot of the two stored
    rows.  `exclude_self` (qdb and db one collection, ids row + offset): a row's own id is left out of its list.  Returns device
    tensors (ids int64 [nq, k], scores f32 [nq, k], counts int32 [nq]) as `search_topk` does; counts[q] == -1 marks a query that
    overflowed the fused path (`knn_exact`).  Async on the current stream of db's device."""
    require_cuda(qdb, "qdb")
    require_cuda(db, "db")
    for t in (qdb, db):
        assert t.dtype == torch.bfloat16 and t.dim() == 4 and t.is_contiguous() and t.shape[1] * TILE_COLS == d_pad_of(d)
    assert n_rows <= db_capacity(db) and qdb.device == db.device
    if q_rows is None:
        assert q_row_hi <= db_capacity(qdb)
    else:
        assert q_rows.dtype == torch.int64 and q_rows.is_contiguous() and q_rows.device == db.device and q_row_hi <= q_rows.numel()
    k_max = RVO_MAX_K - 1 if exclude_self else RVO_MAX_K
    if not 1 <= k <= k_max:
        raise RvoError(f"k={k} outside 1..{k_max}" + (" (a row's own match is left out)" if exclude_self else ""))
    nq = int(q_row_hi) - int(q_row_lo)
    dev = db.device
    if out is None:
        out = (torch.empty((nq, k), dtype=torch.int64, device=dev), torch.empty((nq, k), dtype=torch.float32, device=dev),
               torch.empty((nq,), dtype=torch.int32, device=dev))
    ids, scores, counts = out
    if nq == 0:
        return ids, scores, counts
    lib = _lib.load()
    nbytes = lib.rvo_knn_workspace_bytes(int(n_rows), d, nq, k, int(path))
    if nbytes == 0:
        raise RvoError(f"rvo_knn_workspace_bytes rejected n_rows={n_rows} d={d} nq={nq} k={k} path={path}")
    ws = workspace(dev, nbytes, "knn")
    thr = -math.inf if score_threshold is None else float(score_threshold)
    check(lib.rvo_knn_join(_ptr(qdb), int(q_row_lo), int(q_row_hi), _ptr(q_rows), int(q_id_offset), _ptr(db), int(n_rows), d,
                           d_pad_of(d), int(k), thr, int(id_offset), int(bool(exclude_self)), int(path), _ptr(ids), _ptr(scores),
                           _ptr(counts), _ptr(ws), nbytes, _stream(dev)), "rvo_knn_join")
    return ids, scores, counts


def knn_exact(qdb: torch.Tensor, q_row_lo: int, q_row_hi: int, q_id_offset: int, db: torch.Tensor, n_rows: int, d: int, k: int,
              score_threshold: float | None, id_offset: int, exclude_self: bool, q_rows: torch.Tensor | None = None):
    """`knn_join` plus the overflow protocol of `search_topk_exact`: rows the fused path flags -1 are re-run, as a q_rows list, in
    batches of <= RVO_SMALL_Q through the exact fp32 scan, and what that route flags as well through the dense fp32 route, which
    cannot overflow.  Scores stay the raw dot of the stored rows on every route.  Rows wider than 2048 (d_pad) have no fp32
    route, as in `search_topk_exact`: a flagged row stays -1 there (the public layer raises).  Synchronises (reads counts)."""
    ids, scores, counts = knn_join(qdb, q_row_lo, q_row_hi, q_id_offset, db, n_rows, d, k, score_threshold, id_offset, exclude_self,
                                   q_rows)
    bad = (counts < 0).nonzero().flatten()                      # host sync; pathological inputs only take the branch
    if bad.numel() == 0 or d_pad_of(d) > 2048:
        return ids, scores, counts
    rows = bad + int(q_row_lo) if q_rows is None else q_rows[int(q_row_lo):int(q_row_hi)][bad]
    a, b, c = knn_fp32(qdb, rows, q_id_offset, db, n_rows, d, k, score_threshold, id_offset, exclude_self)
    ids[bad], scores[bad], counts[bad] = a, b, c
    return ids, scores, counts


def knn_fp32(qdb: torch.Tensor, q_rows: torch.Tensor, q_id_offset: int, db: torch.Tensor, n_rows: int, d: int, k: int,
             score_threshold: float | None, id_offset: int, exclude_self: bool):
    """The exact routes of `knn_exact` for the query rows listed in q_rows (device int64): batches of <= RVO_SMALL_Q through the
    fp32 scan, then what that route flags through the dense fp32 route, which cannot overflow.  Every pair is scored by the
    same fp32 arithmetic on both routes, whichever rows the target holds.  Needs d_pad <= 2048.  Returns device tensors as
    `knn_join`; synchronises."""
    nq = q_rows.numel()
    dev = db.device
    ids = torch.empty((nq, k), dtype=torch.int64, device=dev)
    scores = torch.empty((nq, k), dtype=torch.float32, device=dev)
    counts = torch.full((nq,), -1, dtype=torch.int32, device=dev)
    todo = list(range(nq))
    for path in (_lib.RVO_PATH_SMALL, _lib.RVO_PATH_DENSE):
        for i in range(0, len(todo), RVO_SMALL_Q):
            sel = torch.tensor(todo[i:i + RVO_SMALL_Q], device=dev)
            a, b, c = knn_join(qdb, 0, sel.numel(), q_id_offset, db, n_rows, d, k, score_threshold, id_offset, exclude_self,
                               q_rows[sel], path)
            ids[sel], scores[sel], counts[sel] = a, b, c
        todo = (counts < 0).nonzero().flatten().tolist()
        if not todo:
            break
    return ids, scores, counts


def knn_exclude_self(ids: torch.Tensor, scores: torch.Tensor, counts: torch.Tensor, q_row_lo: int, q_id_offset: int,
                     q_rows: torch.Tensor | None = None):
    """rvo_knn_exclude_self: lists of k + 1 (ids [nq, k+1], scores, counts [nq]) -> lists of k without each query's own id,
    q_id_offset + (q_rows[q] if a list is given else q_row_lo + q).  Async."""
    require_cuda(ids, "ids")
    nq, k1 = ids.shape
    assert ids.is_contiguous() and scores.is_contiguous() and counts.is_contiguous() and scores.shape == ids.shape
    if q_rows is not None:
        assert q_rows.dtype == torch.int64 and q_rows.is_contiguous() and q_rows.numel() >= nq and q_rows.device == ids.device
    dev = ids.device
    oi = torch.empty((nq, k1 - 1), dtype=torch.int64, device=dev)
    os_ = torch.empty((nq, k1 - 1), dtype=torch.float32, device=dev)
    oc = torch.empty((nq,), dtype=torch.int32, device=dev)
    check(_lib.load().rvo_knn_exclude_self(_ptr(ids), _ptr(scores), _ptr(counts), nq, k1 - 1, int(q_row_lo), _ptr(q_rows),
                                           int(q_id_offset), _ptr(oi), _ptr(os_), _ptr(oc), _stream(dev)), "rvo_knn_exclude_self")
    return oi, os_, oc


def merge_topk(ids: torch.Tensor, scores: torch.Tensor, counts: torch.Tensor, k: int):
    """K3.  ids int64 [G,nq,k], scores f32 [G,nq,k], counts int32 [G,nq] -> merged (ids, scores, counts)."""
    require_cuda(ids, "ids")
    G, nq, kk = ids.shape
    assert kk == k and ids.is_contiguous() and scores.is_contiguous() and counts.is_contiguous()
    dev = ids.device
    oi = torch.empty((nq, k), dtype=torch.int64, device=dev)
    os_ = torch.empty((nq, k), dtype=torch.float32, device=dev)
    oc = torch.empty((nq,), dtype=torch.int32, device=dev)
    check(_lib.load().rvo_merge_topk(_ptr(ids), _ptr(scores), _ptr(counts), G, nq, k, _ptr(oi), _ptr(os_), _ptr(oc),
                                     _stream(dev)), "rvo_merge_topk")
    return oi, os_, oc


def kmeans_update(db: torch.Tensor, row_lo: int, row_hi: int, d: int, ids: torch.Tensor, n_clusters: int, prev: torch.Tensor | None,
                  labels: torch.Tensor, sums: torch.Tensor, counts: torch.Tensor, changed: torch.Tensor, id_offset: int = 0) -> None:
    """rvo_kmeans_update: the update step of spherical k-means for rows [row_lo, row_hi) of the tiled storage `db`, assigned by
    `ids` (int64 [n] or [n, 1], the k = 1 lists of `knn_join` against the centroids; cluster = id - id_offset).  Writes int32
    `labels` [n] and ADDS to `sums` (int64 [n_clusters, d]: each member's bf16 components as rint(x * 2^31), exact and
    order-independent), `counts` (int64 [n_clusters]) and `changed` (int64 [1]: labels differing from `prev`, all n when prev is
    None).  Async on the current stream of db's device."""
    require_cuda(db, "db")
    assert db.dtype == torch.bfloat16 and db.dim() == 4 and db.is_contiguous() and db.shape[1] * TILE_COLS == d_pad_of(d)
    n = int(row_hi) - int(row_lo)
    assert row_hi <= db_capacity(db) and ids.dtype == torch.int64 and ids.is_contiguous() and ids.numel() == n
    assert labels.dtype == torch.int32 and labels.is_contiguous() and labels.numel() == n
    assert prev is None or (prev.dtype == torch.int32 and prev.is_contiguous() and prev.numel() == n)
    assert sums.dtype == counts.dtype == changed.dtype == torch.int64 and sums.shape == (n_clusters, d) and sums.is_contiguous()
    assert counts.shape == (n_clusters,) and changed.numel() >= 1
    dev = db.device
    lib = _lib.load()
    nbytes = lib.rvo_kmeans_update_workspace_bytes(n, int(n_clusters))
    if nbytes == 0:
        raise RvoError(f"k-means update of {n} rows into {n_clusters} clusters: needs fewer than 2^31 rows and 1 to "
                       f"{_lib.RVO_KMEANS_MAX_CLUSTERS} clusters")
    ws = workspace(dev, nbytes, "kmeans")
    check(lib.rvo_kmeans_update(_ptr(db), int(row_lo), int(row_hi), d, d_pad_of(d), _ptr(ids), int(id_offset), int(n_clusters),
                                _ptr(prev), _ptr(labels), _ptr(sums), _ptr(counts), _ptr(changed), _ptr(ws), nbytes, _stream(dev)),
          "rvo_kmeans_update")


def kmeans_finalize(sums: torch.Tensor, counts: torch.Tensor, d: int, centroids: torch.Tensor, empty: torch.Tensor,
                    n_empty: torch.Tensor) -> None:
    """rvo_kmeans_finalize: new centroids from the (reduced) integer sums, normalised and rounded into rows [0, C) of the tiled
    storage `centroids` as `normalize_rows` does; `empty` (int32 [C]) flags the clusters with no member or an all-zero sum, and
    their number is ADDED to `n_empty` (int64 [1]).  Async on the current stream of the sums' device."""
    require_cuda(sums, "sums")
    C = sums.shape[0]
    assert sums.dtype == counts.dtype == n_empty.dtype == torch.int64 and sums.shape == (C, d) and counts.shape == (C,)
    assert centroids.dtype == torch.bfloat16 and centroids.is_contiguous() and C <= db_capacity(centroids)
    assert centroids.shape[1] * TILE_COLS == d_pad_of(d) and empty.dtype == torch.int32 and empty.numel() == C
    for t in (counts, centroids, empty, n_empty):
        assert t.device == sums.device
    scratch = workspace(sums.device, C * d * 4, "kmeans_f32")
    check(_lib.load().rvo_kmeans_finalize(_ptr(sums), _ptr(counts), C, d, _ptr(scratch), _ptr(centroids), _ptr(empty), _ptr(n_empty),
                                          _stream(sums.device)), "rvo_kmeans_finalize")


def kmeans_exact(db: torch.Tensor, n_rows: int, d: int, centroids: torch.Tensor, n_clusters: int, max_iter: int = 50,
                 id_offset: int = 0):
    """Spherical k-means of the first n_rows rows of the tiled storage `db`, started from rows [0, n_clusters) of the tiled
    centroid storage `centroids` (on db's device; it is not modified).  The loop of `sharded.kmeans_sharded` on one shard:
    assignment `knn_exact(db, 0, n, id_offset, centroids, C, d, 1, None, 0, False)`, integer update, re-seeding of empty
    clusters, until an assignment equals the previous one or max_iter updates have run.  Returns `sharded.KMeansResult`."""
    from .sharded import kmeans_sharded
    return kmeans_sharded([(db, int(n_rows), int(id_offset))], d, centroids, n_clusters, max_iter)
