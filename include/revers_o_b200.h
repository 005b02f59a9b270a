/*
 * revers_o_b200.h — C ABI of the B200-native region-similarity hot path of kolenyo2099/revers-o.
 *
 * This is the drop-in boundary (DESIGN.md §2, SURVEY.md §8b).  The reference has no FFI of its own
 * (it is pure Python); every entry point below names the reference call site whose arithmetic it
 * replaces.  A reference-side maintainer binds these with ctypes (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary;
 *   - every pointer marked [dev] is a device pointer of ONE GPU; the library derives the device
 *     from the first device pointer of the call, makes it current, and borrows the pointers only
 *     for the duration of the call (it never frees or retains them);
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); all work is
 *     enqueued on it and the call returns without synchronising unless stated;
 *   - return value: 0 = ok, negative = error (see RVO_E_*); `rvo_last_error()` gives the text of the
 *     last error on the calling thread.  Python maps errors to the reference's status-string
 *     convention (core_system.py:93-119,652-666); nothing raises into Gradio.
 *   - there is NO CPU fallback: without a Blackwell (sm_100) device every compute entry fails.
 */
#ifndef REVERS_O_B200_H
#define REVERS_O_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RVO_OK               0
#define RVO_E_INVALID      (-1)  /* bad argument (null pointer, unsupported size, misalignment)      */
#define RVO_E_CUDA         (-2)  /* a CUDA runtime/driver call failed                                */
#define RVO_E_NO_DEVICE    (-3)  /* no sm_100 device / driver entry point missing                    */
#define RVO_E_WORKSPACE    (-4)  /* workspace too small (call rvo_*_workspace_bytes)                 */
#define RVO_E_UNSUPPORTED  (-5)  /* shape not covered by this fused entry point: use the two-call form */

/* Limits of the fused search path. */
#define RVO_MAX_K          512   /* largest `limit` served by rvo_search_topk                        */
#define RVO_SMALL_Q        4     /* batches of <= RVO_SMALL_Q queries take the exact fp32 scan       */

/* 16-bit feature types accepted by K1. */
#define RVO_DTYPE_BF16     0
#define RVO_DTYPE_F16      1

/* Library / ABI version (major*10000 + minor*100 + patch). */
int rvo_version(void);

/* Text of the last error raised on this thread ("" if none). */
const char* rvo_last_error(void);

/* Number of SMs of the device that owns `dev_ptr` (148 on B200); <0 on error. */
int rvo_device_sm_count(const void* dev_ptr);

/* ------------------------------------------------------------------------------------------------
 * DB storage layout ("tiled"): bf16, rows padded to a multiple of 128, columns to d_pad = d rounded up
 * to 64 (pad columns/rows are zero):
 *        db[row / 128][col / 64][row % 128][col % 64]
 * i.e. every (128-row block, 64-column chunk) tile is one contiguous 16 KiB block, which is exactly one
 * TMA box of the scan kernel: the scan streams HBM in long contiguous bursts.  Bytes needed for n rows:
 * rvo_db_bytes(n, d).  Element offset: ((row/128)*(d_pad/64) + col/64)*8192 + (row%128)*64 + col%64.
 * ---------------------------------------------------------------------------------------------- */
size_t rvo_db_bytes(int64_t n_rows, int32_t d);

/* ------------------------------------------------------------------------------------------------
 * Ingest: L2-normalise float32 rows and store them as bf16.
 * Replaces: qdrant-local upsert into a COSINE collection (vector normalised, appended to the
 *           collection matrix) behind core_system.py:608-621, and the `e / e.norm()` of
 *           core_system.py:407,447 when called with dst_f32.
 *   src      [dev] float32 [n, d], row pitch src_ld elements
 *   dst_bf16 [dev] may be NULL.
 *            tiled_row0 >= 0: base of a tiled DB (see above) with d_pad == dst_ld; the n rows are
 *                             written at DB rows tiled_row0 .. tiled_row0 + n - 1 (append / overwrite);
 *            tiled_row0 <  0: plain row-major [n, dst_ld] (dst_ld % 8 == 0, >= d), pad columns zeroed.
 *   dst_f32  [dev] float32 [n, d] row pitch d: the normalised rows in float32.  May be NULL.
 * (K1 applies the same rule to a region whose mean is zero or non-finite: its embedding is the zero vector.)
 * A zero row stays zero (qdrant divides by eps; the reference never stores one, see
 * core_system.py:402-404).  A row with a NaN / Inf component is stored as the zero vector too (the reference
 * would store NaNs, which then score NaN against every query and sort to the top of every result).
 * ---------------------------------------------------------------------------------------------- */
int rvo_normalize_rows(const float* src, int64_t n, int32_t d, int64_t src_ld,
                       uint16_t* dst_bf16, int64_t dst_ld, int64_t tiled_row0, float* dst_f32, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K1 — segmented mask pooling + L2 normalise.
 * Replaces: the per-region python loop of core_system.py:363-408 (binarise :398-400, skip empty
 *           :402-404, region embedding + normalise :406-408) with the mask-pooled definition the
 *           reference states (main.py:8-9): e_m = mean of patch features under mask m, then L2.
 *   feats   [dev] 16-bit float [B, P, D]  patch-feature map, D contiguous (D % 8 == 0)
 *   feat_dtype          RVO_DTYPE_BF16 or RVO_DTYPE_F16 (what the reference's `.half()` encoder emits on CUDA,
 *                       core_system.py:195-196): consumed as is, products accumulate in fp32
 *   masks   [dev] uint8 [B, M, P]   nonzero = patch p belongs to region m
 *   max_regions          only the first min(M, max_regions) regions of an image are visited
 *                        (core_system.py:363 uses 50); <=0 means M
 *   out     [dev] float32 [B*M, D]  compacted: rows of non-empty regions in (image, region) order
 *   out_counts [dev] int32 [B]      regions kept per image (M' of core_system.py:402-404)
 *   out_src [dev] int32 [B*M]       for each output row, b*M + m of its source region (may be NULL)
 *   out_total [dev] int32 [1]       number of output rows (sum of out_counts)
 *   workspace [dev]                 rvo_mask_pool_workspace_bytes(B, M, P, D) bytes, 256-B aligned
 * ---------------------------------------------------------------------------------------------- */
size_t rvo_mask_pool_workspace_bytes(int32_t B, int32_t M, int32_t P, int32_t D);
int rvo_mask_pool(const uint16_t* feats, int32_t feat_dtype, const uint8_t* masks, int32_t B, int32_t M, int32_t P, int32_t D,
                  int32_t max_regions, float* out, int32_t* out_counts, int32_t* out_src, int32_t* out_total,
                  void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K1 fused with ingest — mask-pooled region embeddings written straight into the tiled bf16 DB.
 * Replaces: the whole ingest tail of create_database for a batch of images — the per-region loop of
 *           core_system.py:363-408 PLUS the list-of-floats PointStruct + upsert of :596-622 (qdrant COSINE
 *           upsert = normalise + append) — without the fp32 embeddings ever reaching HBM.
 *   feats / masks / max_regions / out_counts / out_src / out_total / workspace: as rvo_mask_pool
 *   db        [dev] bf16 tiled DB storage (see "DB storage layout"), d_pad = D rounded up to 64; the kept
 *             regions land, compacted in (image, region) order, at DB rows db_row0, db_row0 + 1, ...;
 *             capacity needed: db_row0 + B * min(M, max_regions) rows
 *   out_f32   [dev] float32 [B*M, D] optional copy of the embeddings (as rvo_mask_pool's `out`); may be NULL
 * Returns RVO_E_UNSUPPORTED for shapes outside the tensor-core kernel (D % 128 != 0, D > 4096, more than 64 regions
 * per image, more than 1024 patches): call rvo_mask_pool + rvo_normalize_rows instead.  When all D/128 channel slabs of an
 * image's regions do not fit the 512 TMEM columns together (PE-Core-G14: D = 1280 with more than 48 regions) the regions are
 * processed in groups inside the same single launch.  The launch is COOPERATIVE (its compaction offsets need a grid-wide
 * rendezvous): concurrent calls on different streams serialise instead of deadlocking.
 * ---------------------------------------------------------------------------------------------- */
int rvo_mask_pool_to_db(const uint16_t* feats, int32_t feat_dtype, const uint8_t* masks, int32_t B, int32_t M, int32_t P, int32_t D,
                        int32_t max_regions, uint16_t* db, int64_t db_row0, float* out_f32, int32_t* out_counts,
                        int32_t* out_src, int32_t* out_total, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K2 — exact cosine top-k over one DB shard.
 * Replaces: `QdrantClient.search(collection_name, query_vector, limit, score_threshold)` in local
 *           mode behind core_system.py:659-664 (normalise query, scores = vectors @ q over the
 *           whole collection, descending argsort, stop at first score < score_threshold, first
 *           `limit` hits), batched over nq queries row by row.
 *   db      [dev] bf16 tiled DB storage (see "DB storage layout") of L2-normalised rows; d_pad = d
 *           rounded up to 64
 *   queries [dev] float32 [nq, d] row pitch d; NOT required to be normalised.  `queries` and the three out_*
 *           arrays may also be PINNED HOST memory (unified addressing): the first kernel then reads the queries and
 *           the last one writes the results over PCIe, with no copy launches around the call.
 *   k       1..RVO_MAX_K  (`limit`)
 *   score_threshold   hits with score < threshold are dropped; pass -INFINITY for "None"
 *   id_offset         added to local row numbers (row-sharded DB: first global row of the shard)
 *   out_ids    [dev] int64   [nq, k]  global row ids, score-descending, ties by lower id; -1 pad
 *   out_scores [dev] float32 [nq, k]  fp32 cosine (fp32 query x bf16 row, fp32 accumulate); -inf pad
 *   out_counts [dev] int32   [nq]     hits per query (0..k), or -1 if the query OVERFLOWED the
 *                                     candidate buffers of the fused path (pathological tie mass);
 *                                     the caller must re-run such queries in batches of
 *                                     <= RVO_SMALL_Q (fp32 scan) and, should one of those report -1 as well,
 *                                     with rvo_search_topk_ex(path = RVO_PATH_DENSE), which cannot overflow.
 *   workspace  [dev] rvo_search_workspace_bytes(...) bytes, 1024-B aligned.  Contents are scratch.
 * nq <= RVO_SMALL_Q (and d <= 2048): exact fp32 CUDA-core scan (HBM-bound).  nq > RVO_SMALL_Q: bf16 tcgen05 scan
 * with the threshold-select fused in its epilogue, candidates re-scored in fp32.
 * ---------------------------------------------------------------------------------------------- */
size_t rvo_search_workspace_bytes(int64_t n_rows, int32_t d, int32_t nq, int32_t k);
int rvo_search_topk(const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad,
                    const float* queries, int32_t nq, int32_t k, float score_threshold, int64_t id_offset,
                    int64_t* out_ids, float* out_scores, int32_t* out_counts,
                    void* workspace, size_t workspace_bytes, void* stream);

/* The same search with the kernel path chosen by the caller instead of by nq:
 *   RVO_PATH_AUTO    nq <= RVO_SMALL_Q -> fp32 scan, else tcgen05 (what rvo_search_topk does)
 *   RVO_PATH_SMALL   fp32 CUDA-core scan (nq <= RVO_SMALL_Q).  Shards up to 131072 rows: [scan + every score] -> [exact top-k],
 *                    two launches, the reference's own operating point (Q = 1, core_system.py:657).  Larger shards: a row
 *                    sample's k-th best key filters the full scan, so scores never reach HBM; a survivor list that overflows
 *                    (adversarial row order) flags the query with count -1
 *   RVO_PATH_TENSOR  tcgen05 scan + fused select + fp32 re-score, any nq
 *   RVO_PATH_DENSE   fp32 scan keeping every score of the shard (nq <= RVO_SMALL_Q): cannot overflow, whatever the data — the
 *                    last resort of the overflow protocol (workspace: 4 bytes per row per query) */
#define RVO_PATH_AUTO   0
#define RVO_PATH_SMALL  1
#define RVO_PATH_TENSOR 2
#define RVO_PATH_DENSE  3
size_t rvo_search_workspace_bytes_ex(int64_t n_rows, int32_t d, int32_t nq, int32_t k, int32_t path);
int rvo_search_topk_ex(const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad,
                       const float* queries, int32_t nq, int32_t k, float score_threshold, int64_t id_offset, int32_t path,
                       int64_t* out_ids, float* out_scores, int32_t* out_counts,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Rows the tcgen05 path pads a batch of nq queries to (query blocks of <=256, multiples of 16). */
int rvo_padded_queries(int32_t nq, int32_t d);

/* DB rows per scan tile (128 or 256) for a batch of nq queries of dimension d. */
int rvo_scan_tile_rows(int32_t nq, int32_t d);

/* Dense score block (diagnostics / tests; this is the threshold-seeding pass of the fused path):
 * scores[q, c] = <bf16(q_hat), db[r]> computed by the tcgen05 scan in DENSE mode over every
 * tile_stride-th tile of T = rvo_scan_tile_rows(nq, d) rows: column c = t*T + i is row
 * r = t*tile_stride*T + i.  Rows past n_rows are written as -inf.
 *   out [dev] float32 [rvo_padded_queries(nq, d), out_ld], out_ld >= ceil(ceil(n_rows/T)/tile_stride)*T */
int rvo_scores_dense(const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad,
                     const float* queries, int32_t nq, int64_t tile_stride,
                     float* out, int64_t out_ld, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K3 — merge per-shard top-k lists (after one all-gather of [nq,k] ids/scores/counts per rank).
 * No reference counterpart (the reference is single-process); semantics = K2 over the union.
 *   ids [dev] int64 [G, nq, k], scores [dev] float32 [G, nq, k], counts [dev] int32 [G, nq]
 *   (a count of -1 marks an overflowed shard list and propagates to out_counts)
 *   every list must be ordered as rvo_search_topk emits it (score descending, ties by lower id) and global ids
 *   must be unique across lists: the merge ranks each element by binary searches in the other lists.
 *   out_* as in rvo_search_topk.   G <= 64, G*k <= 4096.
 * ---------------------------------------------------------------------------------------------- */
int rvo_merge_topk(const int64_t* ids, const float* scores, const int32_t* counts,
                   int32_t G, int32_t nq, int32_t k,
                   int64_t* out_ids, float* out_scores, int32_t* out_counts, void* stream);

/* Same merge over the buffer ONE all-gather produces: G blobs, `rank_stride_bytes` apart, each laid out
 * as [ids int64 nq*k | scores float32 nq*k | counts int32 nq] (rvo_packed_result_bytes(nq,k) bytes,
 * a multiple of 8). */
size_t rvo_packed_result_bytes(int32_t nq, int32_t k);
int rvo_merge_topk_packed(const void* gathered, int64_t rank_stride_bytes, int32_t G, int32_t nq, int32_t k,
                          int64_t* out_ids, float* out_scores, int32_t* out_counts, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Peer-memory exchange for the row-sharded search: K2's last kernel stores each query's list straight into
 * every peer GPU's exchange region over NVLink and the last CTA publishes an epoch flag; K3 waits for the G
 * flags and merges.  Replaces the NCCL all-gather between rvo_search_topk and rvo_merge_topk_packed (same
 * results; no collective launch).  No reference counterpart.
 *   region: rvo_exchange_bytes(world, nq_max, k_max) bytes from rvo_exchange_alloc (a cudaMalloc allocation,
 *           zeroed) on each rank; exported with rvo_exchange_export (64-byte CUDA IPC handle, exchanged by the
 *           host, e.g. torch.distributed.all_gather_object) and mapped by every peer with rvo_exchange_import.
 *   regions [host] array of `world` device pointers valid in THIS process: regions[rank] is the local region,
 *           regions[g] the imported mapping of rank g's.
 *   epoch   1, 2, 3, ... — the same value on every rank for the same search (every rank calls in the same
 *           order); epoch % 4 selects one of FOUR slot sets, so a rank may enqueue the scan of search e+1 before the
 *           merge of search e (pipelined serving) and still never overwrite a slot a peer has not merged yet.
 * rvo_search_topk_push = rvo_search_topk with the result written to this rank's slot of every region; returns
 * RVO_E_UNSUPPORTED for nq <= RVO_SMALL_Q or an empty shard (take the all-gather path on ALL ranks then).
 * rvo_merge_topk_exchange = rvo_merge_topk over the local region once all `world` flags show `epoch`.  It waits like a
 * collective would; after option "exchange_timeout_ms" (default 60000) without the peers' flags it gives up WITHOUT
 * trapping: every out_counts[q] of the batch is -2 and the caller raises or falls back to the all-gather path.
 * ---------------------------------------------------------------------------------------------- */
size_t rvo_exchange_bytes(int32_t world, int32_t nq_max, int32_t k_max);
int rvo_exchange_alloc(size_t bytes, void** out_region);
int rvo_exchange_free(void* region);
int rvo_exchange_export(void* region, void* out_handle64);
int rvo_exchange_import(const void* handle64, void** out_region);
int rvo_exchange_unimport(void* region);
int rvo_search_topk_push(const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad,
                         const float* queries, int32_t nq, int32_t k, float score_threshold, int64_t id_offset,
                         void* const* regions, int32_t world, int32_t rank, int32_t nq_max, int32_t k_max, uint64_t epoch,
                         void* workspace, size_t workspace_bytes, void* stream);
int rvo_merge_topk_exchange(const void* local_region, int32_t world, int32_t nq, int32_t k, int32_t nq_max, int32_t k_max,
                            uint64_t epoch, int64_t* out_ids, float* out_scores, int32_t* out_counts, void* stream);

/* FUSED exchange + merge (world * k <= 2048): rvo_search_topk whose last kernel also does the exchange AND K3.  The CTA of query q
 * stores its shard's list as one record into every rank's region, publishes a per-(rank, query) flag, waits for the peers'
 * flags of the SAME query and merges the `world` lists in shared memory: out_* receive the MERGED result on every rank.  No
 * grid-wide counter, no separate merge launch (measured at 8 GPUs: the stand-alone merge cost 17.6 us + a launch).  Same region,
 * regions table and epoch rules as rvo_search_topk_push; a peer that never publishes gives count -2 after "exchange_timeout_ms".
 * Every rank must call it for the same searches in the same order.  Returns RVO_E_UNSUPPORTED when world * k > 2048, for
 * nq <= RVO_SMALL_Q or an empty shard (use the push or the all-gather path on ALL ranks then). */
int rvo_search_topk_fused(const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad,
                          const float* queries, int32_t nq, int32_t k, float score_threshold, int64_t id_offset,
                          void* const* regions, int32_t world, int32_t rank, int32_t nq_max, int32_t k_max, uint64_t epoch,
                          int64_t* out_ids, float* out_scores, int32_t* out_counts,
                          void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Near-duplicate self-join (BASELINE.json config 4): all pairs (i, j), row_lo <= i < row_hi, i < j < n_rows,
 * with cos(db[i], db[j]) >= threshold — the reference's `score_threshold` rule (core_system.py:663) with every
 * stored row as a query.  The reference has no such feature (video_processing.py only writes frames).
 * Built on K2: blocks of 4096 query rows, FILTER scan of the upper triangle, exact fp32 re-score of candidates.
 *   out_pairs  [dev] int64 [out_cap][2] (i, j) + id_offset, in no particular order
 *   out_scores [dev] float32 [out_cap]  fp32 dot of the two stored bf16 rows
 *   out_count  [dev] uint64 [1]  pairs found (only the first out_cap are stored)
 *   out_overflowed [dev] int32 [1]  candidate sub-lists that overflowed (> 0: result incomplete; raise "cand_cap")
 *   workspace  [dev] rvo_selfjoin_workspace_bytes(d) bytes, 1024-B aligned
 * Multi-GPU, two ways: (1) DB replicated, ranks take disjoint [row_lo, row_hi) ranges; no collective on the data path.
 * (2) DB row-sharded over the devices of one process (B200VectorDB(devices=[...])): rvo_join_threshold below joins each shard
 * with itself (triangle) and every pair of shards (rectangle, 4096-row query blocks copied to the other shard's device, each
 * rectangle split between its two devices); no shard is moved or replicated.
 * Duplicate groups (the connected components of these pairs) without storing any pair: rvo_join_components below.
 * ---------------------------------------------------------------------------------------------- */
size_t rvo_selfjoin_workspace_bytes(int32_t d);
int rvo_selfjoin_threshold(const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad, int64_t row_lo, int64_t row_hi,
                           float threshold, int64_t id_offset, int64_t* out_pairs, float* out_scores, int64_t out_cap,
                           uint64_t* out_count, int32_t* out_overflowed, void* workspace, size_t workspace_bytes,
                           void* stream);

/* Same join with an explicit candidate capacity per query row (instead of option "cand_cap", default 32768): the host raises
 * it and re-runs when out_overflowed > 0 — a row with more near-duplicates than the lists hold (a static video scene) is
 * then joined exactly instead of failing.  cand_cap >= n_rows + 4096 can never overflow. */
size_t rvo_selfjoin_workspace_bytes_ex(int32_t d, int64_t cand_cap);
int rvo_selfjoin_threshold_ex(const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad, int64_t row_lo, int64_t row_hi,
                              float threshold, int64_t id_offset, int64_t cand_cap, int64_t* out_pairs, float* out_scores,
                              int64_t out_cap, uint64_t* out_count, int32_t* out_overflowed, void* workspace,
                              size_t workspace_bytes, void* stream);

/* Threshold join between two row sets on one device, the building block of the self-join of a row-sharded collection.
 *   qdb        [dev] tiled bf16 storage holding the query rows [q_row_lo, q_row_hi); their ids are row + q_id_offset
 *   db         [dev] tiled bf16 storage of the n_rows target rows (a sub-range must start on a 128-row block); ids row + id_offset
 * qdb == db with q_id_offset == id_offset: TRIANGLE, exactly rvo_selfjoin_threshold_ex(db, ..., q_row_lo, q_row_hi, ...) — pairs
 * (i, j), i in the query rows, i < j < n_rows.  Otherwise RECTANGLE: the two row sets must be disjoint (checked by id and by
 * address; both on the same device) and every (query, target) pair at or above the threshold is emitted.  Either way a pair
 * is stored as (lower id, higher id) with the fp32 dot of its two stored bf16 rows, bit-identical in both modes.
 * Unlike rvo_selfjoin_threshold[_ex] this entry APPENDS: pairs go to out_pairs / out_scores from index *out_count on, the
 * count grows by the pairs found (only indices < out_cap are stored), and overflowed candidate sub-lists are ADDED to
 * *out_overflowed; neither is reset, so every join of a device can share one pair buffer and one host synchronisation.
 * cand_cap as in rvo_selfjoin_threshold_ex (>= n_rows + 4096 can never overflow).  workspace: rvo_join_workspace_bytes(d,
 * cand_cap) bytes, 1024-B aligned. */
size_t rvo_join_workspace_bytes(int32_t d, int64_t cand_cap);
int rvo_join_threshold(const uint16_t* qdb, int64_t q_row_lo, int64_t q_row_hi, int64_t q_id_offset,
                       const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad, float threshold, int64_t id_offset,
                       int64_t cand_cap, int64_t* out_pairs, float* out_scores, int64_t out_cap,
                       uint64_t* out_count, int32_t* out_overflowed, void* workspace, size_t workspace_bytes, void* stream);

/* Threshold join between two collections (left and right) on one device: every (query row, target row) pair with cos >= threshold.
 *   qdb        [dev] tiled bf16 storage holding the query rows [q_row_lo, q_row_hi); their ids are row + q_id_offset
 *   db         [dev] tiled bf16 storage of the n_rows target rows (a sub-range must start on a 128-row block); ids row + id_offset
 *   query_is_right  0: the query rows are the left collection, 1: they are the right one
 * A pair is stored as (left id, right id) whichever side provides the query rows, with the fp32 dot of its two stored bf16 rows;
 * the score is bit-identical in both orientations (and equal to the self-join's score of the same two rows).  The ids of the two
 * sides name rows of different collections, so they may overlap; qdb == db is allowed and is then the full ordered join of those
 * rows with themselves, self pairs (i, i) included.  Both buffers must be on the same device.  Appends exactly like
 * rvo_join_threshold (out_count and out_overflowed are added to, never reset); cand_cap and workspace
 * (rvo_join_workspace_bytes(d, cand_cap) bytes, 1024-B aligned) as there. */
int rvo_cross_join_threshold(const uint16_t* qdb, int64_t q_row_lo, int64_t q_row_hi, int64_t q_id_offset,
                             const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad, float threshold,
                             int64_t id_offset, int32_t query_is_right, int64_t cand_cap,
                             int64_t* out_pairs, float* out_scores, int64_t out_cap, uint64_t* out_count,
                             int32_t* out_overflowed, void* workspace, size_t workspace_bytes, void* stream);

/* Connected components of the self-join's pairs (single-linkage groups at a threshold), with no pair stored.
 * rvo_join_components takes the arguments of rvo_join_threshold and examines exactly the pairs it would emit (same scan, same
 * fp32 re-score, same >= threshold test, triangle or rectangle derived the same way), but unions the two global rows of each
 * into a union-find forest instead of storing the pair:
 *   parent     [dev] int32 [n_labels], indexed by global row (ids = row + offset, every one < n_labels < 2^31); initialise it
 *              to parent[x] = x once, then any number of joins (of one device) may union into it.  The forest keeps
 *              parent[x] <= x: a hook sets the larger of two roots to the smaller, so a component's root is its smallest row.
 *   hit_count  [dev] uint64 [1]  pairs at or above the threshold, ADDED to (never reset), like rvo_join_threshold's out_count
 *   out_overflowed  [dev] int32 [1]  overflowed candidate sub-lists, added to; > 0: edges may be missing, re-run with a larger
 *              cand_cap (re-applying an edge changes nothing, so the forest may be kept; reset hit_count first)
 * cand_cap and workspace (rvo_join_workspace_bytes(d, cand_cap) bytes, 1024-B aligned) as in rvo_join_threshold; parent must be
 * on the target rows' device.
 * rvo_components_flatten: labels_out[x] = root of x (int32 [n]): the canonical label, the smallest row of x's component.
 * rvo_components_merge: union(x, labels_src[x]) for every x with labels_src[x] != x (int32 [n], entries outside [0, n)
 * ignored): folds the flattened forest of another device over the same n rows into `parent`; flatten afterwards.
 * All three are asynchronous on `stream`. */
int rvo_join_components(const uint16_t* qdb, int64_t q_row_lo, int64_t q_row_hi, int64_t q_id_offset,
                        const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad, float threshold, int64_t id_offset,
                        int64_t cand_cap, int32_t* parent, int64_t n_labels, uint64_t* hit_count, int32_t* out_overflowed,
                        void* workspace, size_t workspace_bytes, void* stream);
int rvo_components_flatten(int32_t* parent, int64_t n, int32_t* labels_out, void* stream);
int rvo_components_merge(int32_t* parent, const int32_t* labels_src, int64_t n, void* stream);

/* ------------------------------------------------------------------------------------------------
 * k-nearest-neighbour join: for every query row, in order, the k stored rows of `db` with the highest score — K2 with stored
 * rows as its queries.  No reference counterpart (the reference searches one embedded query at a time).
 *   qdb        [dev] tiled bf16 storage holding the query rows; their ids are row + q_id_offset
 *   q_rows     [dev] int64 or NULL: NULL, the query rows are [q_row_lo, q_row_hi); otherwise they are q_rows[q_row_lo ..
 *              q_row_hi) (rows of qdb's capacity)
 *   db         [dev] tiled bf16 storage of the n_rows target rows (may be qdb itself, and may be empty); ids row + id_offset
 *   score      the fp32 dot of the two stored bf16 rows; the query row is NOT re-normalised.  It equals the threshold joins'
 *              score of the same pair up to fp32 summation order.
 *   k          1..RVO_MAX_K, 1..RVO_MAX_K - 1 with exclude_self
 *   score_threshold   hits with score < threshold are dropped (== is kept); -INFINITY for none
 *   exclude_self      1 (self mode: qdb and db are one collection): the query row's own id never appears in its list, its
 *              exact copies do.  The search keeps k + 1 per row and drops the own id when present, else the last entry.
 *   path       RVO_PATH_AUTO: tcgen05 scan for every block of query rows (option "knn_block", default 8192; tails of <= 4
 *              rows included), fused select
 *              and fp32 re-score.  RVO_PATH_SMALL / RVO_PATH_DENSE: the fp32 overflow routes, for at most RVO_SMALL_Q rows
 *              given as a q_rows list (d_pad <= 2048).
 *   out_ids / out_scores / out_counts   as rvo_search_topk, row q for query row q_row_lo + q: [nq, k] ids (score descending,
 *              ties by lower id, -1 pad), scores (-inf pad), counts [nq] (0..k, or -1: the query overflowed the fused path's
 *              candidate lists, re-run it with path SMALL, then DENSE, exactly as rvo_search_topk's flagged queries)
 *   workspace  [dev] rvo_knn_workspace_bytes(n_rows, d, nq, k, path) bytes with nq = q_row_hi - q_row_lo, 1024-B aligned
 * qdb, db and the workspace must be on one device.  Asynchronous on `stream`.
 * rvo_knn_exclude_self: the self mode's exclusion on its own, for lists of k + 1 merged across shards (rvo_merge_topk):
 * ids/scores [nq, k + 1], counts [nq] -> out_* [nq, k]; query q's own id is q_id_offset + (q_rows ? q_rows[q] : q_row_lo + q).
 * ---------------------------------------------------------------------------------------------- */
size_t rvo_knn_workspace_bytes(int64_t n_rows, int32_t d, int32_t nq, int32_t k, int32_t path);
int rvo_knn_join(const uint16_t* qdb, int64_t q_row_lo, int64_t q_row_hi, const int64_t* q_rows, int64_t q_id_offset,
                 const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad, int32_t k, float score_threshold,
                 int64_t id_offset, int32_t exclude_self, int32_t path, int64_t* out_ids, float* out_scores,
                 int32_t* out_counts, void* workspace, size_t workspace_bytes, void* stream);
int rvo_knn_exclude_self(const int64_t* ids, const float* scores, const int32_t* counts, int32_t nq, int32_t k,
                         int64_t q_row_lo, const int64_t* q_rows, int64_t q_id_offset, int64_t* out_ids, float* out_scores,
                         int32_t* out_counts, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Spherical k-means (B200VectorDB.cluster).  Centroids are stored like rows (L2-normalised bf16, tiled, cluster c = row c);
 * a row's label is its rvo_knn_join(k = 1) match against the centroid buffer (ties by the lower index).  The update step:
 * rvo_kmeans_update reads the assignment of rows [row_lo, row_hi) of the tiled storage `db`:
 *   ids        [dev] int64 [n] (n = row_hi - row_lo; the k = 1 lists): cluster = ids[i] - id_offset, -1 outside [0, n_clusters)
 *   prev_labels  [dev] int32 [n] or NULL: the previous labels (NULL: every row counts as changed)
 *   labels     [dev] int32 [n] out: the clusters, -1 for ids outside the range (such rows add nothing)
 *   sums       [dev] int64 [n_clusters][d], ADDED to: each member's bf16 components as integers rint(x * 2^31) (exact for
 *              |x| >= 2^-24; below 2^63 for fewer than 2^31 rows).  Integer addition, so the sums are bit-identical whatever the
 *              launch configuration, the block order or the split of the rows into calls (shards).
 *   counts     [dev] int64 [n_clusters], ADDED to: members per cluster
 *   changed    [dev] int64 [1], ADDED to: rows whose label differs from prev_labels
 *   workspace  [dev] rvo_kmeans_update_workspace_bytes(n, n_clusters) bytes, 256-B aligned
 * db and sums on one device; 1 <= n_clusters <= RVO_KMEANS_MAX_CLUSTERS, n < 2^31.
 * rvo_kmeans_finalize: the new centroids from the (reduced) sums: scratch_f32 [n_clusters][d] = sums * 2^-31 in fp32, then the
 * rows normalised and rounded into the tiled centroid storage `centroids` exactly as rvo_normalize_rows does (an all-zero row
 * stays zero).  out_empty [n_clusters] int32 = 1 for a cluster with no member or an all-zero sum (re-seeded by the caller),
 * n_empty [dev] int64 [1] is ADDED to by their number.
 * All are asynchronous on `stream`.
 * ---------------------------------------------------------------------------------------------- */
#define RVO_KMEANS_MAX_CLUSTERS 65536
size_t rvo_kmeans_update_workspace_bytes(int64_t n_rows, int32_t n_clusters);
int rvo_kmeans_update(const uint16_t* db, int64_t row_lo, int64_t row_hi, int32_t d, int64_t d_pad, const int64_t* ids,
                      int64_t id_offset, int32_t n_clusters, const int32_t* prev_labels, int32_t* labels, int64_t* sums,
                      int64_t* counts, int64_t* changed, void* workspace, size_t workspace_bytes, void* stream);
int rvo_kmeans_finalize(const int64_t* sums, const int64_t* counts, int32_t n_clusters, int32_t d, float* scratch_f32,
                        uint16_t* centroids, int32_t* out_empty, int64_t* n_empty, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Counters for bench.py's `gpu_launches` claim: number of kernels THIS library has launched on the
 * calling process since load (monotonic).
 * ---------------------------------------------------------------------------------------------- */
int64_t rvo_kernel_launch_count(void);

/* Device time of the dominant scan kernel of the LAST rvo_search_topk call on this process (the full-DB
 * FILTER launch of the tcgen05 path, or the fp32 small-q scan), measured with CUDA events recorded on the
 * call's stream around that one launch.  Only recorded while option "time_scan" is 1.  Synchronises on the
 * stop event.  <0 if nothing was recorded. */
float rvo_last_scan_ms(void);

/* Tuning knobs (benchmarks/tests only; defaults reproduce the documented behaviour).
 *   name: "force_path" (0 auto, 1 small-q scan, 2 tcgen05 scan), "m_sub" (0 auto,1,2),
 *         "cand_cap" (candidates per query, default 32768), "final_ratio" (default 48),
 *         "time_scan" (0/1, see rvo_last_scan_ms), "pool_path" (0 auto: tensor-core mask pooling when the
 *         shape fits TMEM, 1: CUDA-core kernels), "hot" (1 default: hot candidate sub-lists + one-pass final select,
 *         0: general select only), "exchange_timeout_ms" (peer-exchange wait limit, default 60000),
 *         "seed_max" (1 default: the seed scan writes one maximum per 32 sample rows; 0: every score),
 *         "pdl" (programmatic dependent launch along the search chain: 0 default off, 2 tensor-path chain, 1 also the Q <= 4 chain),
 *         "knn_block" (query rows per search block of rvo_knn_join, 256..16384, default 8192; rvo_knn_workspace_bytes follows it),
 *         debugging (value = a device pointer the caller owns, 0 = off): "chain_trace" (u64 [8][2]: earliest start / latest end
 *         of normalise, seed scan, seed threshold, scan, select on %globaltimer; initialise to (UINT64_MAX, 0) pairs),
 *         "select_trace" (u64 [nq][16] phase stamps of the last-level select), "merge_trace" (u64 [3]), "pool_trace".        */
int rvo_set_option(const char* name, int64_t value);

#ifdef __cplusplus
}
#endif
#endif /* REVERS_O_B200_H */
