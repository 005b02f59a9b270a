// Near-duplicate self-join (BASELINE.json config 4; SURVEY.md §8f row 1): every stored row is a query and the
// reference's `score_threshold` (core_system.py:663) is the only selection rule — all pairs (i, j), i < j, with
// cos(db[i], db[j]) >= threshold.  The reference has no such feature; it reuses K2 unchanged:
//   per block of up to 4096 query rows:  gather the rows out of the tiled query buffer (they ARE bf16, so the tensor-core
//   scores are exact up to fp32 summation order) -> FILTER scan of the target rows with tau = threshold - 1e-4 ->
//   `pairs_kernel`: fp32 re-score of every candidate, append (min id, max id, score).
// Two modes share that code:
//   TRIANGLE  query rows and target rows are the same tiled DB: block b scans only rows >= its first row and keeps j > i,
//             i.e. N^2 * D flops, not 2 N^2 D.
//   RECTANGLE the query rows come from another tiled buffer on the same device (a block of another shard copied here) and
//             are disjoint from the target rows: every target row is scanned, every candidate re-scored.  Used for the
//             cross-shard part of the join of a row-sharded collection.
// The re-score runs the same lanes over the same chunks in the same order in both modes and fmaf is commutative in its two
// factors, so a pair scores bit-identically whichever of its rows is the query.
#include "common.cuh"
#include "scan_tc.cuh"
#include "prep_scan_small.cuh"

namespace rvo {

constexpr float kSelfJoinMargin = 1e-4f;   // fp32 summation-order slack between the MMA and the re-score

// q_out[q][:] = qdb row (row0 + q), row-major bf16 [nq_pad][d_pad]; rows q >= nq are zero.  tau[q] = thr or +inf.
__global__ void __launch_bounds__(256) gather_rows_kernel(const uint4* __restrict__ qdb, long long row0, int nq, int nq_pad,
                                                          int d_pad, uint4* __restrict__ q_out, float* __restrict__ tau,
                                                          float thr) {
    const int q = blockIdx.x;
    const int nchunk = d_pad >> 3, nk = d_pad / kTileCols;
    if (threadIdx.x == 0) tau[q] = q < nq ? thr : __int_as_float(0x7f800000);
    const long long r = row0 + q;
    for (int c = threadIdx.x; c < nchunk; c += blockDim.x) {
        uint4 v = make_uint4(0, 0, 0, 0);
        if (q < nq) v = __ldg(qdb + (((size_t)(r >> 7) * nk + (c >> 3)) * kTileRows + (r & 127)) * 8 + (c & 7));
        q_out[(size_t)q * nchunk + c] = v;
    }
    (void)nq_pad;
}

__device__ __forceinline__ float dot8(const uint4 a, const uint4 b, float acc) {
    const uint32_t x[4] = {a.x, a.y, a.z, a.w}, y[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
    for (int h = 0; h < 4; ++h) {
        acc = fmaf(__uint_as_float(x[h] << 16), __uint_as_float(y[h] << 16), acc);
        acc = fmaf(__uint_as_float(x[h] & 0xFFFF0000u), __uint_as_float(y[h] & 0xFFFF0000u), acc);
    }
    return acc;
}

// grid (nq), 256 threads: candidates of query row i = row0 + q; 8 lanes per candidate.  j_floor: a candidate j is re-scored
// when j > j_floor — the query row i in TRIANGLE mode (upper triangle, no self pair), -1 in RECTANGLE mode (every candidate).
// Pairs are emitted as (min, max) of (i + q_id_offset, j + id_offset).
__global__ void __launch_bounds__(256) pairs_kernel(const uint4* __restrict__ db, const uint4* __restrict__ qrows, long long row0,
                                                    long long scan_base, int d_pad, const unsigned long long* __restrict__ cand,
                                                    const int* __restrict__ cnt, int cap, float threshold, bool triangle,
                                                    long long q_id_offset, long long id_offset, long long* __restrict__ out_pairs,
                                                    float* __restrict__ out_scores, long long out_cap,
                                                    unsigned long long* __restrict__ out_count, int* __restrict__ overflowed) {
    const int q = blockIdx.x;
    const long long i = row0 + q;
    const long long j_floor = triangle ? i : -1;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    const int g = lane >> 3, l8 = lane & 7;
    const int nchunk = d_pad >> 3, nk = d_pad / kTileCols;
    const uint4* qr = qrows + (size_t)q * nchunk;
    for (int sgm = 0; sgm < kCandSplit; ++sgm) {
        int c = cnt[q * kCandSplit + sgm];
        if (c > cap) {
            if (threadIdx.x == 0) atomicAdd(overflowed, 1);
            c = cap;
        }
        const unsigned long long* list = cand + ((size_t)q * kCandSplit + sgm) * (size_t)cap;
        for (int e0 = 0; e0 < c; e0 += nwarps * 4) {
            const int e = e0 + warp * 4 + g;
            long long j = -1;
            if (e < c) j = scan_base + (long long)key_row(list[e]);
            const bool active = e < c && j > j_floor;
            float acc = 0.f;
            if (active) {
                const uint4* r = db + ((size_t)(j >> 7) * nk * kTileRows + (j & 127)) * 8;
                for (int cc = l8; cc < nchunk; cc += 8)
                    acc = dot8(__ldg(r + (size_t)(cc >> 3) * kTileRows * 8 + (cc & 7)), __ldg(qr + cc), acc);
            }
#pragma unroll
            for (int o = 4; o > 0; o >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, o);
            const bool hit = active && l8 == 0 && acc >= threshold;
            const unsigned bal = __ballot_sync(0xFFFFFFFFu, hit);
            if (bal) {
                unsigned long long base = 0;
                if (lane == 0) base = atomicAdd(out_count, (unsigned long long)__popc(bal));
                base = __shfl_sync(0xFFFFFFFFu, base, 0);
                if (hit) {
                    const unsigned long long at = base + __popc(bal & ((1u << lane) - 1u));
                    if ((long long)at < out_cap) {
                        const long long gi = i + q_id_offset, gj = j + id_offset;
                        out_pairs[2 * at] = gi < gj ? gi : gj;
                        out_pairs[2 * at + 1] = gi < gj ? gj : gi;
                        out_scores[at] = acc;
                    }
                }
            }
        }
    }
}

constexpr int kSelfJoinBlock = 4096;   // query rows per scan (16 query blocks of 256)

struct SelfJoinPlan {
    TcPlan tc;
    int d_pad, cap;
    uint16_t* qb;
    float* tau;
    int* cnt;
    unsigned long long* cand;
    int* overflowed;
    size_t bytes;
};

static int selfjoin_plan(int d, long long cand_cap, void* ws, size_t ws_bytes, SelfJoinPlan* sp) {
    sp->d_pad = (d + kBlockK - 1) / kBlockK * kBlockK;
    int rc = plan_scan_tc(kSelfJoinBlock, sp->d_pad, 0, &sp->tc);
    if (rc) return rc;
    long long cap = cand_cap / kCandSplit;
    if (cap < 64) cap = 64;
    sp->cap = (int)cap;
    Arena ar(ws, ws_bytes);
    sp->qb = ar.take<uint16_t>((size_t)sp->tc.nq_pad * sp->d_pad, 1024);
    sp->tau = ar.take<float>(sp->tc.nq_pad);
    sp->cnt = ar.take<int>((size_t)sp->tc.nq_pad * kCandSplit);
    sp->overflowed = ar.take<int>(1);
    sp->cand = ar.take<unsigned long long>((size_t)sp->tc.nq_pad * kCandSplit * (size_t)sp->cap);
    sp->bytes = ar.off + 1024;
    if (ws && !ar.ok()) {
        set_error("selfjoin workspace too small: %zu bytes given, %zu needed", ws_bytes, sp->bytes);
        return RVO_E_WORKSPACE;
    }
    return RVO_OK;
}

size_t selfjoin_workspace_bytes(int d, long long cand_cap) {
    SelfJoinPlan sp;
    if (selfjoin_plan(d, cand_cap, nullptr, 0, &sp)) return 0;
    return sp.bytes;
}

// Query rows [q_row_lo, q_row_hi) of `qdb` against the n_rows target rows of `db` (TRIANGLE when qdb == db and the id offsets
// are equal, RECTANGLE otherwise: the caller guarantees disjoint row sets).  append == false: *out_count and *out_overflowed
// are reset first (rvo_selfjoin_threshold[_ex]); append == true: pairs are appended at *out_count and overflowed candidate
// sub-lists are added to *out_overflowed (rvo_join_threshold: every join of a device shares one pair buffer).
int launch_selfjoin(const uint16_t* qdb, long long q_row_lo, long long q_row_hi, long long q_id_offset, const uint16_t* db,
                    long long n_rows, int d, float threshold, long long id_offset, long long cand_cap, long long* out_pairs,
                    float* out_scores, long long out_cap, unsigned long long* out_count, int* out_overflowed, bool append,
                    void* ws, size_t ws_bytes, int sm_count, cudaStream_t stream) {
    SelfJoinPlan sp;
    int rc = selfjoin_plan(d, cand_cap, ws, ws_bytes, &sp);
    if (rc) return rc;
    const bool triangle = qdb == db && q_id_offset == id_offset;
    int* overflowed = append ? out_overflowed : sp.overflowed;
    if (!append) {
        RVO_CUDA(cudaMemsetAsync(out_count, 0, sizeof(unsigned long long), stream));
        RVO_CUDA(cudaMemsetAsync(sp.overflowed, 0, sizeof(int), stream));
    }
    const int nk = sp.d_pad / kTileCols;
    for (long long i0 = q_row_lo; i0 < q_row_hi; i0 += kSelfJoinBlock) {
        const int nq = (int)((q_row_hi - i0) < kSelfJoinBlock ? (q_row_hi - i0) : kSelfJoinBlock);
        gather_rows_kernel<<<sp.tc.nq_pad, 256, 0, stream>>>((const uint4*)qdb, i0, nq, sp.tc.nq_pad, sp.d_pad, (uint4*)sp.qb,
                                                             sp.tau, threshold - kSelfJoinMargin);
        RVO_LAUNCHED();
        RVO_CUDA(cudaMemsetAsync(sp.cnt, 0, (size_t)sp.tc.nq_pad * kCandSplit * sizeof(int), stream));
        // upper triangle: scan only the 128-row blocks at or after the first query row of this block; rectangle: every row
        const long long blk0 = triangle ? i0 / kTileRows : 0;
        const long long scan_base = blk0 * kTileRows;
        const uint16_t* db_sub = db + (size_t)blk0 * nk * kTileRows * kTileCols;
        rc = launch_scan_tc(kModeFilter, db_sub, n_rows - scan_base, 1, sp.d_pad, sp.qb, sp.tc, sp.tau, sp.cand, sp.cnt, sp.cap,
                            nullptr, 0, sm_count, stream);
        if (rc) return rc;
        pairs_kernel<<<nq, 256, 0, stream>>>((const uint4*)db, (const uint4*)sp.qb, i0, scan_base, sp.d_pad, sp.cand, sp.cnt,
                                             sp.cap, threshold, triangle, q_id_offset, id_offset, out_pairs, out_scores, out_cap,
                                             out_count, overflowed);
        RVO_LAUNCHED();
    }
    if (!append && out_overflowed)
        RVO_CUDA(cudaMemcpyAsync(out_overflowed, sp.overflowed, sizeof(int), cudaMemcpyDeviceToDevice, stream));
    return RVO_OK;
}

}  // namespace rvo
