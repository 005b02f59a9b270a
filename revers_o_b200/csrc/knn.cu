// k-nearest-neighbour join (rvo_knn_join): stored rows as K2 queries, and the self exclusion of the self mode.
//   intake    the counterpart of the normalise launch for rows that are already stored: the query operand is copied out of
//             the tiled storage as is.  The rows ARE the bf16 MMA operand and their fp32 upconvert is exact, so the re-score
//             query equals the MMA query and the admission margin is query_margin(0) (common.cuh).  No re-normalisation: a
//             score is the fp32 dot of the two stored rows, the quantity the threshold joins report.
//   exclude   [nq][k+1] lists -> [nq][k] without the query row itself.
// The intake is kept apart from selfjoin.cu's gather_rows_kernel: that kernel also writes the join's threshold vector, and
// extending it with the fp32 copy, the margin and the counter clearing would change the code the self-join runs.
#include "common.cuh"

namespace rvo {

// grid (n_pad_rows), 256 threads.  Row q < nq of the query operand is row (rows ? rows[q] : row0 + q) of the tiled storage
// qdb: qb[q][:] its bf16 copy (row-major [n_pad_rows][d_pad]; null on the fp32 scan, which needs none), qn[q][:] the exact
// fp32 upconvert ([n_pad_rows][d_pad]), margin[q] = query_margin(0) (may be null).  Rows q >= nq are zero with margin 0.  The
// same launch clears zero_u4 16-byte words at zero_base (the candidate counters), as the normalise launch does.
__global__ void __launch_bounds__(256) knn_intake_kernel(const uint4* __restrict__ qdb, long long row0,
                                                         const long long* __restrict__ rows, int nq, int d_pad,
                                                         uint4* __restrict__ qb, float4* __restrict__ qn,
                                                         float* __restrict__ margin, uint4* __restrict__ zero_base,
                                                         long long zero_u4) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < zero_u4; i += (long long)gridDim.x * blockDim.x)
        zero_base[i] = make_uint4(0, 0, 0, 0);
    const int q = blockIdx.x;
    const int nchunk = d_pad >> 3, nk = d_pad / kTileCols;
    const bool live = q < nq;
    const long long r = live ? (rows ? rows[q] : row0 + q) : 0;
    if (margin && threadIdx.x == 0) margin[q] = live ? query_margin(0.f) : 0.f;
    for (int c = threadIdx.x; c < nchunk; c += blockDim.x) {
        uint4 v = make_uint4(0, 0, 0, 0);
        if (live) v = __ldg(qdb + (((size_t)(r >> 7) * nk + (c >> 3)) * kTileRows + (r & 127)) * 8 + (c & 7));
        if (qb) qb[(size_t)q * nchunk + c] = v;
        // bf16 element 2h is the low half of word h, element 2h + 1 the high half
        qn[((size_t)q * nchunk + c) * 2] = make_float4(__uint_as_float(v.x << 16), __uint_as_float(v.x & 0xFFFF0000u),
                                                       __uint_as_float(v.y << 16), __uint_as_float(v.y & 0xFFFF0000u));
        qn[((size_t)q * nchunk + c) * 2 + 1] = make_float4(__uint_as_float(v.z << 16), __uint_as_float(v.z & 0xFFFF0000u),
                                                           __uint_as_float(v.w << 16), __uint_as_float(v.w & 0xFFFF0000u));
    }
}

// One warp per query.  Query q's own id is q_id_offset + (rows ? rows[q] : row0 + q).  Its list of k + 1 (ids, scores, count)
// becomes a list of k: the entry with the query's id is dropped when present, otherwise the last entry is.  This is exact: the
// top k of "every row but i" is the top k + 1 of every row with i removed when present, and otherwise its first k, because
// removing one element from a total order does not reorder the others.  A count of -1 (overflowed) stays -1.
__global__ void __launch_bounds__(256) knn_exclude_kernel(const int64_t* __restrict__ ids, const float* __restrict__ scores,
                                                          const int32_t* __restrict__ counts, int nq, int k, long long row0,
                                                          const long long* __restrict__ rows, long long q_id_offset,
                                                          int64_t* __restrict__ out_ids, float* __restrict__ out_scores,
                                                          int32_t* __restrict__ out_counts) {
    const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= nq) return;
    const int kin = k + 1;
    const int c = counts[w];
    const long long self = q_id_offset + (rows ? rows[w] : row0 + w);
    const int64_t* in_ids = ids + (size_t)w * kin;
    const float* in_scores = scores + (size_t)w * kin;
    int pos = c > 0 ? c : 0;       // position of the query's own id among the first c entries (c: absent)
    for (int j = lane; j < c; j += 32)
        if (in_ids[j] == self) pos = j;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) pos = min(pos, __shfl_xor_sync(0xFFFFFFFFu, pos, o));
    const int cout = c < 0 ? -1 : (pos < c ? c - 1 : min(c, k));
    for (int j = lane; j < k; j += 32) {
        const int src = j < pos ? j : j + 1;
        const bool valid = j < cout;
        out_ids[(size_t)w * k + j] = valid ? in_ids[src] : -1;
        out_scores[(size_t)w * k + j] = valid ? in_scores[src] : -__int_as_float(0x7f800000);
    }
    if (lane == 0) out_counts[w] = cout;
}

int launch_knn_intake(const uint16_t* qdb, long long row0, const int64_t* rows, int nq, int n_pad_rows, int d_pad, uint16_t* qb,
                      float* qn, float* margin, void* zero_base, size_t zero_bytes, cudaStream_t stream) {
    knn_intake_kernel<<<n_pad_rows, 256, 0, stream>>>((const uint4*)qdb, row0, (const long long*)rows, nq, d_pad, (uint4*)qb,
                                                      (float4*)qn, margin, (uint4*)zero_base, (long long)(zero_bytes / 16));
    RVO_LAUNCHED();
    return RVO_OK;
}

int launch_knn_exclude(const int64_t* ids, const float* scores, const int32_t* counts, int nq, int k, long long row0,
                       const int64_t* rows, long long q_id_offset, int64_t* out_ids, float* out_scores, int32_t* out_counts,
                       cudaStream_t stream) {
    if (nq <= 0) return RVO_OK;
    knn_exclude_kernel<<<(unsigned)((nq + 7) / 8), 256, 0, stream>>>(ids, scores, counts, nq, k, row0, (const long long*)rows,
                                                                    q_id_offset, out_ids, out_scores, out_counts);
    RVO_LAUNCHED();
    return RVO_OK;
}

}  // namespace rvo
