// Spherical k-means (rvo_kmeans_update, rvo_kmeans_finalize): the update step of B200VectorDB.cluster.  The assignment is
// rvo_knn_join with k = 1 against the centroid buffer; this file turns it into labels and per-cluster integer sums.
//   label     ids [n] (the k = 1 lists) -> int32 labels, the count of labels that differ from the previous ones, a label
//             histogram in the workspace
//   scan      exclusive scan of the histogram (one CTA), added to the caller's member counts
//   scatter   row indices counting-sorted by label (the order inside one label is whatever the atomics give: irrelevant,
//             the sums are integer)
//   sum       each CTA walks kSumRows consecutive sorted positions with one thread per 8 columns, sums runs of equal labels
//             in int64 registers and flushes a run once with integer atomics: about (n / kSumRows + C) * d atomics instead of
//             n * d.  Each bf16 component x is taken as the integer rint(x * 2^31): exact for |x| >= 2^-24 (8 significant
//             bits), and a sum of fewer than 2^31 rows with |x| <= 1 + 2^-8 stays below 2^63.  Integer addition is
//             associative, so the sums are bit-identical for any grouping: CTA, block order, shard layout.
//   finalize  sums -> fp32 (x 2^-31, exact scaling) and the empty-cluster flags (no member, or an all-zero sum); the caller's
//             fp32 rows are then normalised into the tiled centroid buffer by the normalise launch rvo_normalize_rows uses.
#include "common.cuh"

namespace rvo {

constexpr int kSumRows = 256;      // sorted positions per CTA of the sum kernel
constexpr int kSumThreads = 128;   // column groups of 8 per CTA (blockIdx.y walks wider rows)

__global__ void __launch_bounds__(256) kmeans_label_kernel(const int64_t* __restrict__ ids, long long n, int C, long long id_offset,
                                                           const int32_t* __restrict__ prev, int32_t* __restrict__ labels,
                                                           unsigned long long* __restrict__ changed, int* __restrict__ hist) {
    for (long long base = (long long)blockIdx.x * blockDim.x; base < n; base += (long long)gridDim.x * blockDim.x) {
        const long long i = base + threadIdx.x;
        bool diff = false;
        if (i < n) {
            const long long c = ids[i] - id_offset;
            const int lab = (c >= 0 && c < C) ? (int)c : -1;
            labels[i] = lab;
            diff = !prev || prev[i] != lab;
            if (lab >= 0) atomicAdd(hist + lab, 1);
        }
        const unsigned b = __ballot_sync(0xFFFFFFFFu, diff);
        if ((threadIdx.x & 31) == 0 && b) atomicAdd(changed, (unsigned long long)__popc(b));
    }
}

// One CTA of 1024 threads, thread t owns clusters [t * per, (t + 1) * per).  offs[c] = members of clusters < c (the scatter
// cursor); offs[C] = all labelled rows.  counts[c] += hist[c].
__global__ void __launch_bounds__(1024) kmeans_scan_kernel(const int* __restrict__ hist, int C, int* __restrict__ offs,
                                                           unsigned long long* __restrict__ counts) {
    __shared__ int part[1024];
    const int per = (C + 1023) / 1024;
    const int c0 = threadIdx.x * per, c1 = min(C, c0 + per);
    int s = 0;
    for (int c = c0; c < c1; ++c) s += hist[c];
    part[threadIdx.x] = s;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {               // inclusive Hillis-Steele scan of the 1024 partial sums
        const int v = threadIdx.x >= o ? part[threadIdx.x - o] : 0;
        __syncthreads();
        part[threadIdx.x] += v;
        __syncthreads();
    }
    int run = part[threadIdx.x] - s;
    for (int c = c0; c < c1; ++c) {
        const int h = hist[c];
        offs[c] = run;
        run += h;
        if (h) counts[c] += (unsigned long long)h;
    }
    if (threadIdx.x == 1023) offs[C] = part[1023];
}

__global__ void __launch_bounds__(256) kmeans_scatter_kernel(const int32_t* __restrict__ labels, long long n, int* __restrict__ cursor,
                                                             int* __restrict__ order) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int lab = labels[i];
        if (lab >= 0) order[atomicAdd(cursor + lab, 1)] = (int)i;
    }
}

__device__ __forceinline__ void kmeans_flush(long long* __restrict__ sums, int lab, int d, int col0, const long long* acc) {
#pragma unroll
    for (int j = 0; j < 8; ++j)
        if (acc[j] && col0 + j < d) atomicAdd((unsigned long long*)(sums + (size_t)lab * d + col0 + j), (unsigned long long)acc[j]);
}

// grid (ceil(n / kSumRows), ceil(d_pad / 8 / kSumThreads)), kSumThreads threads.  Sorted positions [p0, p0 + kSumRows) of
// `order` (local rows of the range starting at row_lo of the tiled storage db); thread t sums columns [8 g, 8 g + 8),
// g = blockIdx.y * kSumThreads + t.
__global__ void __launch_bounds__(kSumThreads) kmeans_sum_kernel(const uint4* __restrict__ db, long long row_lo, int d, int d_pad,
                                                                 const int* __restrict__ order, const int32_t* __restrict__ labels,
                                                                 const int* __restrict__ total, long long* __restrict__ sums) {
    __shared__ int s_row[kSumRows], s_lab[kSumRows];
    const long long p0 = (long long)blockIdx.x * kSumRows;
    const int m = *total;
    if (p0 >= m) return;
    const int cnt = (int)min((long long)kSumRows, m - p0);
    for (int j = threadIdx.x; j < cnt; j += kSumThreads) {
        const int r = order[p0 + j];
        s_row[j] = r;
        s_lab[j] = labels[r];
    }
    __syncthreads();
    const int nchunk = d_pad >> 3, nk = d_pad / kTileCols;
    const int g = blockIdx.y * kSumThreads + threadIdx.x;
    if (g >= nchunk) return;
    long long acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0;
    int cur = s_lab[0];
    for (int p = 0; p < cnt; p += 4) {
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {                  // four loads in flight before any arithmetic
            v[u] = make_uint4(0, 0, 0, 0);
            if (p + u < cnt) {
                const long long r = row_lo + s_row[p + u];
                v[u] = __ldg(db + (((size_t)(r >> 7) * nk + (g >> 3)) * kTileRows + (r & 127)) * 8 + (g & 7));
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (p + u >= cnt) break;
            const int lab = s_lab[p + u];
            if (lab != cur) {
                kmeans_flush(sums, cur, d, g * 8, acc);
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[j] = 0;
                cur = lab;
            }
            const uint32_t w[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
            for (int h = 0; h < 4; ++h) {              // bf16 element 2h is the low half of word h, element 2h + 1 the high half
                acc[2 * h] += __float2ll_rn(__uint_as_float(w[h] << 16) * 2147483648.0f);
                acc[2 * h + 1] += __float2ll_rn(__uint_as_float(w[h] & 0xFFFF0000u) * 2147483648.0f);
            }
        }
    }
    kmeans_flush(sums, cur, d, g * 8, acc);
}

// One CTA per cluster.  out[c][:] = sums[c][:] * 2^-31 in fp32; empty[c] = no member or an all-zero sum, counted in n_empty.
__global__ void __launch_bounds__(256) kmeans_finalize_kernel(const long long* __restrict__ sums, const long long* __restrict__ counts,
                                                              int d, float* __restrict__ out, int32_t* __restrict__ empty,
                                                              unsigned long long* __restrict__ n_empty) {
    const int c = blockIdx.x;
    bool nz = false;
    for (int j = threadIdx.x; j < d; j += blockDim.x) {
        const long long v = sums[(size_t)c * d + j];
        nz |= v != 0;
        out[(size_t)c * d + j] = __ll2float_rn(v) * 4.656612873077393e-10f;
    }
    nz = __syncthreads_or(nz);
    if (threadIdx.x == 0) {
        const bool e = counts[c] == 0 || !nz;
        empty[c] = e;
        if (e) atomicAdd(n_empty, 1ull);
    }
}

// Workspace of launch_kmeans_update: histogram [C], cursor [C + 1], order [n].
size_t kmeans_update_workspace_bytes(long long n, int C) {
    return align_up((size_t)C * 4, 256) + align_up((size_t)(C + 1) * 4, 256) + align_up((size_t)n * 4, 256);
}

int launch_kmeans_update(const uint16_t* db, long long row_lo, long long n, int d, int d_pad, const int64_t* ids, long long id_offset,
                         int C, const int32_t* prev, int32_t* labels, int64_t* sums, int64_t* counts, int64_t* changed, void* ws,
                         int sm_count, cudaStream_t stream) {
    char* w = (char*)ws;
    int* hist = (int*)w;
    int* offs = (int*)(w + align_up((size_t)C * 4, 256));
    int* order = (int*)((char*)offs + align_up((size_t)(C + 1) * 4, 256));
    RVO_CUDA(cudaMemsetAsync(hist, 0, (size_t)C * 4, stream));
    if (n == 0) return RVO_OK;
    const unsigned grid = (unsigned)min((n + 255) / 256, (long long)sm_count * 8);
    kmeans_label_kernel<<<grid, 256, 0, stream>>>(ids, n, C, id_offset, prev, labels, (unsigned long long*)changed, hist);
    RVO_LAUNCHED();
    kmeans_scan_kernel<<<1, 1024, 0, stream>>>(hist, C, offs, (unsigned long long*)counts);
    RVO_LAUNCHED();
    kmeans_scatter_kernel<<<grid, 256, 0, stream>>>(labels, n, offs, order);
    RVO_LAUNCHED();
    // the scatter leaves offs[c] at the end of cluster c; offs[C] (all labelled rows) is untouched
    const dim3 sgrid((unsigned)((n + kSumRows - 1) / kSumRows), (unsigned)((d_pad / 8 + kSumThreads - 1) / kSumThreads));
    kmeans_sum_kernel<<<sgrid, kSumThreads, 0, stream>>>((const uint4*)db, row_lo, d, d_pad, order, labels, offs + C, (long long*)sums);
    RVO_LAUNCHED();
    return RVO_OK;
}

int launch_kmeans_finalize(const int64_t* sums, const int64_t* counts, int C, int d, float* out, int32_t* empty, int64_t* n_empty,
                           cudaStream_t stream) {
    kmeans_finalize_kernel<<<C, 256, 0, stream>>>((const long long*)sums, (const long long*)counts, d, out, empty,
                                                  (unsigned long long*)n_empty);
    RVO_LAUNCHED();
    return RVO_OK;
}

}  // namespace rvo
