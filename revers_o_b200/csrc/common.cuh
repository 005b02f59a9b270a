// Shared host/device helpers for the revers-o B200 hot-path library.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <atomic>

#include "../../include/revers_o_b200.h"

namespace rvo {

// ---- error plumbing (thread-local text behind rvo_last_error) --------------------------------
void set_error(const char* fmt, ...);
extern std::atomic<long long> g_launches;

#define RVO_CUDA(call)                                                                        \
    do {                                                                                      \
        cudaError_t e__ = (call);                                                             \
        if (e__ != cudaSuccess) {                                                             \
            rvo::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, \
                           __LINE__);                                                         \
            return RVO_E_CUDA;                                                                \
        }                                                                                     \
    } while (0)

#define RVO_REQUIRE(cond, ...)          \
    do {                                \
        if (!(cond)) {                  \
            rvo::set_error(__VA_ARGS__); \
            return RVO_E_INVALID;       \
        }                               \
    } while (0)

// every kernel launch of the library goes through this so that bench.py's gpu_launches is a count
#define RVO_LAUNCHED()                                  \
    do {                                                \
        rvo::g_launches.fetch_add(1);                   \
        RVO_CUDA(cudaGetLastError());                   \
    } while (0)

int select_device_of(const void* dev_ptr, int* sm_count);

// Launch with programmatic stream serialization (see ptx.cuh): the kernel must call grid_dependency_wait() before it
// reads or writes global memory a predecessor may touch.
// option "pdl": 0 (default) off; 2 the tensor-path chain only — normalise -> seed scan -> seed threshold -> scan -> select overlap
// their launch latencies and prologues; 1 also the Q <= 4 chain.  Measured with the in-stream timeline (scripts/dev/trace_chain.py)
// and same-box bench runs: 96.3 -> 92.2 us per step on a 125k-row shard (the 8-GPU shard of configs[1]), but nothing at 1M rows,
// where the board's power cap sets the period (serial 0.4669 -> 0.4648 ms, two batches in flight 0.4604 -> 0.4634), and 30 us
// WORSE on the Q <= 4 chain — hence off by default.
extern std::atomic<long long> g_use_pdl;
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl_if(bool on, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                        cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = on ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                     Args... args) {
    return launch_pdl_if(g_use_pdl.load() != 0, kernel, grid, block, smem, stream, args...);
}
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl_small(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                           Args... args) {
    return launch_pdl_if(g_use_pdl.load() == 1, kernel, grid, block, smem, stream, args...);
}

// option "chain_trace": device buffer u64 [8][2] (earliest start, latest end of the CTAs of one kernel, %globaltimer ns) filled
// by the kernels of the search chain: 0 normalise, 1 seed scan, 2 seed threshold, 3 FILTER scan(s), 4 select.  The caller initialises
// it to (UINT64_MAX, 0) pairs (scripts/dev/trace_chain.py); nullptr (the default) costs one predicated branch per CTA.
extern std::atomic<long long> g_chain_trace;
#ifdef __CUDACC__
__device__ __forceinline__ void chain_stamp(unsigned long long* tr, int id, bool end) {
    if (tr && threadIdx.x == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
        if (end) atomicMax(tr + 2 * id + 1, t);
        else atomicMin(tr + 2 * id, t);
    }
}
#endif

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// bump allocator over the caller's workspace
struct Arena {
    char* base;
    size_t size, off;
    Arena(void* p, size_t n) : base((char*)p), size(n), off(0) {}
    template <typename T>
    T* take(size_t count, size_t align = 256) {
        off = align_up(off, align);
        T* r = (T*)(base ? base + off : nullptr);
        off += count * sizeof(T);
        return r;
    }
    bool ok() const { return off <= size; }
};

// ---- ordering keys -----------------------------------------------------------------------------
// 64-bit key = (orderable(score) << 32) | (0xFFFFFFFF - row): a DESCENDING sort of keys is
// score-descending with ties broken by LOWER row.  Key 0 is "empty" (below every real key).
__host__ __device__ __forceinline__ uint32_t f32_orderable(float f) {
#ifdef __CUDA_ARCH__
    uint32_t b = __float_as_uint(f);
#else
    uint32_t b;
    memcpy(&b, &f, 4);
#endif
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__host__ __device__ __forceinline__ float orderable_f32(uint32_t o) {
    uint32_t b = (o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o;
#ifdef __CUDA_ARCH__
    return __uint_as_float(b);
#else
    float f;
    memcpy(&f, &b, 4);
    return f;
#endif
}
__host__ __device__ __forceinline__ unsigned long long make_key(float score, uint32_t row) {
    return ((unsigned long long)f32_orderable(score) << 32) | (unsigned long long)(0xFFFFFFFFu - row);
}
__host__ __device__ __forceinline__ float key_score(unsigned long long k) { return orderable_f32((uint32_t)(k >> 32)); }
__host__ __device__ __forceinline__ uint32_t key_row(unsigned long long k) { return 0xFFFFFFFFu - (uint32_t)(k & 0xFFFFFFFFu); }

// ---- tiled DB storage ------------------------------------------------------------------------------
// bf16 element (row, col) of a DB stored as [row / 128][d_pad / 64][128][64]: every (row block, k-chunk)
// tile is one contiguous 16 KiB block, which is exactly one TMA box of the scan kernel, so the scan
// streams HBM in long contiguous bursts instead of 128-byte pieces 2 KiB apart (DESIGN.md §3).
constexpr int kTileRows = 128;
constexpr int kTileCols = 64;
__host__ __device__ __forceinline__ size_t tiled_offset(long long row, int col, int nk) {
    return ((size_t)(row >> 7) * (size_t)nk + (size_t)(col >> 6)) * (size_t)(kTileRows * kTileCols) +
           (size_t)(row & 127) * kTileCols + (size_t)(col & 63);
}

// Admission margin of a query whose MMA operand is bf16(q_hat) while the final ranking uses the fp32 re-score
// f = <q_hat, d>.  DB rows are L2-normalised bf16 values (||d|| <= 1 + 2^-8), so
//     |<bf16(q_hat), d> - <q_hat, d>|  <=  ||bf16(q_hat) - q_hat|| * ||d||  =: eps_q      (Cauchy-Schwarz),
// with ||bf16(q_hat) - q_hat|| MEASURED per query by the normalise kernel (about 1.7e-3 for random directions, 2.3x
// below the worst case 2^-8).  If t(k) is the k-th best TENSOR score of any subset of the DB, k rows have tensor score >= t(k),
// hence f >= t(k) - eps_q; so the k-th best f is >= t(k) - eps_q, and every row of the true top-k has tensor score
// >= t(k) - 2 eps_q.  Thresholds taken from tensor-core scores are therefore lowered by margin = 2 eps_q, where eps_q
// also carries 2^-13 of slack for fp32 accumulation-order differences between tile shapes and the fp32 FMA re-score.
// A STORED row as the query (rvo_knn_join) is its own bf16 operand: bf16(q) == q, so ||bf16(q) - q|| = 0 and eps_q is the
// accumulation slack alone, query_margin(0) = 2^-12.  The re-score query is the exact fp32 upconvert of the same row, so the
// bound above holds unchanged with the raw (not re-normalised) row; ||q|| <= 1 + 2^-8 like any stored row.
__host__ __device__ __forceinline__ float query_margin(float bf16_err_norm) {
    return 2.0f * (bf16_err_norm * (1.0f + 0.00390625f) + 0.0001220703125f);
}
// worst case of query_margin (||bf16(q)-q|| <= 2^-8 ||q||): used where no per-query value exists
constexpr float kBf16QueryMargin = 0.0082f;

// Threshold join modes (selfjoin.cu): the self-join's upper triangle, a rectangle between two disjoint row sets of one
// collection (pairs as (lower id, higher id)), and a join across two collections with the query rows from the left or the
// right collection (pairs as (left id, right id)).
enum JoinMode : int { kJoinTriangle = 0, kJoinRectangle = 1, kJoinCrossLeft = 2, kJoinCrossRight = 3 };

}  // namespace rvo
