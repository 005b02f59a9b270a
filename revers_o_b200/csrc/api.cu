// C-ABI entry points (include/revers_o_b200.h) and the search driver that sequences the kernels.
#include <stdarg.h>
#include <string.h>
#include <math.h>
#include <mutex>

#include "common.cuh"
#include "scan_tc.cuh"
#include "select.cuh"
#include "prep_scan_small.cuh"

namespace rvo {

extern bool g_force_cuda_core_pool;
extern std::atomic<long long> g_exchange_timeout_ms;
extern std::atomic<long long> g_merge_trace;
extern void* g_pool_trace;
static std::atomic<long long> opt_select_trace{0};
size_t selfjoin_workspace_bytes(int d, long long cand_cap);
int launch_selfjoin(const uint16_t* qdb, long long q_row_lo, long long q_row_hi, long long q_id_offset, const uint16_t* db,
                    long long n_rows, int d, float threshold, long long id_offset, long long cand_cap, long long* out_pairs,
                    float* out_scores, long long out_cap, int* parent, unsigned long long* out_count, int* out_overflowed, int mode,
                    bool append, void* ws, size_t ws_bytes, int sm_count, cudaStream_t stream);
int launch_components_flatten(int* parent, int n, int* labels, int sm_count, cudaStream_t stream);
int launch_components_merge(int* parent, const int* labels_src, int n, int sm_count, cudaStream_t stream);
int launch_knn_intake(const uint16_t* qdb, long long row0, const int64_t* rows, int nq, int n_pad_rows, int d_pad, uint16_t* qb,
                      float* qn, float* margin, void* zero_base, size_t zero_bytes, cudaStream_t stream);
int launch_knn_exclude(const int64_t* ids, const float* scores, const int32_t* counts, int nq, int k, long long row0,
                       const int64_t* rows, long long q_id_offset, int64_t* out_ids, float* out_scores, int32_t* out_counts,
                       cudaStream_t stream);
size_t kmeans_update_workspace_bytes(long long n, int C);
int launch_kmeans_update(const uint16_t* db, long long row_lo, long long n, int d, int d_pad, const int64_t* ids, long long id_offset,
                         int C, const int32_t* prev, int32_t* labels, int64_t* sums, int64_t* counts, int64_t* changed, void* ws,
                         int sm_count, cudaStream_t stream);
int launch_kmeans_finalize(const int64_t* sums, const int64_t* counts, int C, int d, float* out, int32_t* empty, int64_t* n_empty,
                           cudaStream_t stream);
static thread_local char g_err[512] = "";
std::atomic<long long> g_launches{0};
std::atomic<long long> g_chain_trace{0};
std::atomic<long long> g_use_pdl{0};   // see common.cuh launch_pdl

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static std::atomic<long long> opt_force_path{0}, opt_m_sub{0}, opt_cand_cap{32768}, opt_final_ratio{48}, opt_time_scan{0}, opt_hot{1}, opt_seed_max{1},
    opt_knn_block{8192};
static cudaEvent_t g_ev0 = nullptr, g_ev1 = nullptr;
static bool g_ev_valid = false;

static int scan_timer(bool start, cudaStream_t stream) {
    if (!opt_time_scan.load()) return RVO_OK;
    if (!g_ev0) {
        RVO_CUDA(cudaEventCreate(&g_ev0));
        RVO_CUDA(cudaEventCreate(&g_ev1));
    }
    RVO_CUDA(cudaEventRecord(start ? g_ev0 : g_ev1, stream));
    if (!start) g_ev_valid = true;
    return RVO_OK;
}

// Every exported entry point makes the device that owns its pointers current for the duration of the call and restores the
// caller's device on return (a single process may drive several GPUs, B200VectorDB(devices=[...]); torch tracks its own
// current device per thread and must not find it changed).
struct DeviceGuard {
    int prev = -1;
    DeviceGuard() {
        if (cudaGetDevice(&prev) != cudaSuccess) {
            prev = -1;
            cudaGetLastError();
        }
    }
    ~DeviceGuard() {
        int cur = -1;
        if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
    }
};

// per-device properties, filled once per device (Gradio worker threads may race here: std::call_once)
constexpr int kMaxDevices = 64;
static std::once_flag g_prop_once[kMaxDevices];
static int g_prop_sm[kMaxDevices], g_prop_major[kMaxDevices];

int select_device_of(const void* dev_ptr, int* sm_count) {
    cudaPointerAttributes at;
    cudaError_t e = cudaPointerGetAttributes(&at, dev_ptr);
    if (e != cudaSuccess) {
        set_error("cudaPointerGetAttributes failed: %s", cudaGetErrorString(e));
        cudaGetLastError();
        return RVO_E_NO_DEVICE;
    }
    if (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) {
        set_error("pointer %p is not device memory (type %d)", dev_ptr, (int)at.type);
        return RVO_E_INVALID;
    }
    if (at.device < 0 || at.device >= kMaxDevices) {
        set_error("device ordinal %d out of range", at.device);
        return RVO_E_NO_DEVICE;
    }
    RVO_CUDA(cudaSetDevice(at.device));
    const int dev = at.device;
    std::call_once(g_prop_once[dev], [dev]() {
        int sm = 0, major = 0;
        if (cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) {
            cudaGetLastError();
            sm = 0;
            major = 0;
        }
        g_prop_sm[dev] = sm;
        g_prop_major[dev] = major;
    });
    if (g_prop_major[dev] != 10) {
        set_error("device %d is sm_%d0, this library is built for sm_100a (B200) only", dev, g_prop_major[dev]);
        return RVO_E_NO_DEVICE;
    }
    if (sm_count) *sm_count = g_prop_sm[dev];
    return RVO_OK;
}

__global__ void fill_outputs_kernel(int64_t* ids, float* scores, int32_t* counts, long long n, int nq) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        ids[i] = -1;
        scores[i] = -__int_as_float(0x7f800000);
    }
    if (i < nq) counts[i] = 0;
}

__global__ void init_tau_kernel(float* tau, int nq, int nq_pad, float floor_t, int copies) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq_pad * copies) return;
    tau[i] = (i % nq_pad) < nq ? floor_t : __int_as_float(0x7f800000);
}

static int next_pow2_host(int x) {
    int p = 2;
    while (p < x) p <<= 1;
    return p;
}

// ---- search plan (shared by the workspace query and the driver) --------------------------------
constexpr long long kSeedRows = 16384;  // rows of the DENSE threshold-seeding sample

constexpr long long kSmallDenseRows = 131072;   // Q <= 4: shards up to this many rows keep EVERY score (<= 512 KB per query, L2)
constexpr int kSmallSegCap = 4096;              // Q <= 4, larger shards: capacity of one of the 16 survivor sub-lists per query

struct SearchPlan {
    bool small;
    long long pair_stride, n_cols;   // small path: row pairs visited by the DENSE pass (1 = every row) and its columns
    unsigned long long* tau_key;     // small path, sampled: k-th best ordering key of the sample per query
    int d_pad, K2, cap, n_levels;
    long long level_stride[8];       // super-tile stride of each FILTER level (last one is 1)
    long long seed_stride, seed_cols;
    TcPlan tc;
    // workspace slices
    float* qn;
    uint16_t* qb;
    float* tau;       // [n_levels+1][nq_pad]
    float* tau_hot;   // [nq_pad] hot threshold of the LAST level (scan_tc.cuh kHotSplit)
    int hot_rank;     // rank (in the sample the last threshold comes from) whose score becomes tau_hot
    float* margin;    // [nq_pad] per-query admission margin (common.cuh query_margin)
    int* cnt;         // [n_levels+1][nq_pad]
    unsigned long long* cand;
    float* dense;
    long long dense_ld;
    size_t cnt_bytes;             // candidate counters (multiple of 16 bytes), cleared by the normalise launch
    size_t bytes;
};

static int make_plan(long long n_rows, int d, int nq, int k, int path, void* ws, size_t ws_bytes, SearchPlan* sp) {
    memset(sp, 0, sizeof(*sp));
    sp->d_pad = (d + kBlockK - 1) / kBlockK * kBlockK;
    const long long force = path != RVO_PATH_AUTO ? (long long)path : opt_force_path.load();
    sp->small = (force == RVO_PATH_SMALL || force == RVO_PATH_DENSE) ||
                (force != RVO_PATH_TENSOR && nq <= RVO_SMALL_Q && scan_small_supports(sp->d_pad));
    if (sp->small && nq > RVO_SMALL_Q) {
        set_error("the fp32 scan (path %lld) needs nq <= %d", force, RVO_SMALL_Q);
        return RVO_E_INVALID;
    }
    if (sp->small && !scan_small_supports(sp->d_pad)) {
        set_error("the fp32 scan (path %lld) does not cover d = %d", force, d);
        return RVO_E_UNSUPPORTED;
    }
    Arena ar(ws, ws_bytes);
    if (sp->small) {
        // DENSE pass over every row (small shard, or path DENSE: the unconditional exact route) or over a strided sample whose
        // k-th best key then filters the full scan: expected survivors = k * n / sample <= ~8k per query
        sp->K2 = next_pow2_host((2 * k > k + 64) ? 2 * k : k + 64);
        if (sp->K2 > 1024) sp->K2 = 1024;
        const long long npairs = (n_rows + 1) / 2;
        sp->pair_stride = 1;
        if (n_rows > kSmallDenseRows && force != RVO_PATH_DENSE) {
            long long sample = n_rows / 96;
            if (sample < 16384) sample = 16384;       // <= 16k columns: the selection kernel keeps them in registers
            const long long by_k = (long long)k * (n_rows / 8192 + 1);
            if (sample < by_k) sample = by_k;
            const long long sample_pairs = (sample + 1) / 2;
            sp->pair_stride = (npairs + sample_pairs - 1) / sample_pairs;     // rounded up: at most `sample` columns
            if (sp->pair_stride < 1) sp->pair_stride = 1;
        }
        sp->n_cols = 2 * ((npairs + sp->pair_stride - 1) / sp->pair_stride);
        sp->dense_ld = (sp->n_cols + 63) / 64 * 64;
        if (sp->dense_ld < 64) sp->dense_ld = 64;
        sp->qn = ar.take<float>((size_t)RVO_SMALL_Q * sp->d_pad, 1024);
        sp->dense = ar.take<float>((size_t)nq * (size_t)sp->dense_ld);
        if (sp->pair_stride > 1) {
            sp->cap = kSmallSegCap;
            sp->tau_key = ar.take<unsigned long long>(RVO_SMALL_Q);
            sp->cnt_bytes = align_up((size_t)RVO_SMALL_Q * kCandSplit * sizeof(int), 16);
            sp->cnt = (int*)ar.take<char>(sp->cnt_bytes, 256);
            sp->cand = ar.take<unsigned long long>((size_t)nq * kCandSplit * (size_t)sp->cap);
        }
    } else {
        int rc = plan_scan_tc(nq, sp->d_pad, (int)opt_m_sub.load(), &sp->tc);
        if (rc) return rc;
        const int nq_pad = sp->tc.nq_pad;
        const long long T = (long long)kBlockM * sp->tc.m_sub;
        const long long supers = (n_rows + T - 1) / T;
        sp->K2 = next_pow2_host((2 * k > k + 64) ? 2 * k : k + 64);
        if (sp->K2 > 1024) sp->K2 = 1024;
        long long cap = opt_cand_cap.load() / kCandSplit;  // per sub-list
        if (cap < 64) cap = 64;
        sp->cap = (int)cap;
        // levels: DENSE seed over ~16k rows (every seed_stride-th super-tile), then geometric FILTER samples,
        // then the full scan.  Any sample gives a valid threshold (k-th best of a subset <= k-th best overall).
        if (supers * T <= kSeedRows) {
            sp->seed_stride = 1;
            sp->n_levels = 0;
        } else {
            // seed sample: a fixed 16k rows whatever the shard size.  Survivors per scanned row = Q * k / seed_rows, so a
            // smaller seed on a smaller shard (tried: n/32) makes the candidate appends, not HBM, the limit of the scan
            // (1M x 1024 over 8 GPUs: scan 54 -> 116 us per shard with a 4k-row seed).
            const long long seed_rows = kSeedRows;
            sp->seed_stride = supers / ((seed_rows + T - 1) / T);
            if (sp->seed_stride < 1) sp->seed_stride = 1;
            long long ratio = opt_final_ratio.load();
            if (ratio < 2) ratio = 2;
            long long sizes[8];
            int ns = 0;
            for (long long s = n_rows / ratio; s >= 2 * kSeedRows && ns < 6; s /= 64) sizes[ns++] = s;
            int L = 0;
            for (int i = ns - 1; i >= 0; --i) {
                const long long r = supers / ((sizes[i] + T - 1) / T);
                if (r <= 1 || r >= sp->seed_stride) continue;
                sp->level_stride[L++] = r;
            }
            sp->level_stride[L] = 1;
            sp->n_levels = L + 1;
        }
        sp->seed_cols = scan_tc_sample_rows(n_rows, sp->tc, sp->seed_stride);
        sp->qb = ar.take<uint16_t>((size_t)nq_pad * sp->d_pad, 1024);
        sp->cnt_bytes = align_up((size_t)(sp->n_levels + 1) * nq_pad * kCandSegs * sizeof(int), 16);
        sp->cnt = (int*)ar.take<char>(sp->cnt_bytes, 256);
        sp->qn = ar.take<float>((size_t)nq_pad * sp->d_pad, 1024);
        sp->tau = ar.take<float>((size_t)(sp->n_levels + 1) * nq_pad);
        sp->margin = ar.take<float>((size_t)nq_pad);
        sp->tau_hot = ar.take<float>((size_t)nq_pad);
        {
            // hot threshold: aim at ~kHotTarget rows of the shard above it.  The last threshold level sees `prev` rows (the seed
            // sample, or the previous FILTER level's tile sample): the r-th best of that sample has about r * n_rows / prev rows of
            // the shard above it; r >= 10 keeps the relative spread of that count (1/sqrt(r)) small enough that fewer than k hot
            // rows (-> general path) stays a < 1e-3 event per query.
            constexpr double kHotTarget = 600.0;
            long long prev = sp->seed_cols;
            if (sp->n_levels >= 2) {
                const long long st = sp->level_stride[sp->n_levels - 2];
                prev = (supers + st - 1) / st * T;
            }
            long long r = (long long)(kHotTarget * (double)prev / (double)(n_rows > 0 ? n_rows : 1) + 0.999);
            if (r < 10) r = 10;
            if (r > k) r = k;
            sp->hot_rank = (int)r;
        }
        sp->dense_ld = (sp->seed_cols + 63) / 64 * 64;
        sp->dense = ar.take<float>((size_t)nq_pad * (size_t)sp->dense_ld);
        if (sp->n_levels > 0) sp->cand = ar.take<unsigned long long>((size_t)nq_pad * kCandSegs * (size_t)sp->cap);
    }
    sp->bytes = ar.off + 1024;
    if (ws && !ar.ok()) {
        set_error("search workspace too small: %zu bytes given, %zu needed", ws_bytes, sp->bytes);
        return RVO_E_WORKSPACE;
    }
    return RVO_OK;
}

static int prep_queries(const SearchPlan& sp, const float* queries, int nq, int d, cudaStream_t stream) {
    // one launch: normalise, zero the padding rows of the query operand, clear the candidate counters (no memset node)
    return launch_normalize_rows(queries, nq, d, d, sp.qb, sp.d_pad, -1, sp.qn, sp.d_pad, stream, sp.margin, sp.tc.nq_pad,
                                 (void*)sp.cnt, sp.cnt_bytes);
}

// Stored rows as the queries of a search (rvo_knn_join): query q is row (rows ? rows[q] : row0 + q) of the tiled storage qdb,
// on the searched rows' device.  It replaces the normalise launch: knn.cu's intake writes the query operand, its fp32 copy,
// the margins and the cleared counters in one launch.
struct StoredQueries {
    const uint16_t* qdb;
    long long row0;
    const int64_t* rows;
};

}  // namespace rvo

using namespace rvo;

extern "C" {

int rvo_version(void) { return 100; }

const char* rvo_last_error(void) { return g_err; }

int64_t rvo_kernel_launch_count(void) { return (int64_t)g_launches.load(); }

float rvo_last_scan_ms(void) {
    if (!g_ev_valid) return -1.f;
    float ms = -1.f;
    if (cudaEventSynchronize(g_ev1) != cudaSuccess || cudaEventElapsedTime(&ms, g_ev0, g_ev1) != cudaSuccess) {
        cudaGetLastError();
        return -1.f;
    }
    return ms;
}

int rvo_device_sm_count(const void* dev_ptr) {
    DeviceGuard device_guard;
    int sm = 0;
    int rc = select_device_of(dev_ptr, &sm);
    return rc ? rc : sm;
}

int rvo_set_option(const char* name, int64_t value) {
    if (!name) return RVO_E_INVALID;
    if (!strcmp(name, "force_path")) opt_force_path = value;
    else if (!strcmp(name, "m_sub")) opt_m_sub = value;
    else if (!strcmp(name, "cand_cap")) opt_cand_cap = value;
    else if (!strcmp(name, "final_ratio")) opt_final_ratio = value;
    else if (!strcmp(name, "time_scan")) opt_time_scan = value;
    else if (!strcmp(name, "hot")) opt_hot = value;
    else if (!strcmp(name, "seed_max")) opt_seed_max = value;
    else if (!strcmp(name, "knn_block")) {
        RVO_REQUIRE(value >= 256 && value <= 16384, "option knn_block=%lld outside 256..16384", (long long)value);
        opt_knn_block = value;
    }
    else if (!strcmp(name, "exchange_timeout_ms")) g_exchange_timeout_ms = value > 0 ? value : 1;
    else if (!strcmp(name, "merge_trace")) g_merge_trace = value;
    else if (!strcmp(name, "pool_path")) g_force_cuda_core_pool = value == 1;
    else if (!strcmp(name, "pdl")) g_use_pdl = value;
    else if (!strcmp(name, "select_trace")) opt_select_trace = value;
    else if (!strcmp(name, "chain_trace")) g_chain_trace = value;
    else if (!strcmp(name, "pool_trace")) g_pool_trace = (void*)(uintptr_t)value;
    else {
        set_error("unknown option '%s'", name);
        return RVO_E_INVALID;
    }
    return RVO_OK;
}

size_t rvo_db_bytes(int64_t n_rows, int32_t d) {
    if (n_rows < 0 || d <= 0) return 0;
    const size_t d_pad = (size_t)(d + kBlockK - 1) / kBlockK * kBlockK;
    return (size_t)((n_rows + kTileRows - 1) / kTileRows) * kTileRows * d_pad * 2;
}

int rvo_normalize_rows(const float* src, int64_t n, int32_t d, int64_t src_ld, uint16_t* dst_bf16, int64_t dst_ld,
                       int64_t tiled_row0, float* dst_f32, void* stream) {
    DeviceGuard device_guard;
    RVO_REQUIRE(src && (dst_bf16 || dst_f32), "normalize_rows: null pointer");
    RVO_REQUIRE(n >= 0 && d > 0 && src_ld >= d, "normalize_rows: bad shape n=%lld d=%d ld=%lld", (long long)n, d,
                (long long)src_ld);
    RVO_REQUIRE(!dst_bf16 || (dst_ld >= d && dst_ld % 8 == 0), "normalize_rows: dst_ld=%lld must be >= d and %% 8 == 0",
                (long long)dst_ld);
    int rc = select_device_of(src, nullptr);
    if (rc) return rc;
    RVO_REQUIRE(tiled_row0 < 0 || !dst_bf16 || dst_ld % kBlockK == 0, "normalize_rows: tiled storage needs d_pad %% 64 == 0");
    return launch_normalize_rows(src, n, d, src_ld, dst_bf16, dst_ld, tiled_row0, dst_f32, d, (cudaStream_t)stream);
}

size_t rvo_mask_pool_workspace_bytes(int32_t B, int32_t M, int32_t P, int32_t D) {
    return mask_pool_workspace_bytes(B, M, P, D);
}

int rvo_mask_pool(const uint16_t* feats, int32_t feat_dtype, const uint8_t* masks, int32_t B, int32_t M, int32_t P, int32_t D,
                  int32_t max_regions, float* out, int32_t* out_counts, int32_t* out_src, int32_t* out_total,
                  void* workspace, size_t workspace_bytes, void* stream) {
    DeviceGuard device_guard;
    RVO_REQUIRE(feats && masks && out && out_counts && out_total && workspace, "mask_pool: null pointer");
    RVO_REQUIRE(feat_dtype == RVO_DTYPE_BF16 || feat_dtype == RVO_DTYPE_F16, "mask_pool: feat_dtype %d (bf16 = 0, fp16 = 1)", feat_dtype);
    RVO_REQUIRE(B > 0 && M > 0 && P > 0 && D > 0, "mask_pool: bad shape B=%d M=%d P=%d D=%d", B, M, P, D);
    RVO_REQUIRE(((uintptr_t)feats & 15) == 0 && ((uintptr_t)out & 15) == 0 && ((uintptr_t)masks & 3) == 0,
                "mask_pool: feats/out must be 16-byte aligned, masks 4-byte aligned");
    int sm = 0;
    int rc = select_device_of(feats, &sm);
    if (rc) return rc;
    return launch_mask_pool(feats, masks, B, M, P, D, max_regions, out, out_counts, out_src, out_total, workspace,
                            workspace_bytes, sm, (cudaStream_t)stream, nullptr, 0, feat_dtype == RVO_DTYPE_F16);
}

int rvo_mask_pool_to_db(const uint16_t* feats, int32_t feat_dtype, const uint8_t* masks, int32_t B, int32_t M, int32_t P, int32_t D,
                        int32_t max_regions, uint16_t* db, int64_t db_row0, float* out_f32, int32_t* out_counts,
                        int32_t* out_src, int32_t* out_total, void* workspace, size_t workspace_bytes, void* stream) {
    DeviceGuard device_guard;
    RVO_REQUIRE(feats && masks && db && out_counts && out_total && workspace, "mask_pool_to_db: null pointer");
    RVO_REQUIRE(feat_dtype == RVO_DTYPE_BF16 || feat_dtype == RVO_DTYPE_F16, "mask_pool_to_db: feat_dtype %d (bf16 = 0, fp16 = 1)", feat_dtype);
    RVO_REQUIRE(B > 0 && M > 0 && P > 0 && D > 0 && db_row0 >= 0, "mask_pool_to_db: bad shape B=%d M=%d P=%d D=%d row0=%lld", B,
                M, P, D, (long long)db_row0);
    RVO_REQUIRE(((uintptr_t)feats & 15) == 0 && ((uintptr_t)db & 15) == 0 && ((uintptr_t)masks & 3) == 0 &&
                    (!out_f32 || ((uintptr_t)out_f32 & 15) == 0),
                "mask_pool_to_db: feats/db/out must be 16-byte aligned, masks 4-byte aligned");
    int sm = 0;
    int rc = select_device_of(feats, &sm);
    if (rc) return rc;
    if (D % 128 != 0) {
        set_error("mask_pool_to_db: D=%d is outside the fused kernel (D %% 128 != 0): use rvo_mask_pool + rvo_normalize_rows", D);
        return RVO_E_UNSUPPORTED;
    }
    rc = launch_mask_pool(feats, masks, B, M, P, D, max_regions, out_f32, out_counts, out_src, out_total, workspace,
                          workspace_bytes, sm, (cudaStream_t)stream, db, db_row0, feat_dtype == RVO_DTYPE_F16);
    if (rc == RVO_E_UNSUPPORTED)
        set_error("mask_pool_to_db: shape B=%d M=%d P=%d D=%d is outside the fused kernel: use rvo_mask_pool + rvo_normalize_rows",
                  B, M, P, D);
    return rc;
}

size_t rvo_search_workspace_bytes(int64_t n_rows, int32_t d, int32_t nq, int32_t k) {
    return rvo_search_workspace_bytes_ex(n_rows, d, nq, k, RVO_PATH_AUTO);
}

size_t rvo_search_workspace_bytes_ex(int64_t n_rows, int32_t d, int32_t nq, int32_t k, int32_t path) {
    if (n_rows < 0 || d <= 0 || nq <= 0 || k <= 0 || k > RVO_MAX_K || path < RVO_PATH_AUTO || path > RVO_PATH_DENSE) return 0;
    SearchPlan sp;
    if (make_plan(n_rows, d, nq, k, path, nullptr, 0, &sp)) return 0;
    return sp.bytes;
}

static int search_impl(const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad_in, const float* queries, int32_t nq,
                       int32_t k, float score_threshold, int64_t id_offset, int64_t* out_ids, float* out_scores,
                       int32_t* out_counts, void* workspace, size_t workspace_bytes, void* stream_, const PushArgs* push,
                       int path = RVO_PATH_AUTO, const StoredQueries* stored = nullptr) {
    DeviceGuard device_guard;
    RVO_REQUIRE(path >= RVO_PATH_AUTO && path <= RVO_PATH_DENSE, "search_topk: path %d (0 auto, 1 fp32 scan, 2 tcgen05, 3 dense fp32)", path);
    cudaStream_t stream = (cudaStream_t)stream_;
    RVO_REQUIRE((queries || stored) && out_ids && out_scores && out_counts && workspace, "search_topk: null pointer");
    RVO_REQUIRE(n_rows >= 0 && d > 0 && nq > 0, "search_topk: bad shape n_rows=%lld d=%d nq=%d", (long long)n_rows, d, nq);
    RVO_REQUIRE(k >= 1 && k <= RVO_MAX_K, "search_topk: k=%d outside 1..%d", k, RVO_MAX_K);
    RVO_REQUIRE(n_rows == 0 || db, "search_topk: null db");
    RVO_REQUIRE(d_pad_in == (d + kBlockK - 1) / kBlockK * kBlockK, "search_topk: d_pad=%lld must be d rounded up to 64",
                (long long)d_pad_in);
    RVO_REQUIRE(((uintptr_t)db & 15) == 0 && ((uintptr_t)workspace & 1023) == 0 && ((uintptr_t)queries & 3) == 0,
                "search_topk: db must be 16-byte and workspace 1024-byte aligned");
    RVO_REQUIRE(n_rows < (1ll << 31), "search_topk: shard of %lld rows too large, shard the DB", (long long)n_rows);
    int sm = 0;
    // the device comes from the workspace (always device memory); `queries` and the outputs may be pinned host memory
    int rc = select_device_of(workspace, &sm);
    if (rc) return rc;

    if (push && n_rows == 0) {
        set_error("search_topk_push: the fused exchange needs a non-empty shard (use the all-gather path)");
        return RVO_E_UNSUPPORTED;
    }
    if (n_rows == 0) {
        const long long n = (long long)nq * k;
        fill_outputs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(out_ids, out_scores, out_counts, n, nq);
        RVO_LAUNCHED();
        return RVO_OK;
    }

    SearchPlan sp;
    rc = make_plan(n_rows, d, nq, k, path, workspace, workspace_bytes, &sp);
    if (rc) return rc;
    if (push && sp.small) {
        set_error("search_topk_push: the fused exchange serves the tcgen05 path only");
        return RVO_E_UNSUPPORTED;
    }

    FinalArgs fa;
    memset(&fa, 0, sizeof(fa));
    fa.k = k;
    fa.K2 = sp.K2;
    fa.score_threshold = score_threshold;
    fa.db = db;
    fa.d_pad = sp.d_pad;
    fa.qn = sp.qn;
    fa.qn_ld = sp.d_pad;
    fa.id_offset = id_offset;
    fa.out_ids = out_ids;
    fa.out_scores = out_scores;
    fa.out_counts = out_counts;
    if (push) fa.push = *push;

    if (sp.small) {
        // The reference's own operating point (Q = 1, core_system.py:657): exact fp32 scores on CUDA cores.
        //   small shard (or path DENSE): [scan: normalise + every score] -> [exact top-k of the dense row]          2 launches
        //   large shard: [scan of a row sample] -> [k-th best key of the sample] -> [full scan, survivors only] -> [exact top-k]
        // Scores are final (no re-score); the dense scores of a large shard never reach HBM.
        SmallScanArgs sa;
        memset(&sa, 0, sizeof(sa));
        sa.db = (const uint4*)db;
        sa.n_rows = n_rows;
        sa.nk = sp.d_pad / kTileCols;
        sa.nchunks = sp.d_pad / 8;
        sa.nq = nq;
        sa.d = d;
        sa.q = queries;
        sa.q_ld = d;
        sa.qn_out = sp.qn;
        sa.qn_ld = sp.d_pad;
        sa.out = sp.dense;
        sa.out_ld = sp.dense_ld;
        sa.pair_stride = sp.pair_stride;
        const bool sampled = sp.pair_stride > 1;
        if (sampled) {
            sa.zero_base = (uint4*)sp.cnt;
            sa.zero_u4 = (long long)(sp.cnt_bytes / 16);
        }
        if (stored) {
            // the fp32 scan reads the stored rows' fp32 copy instead of normalising raw queries; the intake also clears the
            // FILTER pass's counters, which only the normalising scan would otherwise clear
            rc = launch_knn_intake(stored->qdb, stored->row0, stored->rows, nq, RVO_SMALL_Q, sp.d_pad, nullptr, sp.qn, nullptr,
                                   (void*)sp.cnt, sp.cnt_bytes, stream);
            if (rc) return rc;
            sa.q = sp.qn;
            sa.q_ld = sp.d_pad;
        }
        if (!sampled && (rc = scan_timer(true, stream))) return rc;
        rc = launch_scan_small(sa, true, !stored, sm, stream);
        if (rc) return rc;
        if (!sampled && (rc = scan_timer(false, stream))) return rc;
        DenseTopkArgs da;
        memset(&da, 0, sizeof(da));
        da.dense = sp.dense;
        da.dense_ld = sp.dense_ld;
        da.n_cols = sp.n_cols;
        da.n_rows = n_rows;
        da.pair_stride = sp.pair_stride;
        da.k = k;
        da.trace = (unsigned long long*)(uintptr_t)opt_select_trace.load();
        fa.rescore = 0;
        fa.margin = nullptr;
        if (!sampled) return launch_dense_topk(da, &fa, nq, stream);
        da.tau_key_out = sp.tau_key;
        rc = launch_dense_topk(da, nullptr, nq, stream);
        if (rc) return rc;
        sa.q = sp.qn;                    // normalised by the first pass
        sa.q_ld = sp.d_pad;
        sa.tau_key = sp.tau_key;
        sa.cand = sp.cand;
        sa.cnt = sp.cnt;
        sa.nseg = kCandSplit;
        sa.cap = sp.cap;
        if ((rc = scan_timer(true, stream))) return rc;
        rc = launch_scan_small(sa, false, false, sm, stream);
        if (rc) return rc;
        if ((rc = scan_timer(false, stream))) return rc;
        SelectArgs sl;
        memset(&sl, 0, sizeof(sl));
        sl.nq = nq;
        sl.keys = sp.cand;
        sl.cnt = sp.cnt;
        sl.nseg = kCandSplit;
        sl.cap = sp.cap;
        sl.K = sp.K2;
        sl.score_floor = score_threshold;
        return launch_select_final(sl, fa, nq, stream);     // a sub-list that overflowed flags the query (-1): path DENSE serves it
    }
    rc = stored ? launch_knn_intake(stored->qdb, stored->row0, stored->rows, nq, sp.tc.nq_pad, sp.d_pad, sp.qb, sp.qn, sp.margin,
                                    (void*)sp.cnt, sp.cnt_bytes, stream)
                : prep_queries(sp, queries, nq, d, stream);
    if (rc) return rc;

    const int nq_pad = sp.tc.nq_pad;
    fa.rescore = 1;
    fa.margin = sp.margin;

    SelectArgs sa;
    memset(&sa, 0, sizeof(sa));
    sa.nq = nq;
    sa.margin = sp.margin;
    sa.score_floor = score_threshold;   // nothing below score_threshold - margin is ever queued (-inf stays -inf)
    sa.tau_k = k;

    // level 0: DENSE pass over the seed sample (or the whole shard when it is small)
    // When the sample only seeds a threshold through seed_tau_kernel, the scan writes one maximum per 32 sample rows instead of
    // every score (kModeDenseMax): 32x less to write and to read back, same guarantee.
    const bool seed_max = sp.n_levels > 0 && k <= kSeedTauMaxK && opt_seed_max.load() != 0;
    rc = launch_scan_tc(seed_max ? kModeDenseMax : kModeDense, db, n_rows, sp.seed_stride, sp.d_pad, sp.qb, sp.tc, nullptr, nullptr,
                        nullptr, 0, sp.dense, sp.dense_ld, sm, stream);
    if (rc) return rc;
    sa.dense = sp.dense;
    sa.dense_ld = sp.dense_ld;
    sa.n_dense = sp.seed_cols;
    if (sp.n_levels == 0) {
        // the sample IS the shard (dense column == row): exact candidates by tensor score, fp32 re-score, final order
        sa.K = sp.K2;
        return launch_select_final(sa, fa, nq, stream);
    }
    sa.K = k;
    sa.tau_out = sp.tau;
    const bool seed_is_last = sp.n_levels == 1;    // the seed threshold feeds the full scan directly: it also proposes tau_hot
    if (k <= kSeedTauMaxK)   // one pass + one 512-key sort: k-th largest of the per-thread maxima (select.cuh)
        rc = launch_seed_tau(sp.dense, sp.dense_ld, seed_max ? sp.seed_cols / 32 : sp.seed_cols, nq, nq_pad, k, sp.margin,
                             score_threshold, sp.tau, stream,
                             sp.hot_rank, seed_is_last ? sp.tau_hot : nullptr);
    else {
        sa.hot_rank = sp.hot_rank;
        sa.tau_hot_out = seed_is_last ? sp.tau_hot : nullptr;
        rc = launch_select(sa, nq_pad, stream);
    }
    if (rc) return rc;

    // FILTER levels: each tightens tau on a larger tile sample; the last one scans every row
    const bool use_hot = opt_hot.load() != 0;
    for (int L = 0; L < sp.n_levels; ++L) {
        const bool last = L == sp.n_levels - 1;
        int* cnt = sp.cnt + (size_t)L * nq_pad * kCandSegs;
        const float* tau_in = sp.tau + (size_t)L * nq_pad;
        if (last && (rc = scan_timer(true, stream))) return rc;
        rc = launch_scan_tc(kModeFilter, db, n_rows, sp.level_stride[L], sp.d_pad, sp.qb, sp.tc, tau_in, sp.cand, cnt, sp.cap,
                            nullptr, 0, sm, stream, last && use_hot && opt_hot.load() != 2 ? sp.tau_hot : nullptr, kCandSegs);
        if (rc) return rc;
        if (last && (rc = scan_timer(false, stream))) return rc;
        memset(&sa, 0, sizeof(sa));
        sa.nq = nq;
        sa.keys = sp.cand;
        sa.range_lo = tau_in;
        sa.cnt = cnt;
        sa.nseg = kCandSegs;
        sa.cap = sp.cap;
        sa.margin = sp.margin;
        sa.score_floor = score_threshold;
        if (!last) {
            sa.K = k;
            sa.tau_out = sp.tau + (size_t)(L + 1) * nq_pad;
            sa.tau_prev = tau_in;
            sa.tau_k = k;
            if (L == sp.n_levels - 2) {   // this level's threshold feeds the full scan: propose tau_hot as well
                sa.hot_rank = sp.hot_rank;
                sa.tau_hot_out = sp.tau_hot;
            }
            rc = launch_select(sa, nq_pad, stream);
            if (rc) return rc;
        } else {
            // last level: exact candidate selection fused with the fp32 re-score and the final ordering
            sa.K = sp.K2;
            sa.trace = (unsigned long long*)(uintptr_t)opt_select_trace.load();
            if (use_hot) {
                sa.tau_hot = sp.tau_hot;
                sa.hot_seg0 = kCandSplit;
                sa.hot_nseg = kHotSplit;
            }
            rc = launch_select_final(sa, fa, nq, stream);
            if (rc) return rc;
        }
    }
    return RVO_OK;
}

int rvo_search_topk(const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad, const float* queries, int32_t nq,
                    int32_t k, float score_threshold, int64_t id_offset, int64_t* out_ids, float* out_scores,
                    int32_t* out_counts, void* workspace, size_t workspace_bytes, void* stream) {
    return search_impl(db, n_rows, d, d_pad, queries, nq, k, score_threshold, id_offset, out_ids, out_scores, out_counts,
                       workspace, workspace_bytes, stream, nullptr);
}

int rvo_search_topk_ex(const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad, const float* queries, int32_t nq,
                       int32_t k, float score_threshold, int64_t id_offset, int32_t path, int64_t* out_ids, float* out_scores,
                       int32_t* out_counts, void* workspace, size_t workspace_bytes, void* stream) {
    return search_impl(db, n_rows, d, d_pad, queries, nq, k, score_threshold, id_offset, out_ids, out_scores, out_counts,
                       workspace, workspace_bytes, stream, nullptr, path);
}

// ---- k-nearest-neighbour join (knn.cu) --------------------------------------------------------------------------------
// Query blocks of option "knn_block" stored rows (default 8192), each one K2 search.  The block's candidate lists dominate the
// workspace (3.3 GB at 8192 rows, d = 1024).  Measured on the 2M x 1024 self kNN at k = 10 (scripts/bench_knn_join.py, DESIGN.md
// §4): larger blocks stream each DB tile for more queries; 8192 rows beat 4096 by ~3 % for twice the workspace.

struct KnnLayout {
    int block, kk, search_path;
    size_t search_bytes, lists_off, scores_off, counts_off, bytes;
};

// Workspace of rvo_knn_join: one block's search workspace, then (self mode) the block's [block][k+1] lists before exclusion.
// Sized for k + 1 lists whichever the mode, so that one size serves both.
static bool knn_layout(int64_t n_rows, int32_t d, int64_t nq, int32_t k, int32_t path, KnnLayout* L) {
    if (n_rows < 0 || d <= 0 || nq <= 0 || k <= 0 || k > RVO_MAX_K || path < RVO_PATH_AUTO || path > RVO_PATH_DENSE) return false;
    const long long block = opt_knn_block.load();
    L->block = (int)(nq < block ? nq : block);
    L->kk = k < RVO_MAX_K ? k + 1 : k;
    L->search_path = path == RVO_PATH_AUTO ? RVO_PATH_TENSOR : path;   // AUTO: tcgen05 for every block, tails of <= 4 rows too
    SearchPlan sp;
    if (make_plan(n_rows, d, L->block, L->kk, L->search_path, nullptr, 0, &sp)) return false;
    L->search_bytes = sp.bytes;
    L->lists_off = align_up(L->search_bytes, 256);
    L->scores_off = L->lists_off + align_up((size_t)L->block * L->kk * 8, 256);
    L->counts_off = L->scores_off + align_up((size_t)L->block * L->kk * 4, 256);
    L->bytes = L->counts_off + align_up((size_t)L->block * 4, 256);
    return true;
}

size_t rvo_knn_workspace_bytes(int64_t n_rows, int32_t d, int32_t nq, int32_t k, int32_t path) {
    KnnLayout L;
    return knn_layout(n_rows, d, nq, k, path, &L) ? L.bytes : 0;
}

int rvo_knn_join(const uint16_t* qdb, int64_t q_row_lo, int64_t q_row_hi, const int64_t* q_rows, int64_t q_id_offset,
                 const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad_in, int32_t k, float score_threshold, int64_t id_offset,
                 int32_t exclude_self, int32_t path, int64_t* out_ids, float* out_scores, int32_t* out_counts, void* workspace,
                 size_t workspace_bytes, void* stream_) {
    DeviceGuard device_guard;
    cudaStream_t stream = (cudaStream_t)stream_;
    RVO_REQUIRE(qdb && out_ids && out_scores && out_counts && workspace, "knn join: null pointer");
    RVO_REQUIRE(n_rows == 0 || db, "knn join: null db");
    RVO_REQUIRE(exclude_self == 0 || exclude_self == 1, "knn join: exclude_self must be 0 or 1, got %d", (int)exclude_self);
    RVO_REQUIRE(path >= RVO_PATH_AUTO && path <= RVO_PATH_DENSE, "knn join: path %d (0 auto, 1 fp32 scan, 2 tcgen05, 3 dense fp32)",
                (int)path);
    const int k_max = exclude_self ? RVO_MAX_K - 1 : RVO_MAX_K;
    RVO_REQUIRE(k >= 1 && k <= k_max, "knn join: k=%d outside 1..%d%s", k, k_max, exclude_self ? " (self mode)" : "");
    RVO_REQUIRE(n_rows >= 0 && n_rows < (1ll << 31) && d > 0 && q_row_lo >= 0 && q_row_lo <= q_row_hi,
                "knn join: bad shape n_rows=%lld query rows [%lld,%lld)", (long long)n_rows, (long long)q_row_lo,
                (long long)q_row_hi);
    RVO_REQUIRE(d_pad_in == (d + kBlockK - 1) / kBlockK * kBlockK, "knn join: d_pad must be d rounded up to 64");
    RVO_REQUIRE(((uintptr_t)workspace & 1023) == 0 && ((uintptr_t)db & 15) == 0 && ((uintptr_t)qdb & 15) == 0 &&
                    ((uintptr_t)q_rows & 7) == 0,
                "knn join: alignment");
    const long long nq = q_row_hi - q_row_lo;
    RVO_REQUIRE((path != RVO_PATH_SMALL && path != RVO_PATH_DENSE) || (q_rows && nq <= RVO_SMALL_Q),
                "knn join: the fp32 routes (path %d) take a q_rows list of at most %d rows, got %lld rows%s", (int)path, RVO_SMALL_Q,
                nq, q_rows ? "" : " and no list");
    if (qdb == db && !q_rows)
        RVO_REQUIRE(q_row_hi <= n_rows, "knn join: query rows [%lld,%lld) outside the %lld rows of the DB", (long long)q_row_lo,
                    (long long)q_row_hi, (long long)n_rows);
    // both buffers on one device (the workspace's: search_impl takes the device from it)
    int qdev = -1, tdev = -1, wdev = -1;
    int rc = select_device_of(qdb, nullptr);
    if (rc) return rc;
    RVO_CUDA(cudaGetDevice(&qdev));
    if (n_rows > 0) {
        rc = select_device_of(db, nullptr);
        if (rc) return rc;
        RVO_CUDA(cudaGetDevice(&tdev));
        RVO_REQUIRE(qdev == tdev, "knn join: query rows on device %d, target rows on device %d", qdev, tdev);
    }
    rc = select_device_of(workspace, nullptr);
    if (rc) return rc;
    RVO_CUDA(cudaGetDevice(&wdev));
    RVO_REQUIRE(wdev == qdev, "knn join: workspace on device %d, query rows on device %d", wdev, qdev);
    if (nq == 0) return RVO_OK;
    KnnLayout L;
    if (!knn_layout(n_rows, d, nq, k, path, &L)) {
        set_error("knn join: no plan for n_rows=%lld d=%d k=%d path=%d", (long long)n_rows, d, k, (int)path);
        return RVO_E_INVALID;
    }
    if (workspace_bytes < L.bytes) {
        set_error("knn join workspace too small: %zu bytes given, %zu needed", workspace_bytes, L.bytes);
        return RVO_E_WORKSPACE;
    }
    char* ws = (char*)workspace;
    int64_t* lst_ids = (int64_t*)(ws + L.lists_off);
    float* lst_scores = (float*)(ws + L.scores_off);
    int32_t* lst_counts = (int32_t*)(ws + L.counts_off);
    const int kk = exclude_self ? k + 1 : k;
    for (long long i0 = q_row_lo; i0 < q_row_hi; i0 += L.block) {
        const int nb = (int)(q_row_hi - i0 < L.block ? q_row_hi - i0 : L.block);
        const StoredQueries sq{qdb, q_rows ? 0 : i0, q_rows ? q_rows + i0 : nullptr};
        const size_t o = (size_t)(i0 - q_row_lo) * k;
        rc = search_impl(db, n_rows, d, d_pad_in, nullptr, nb, kk, score_threshold, id_offset,
                         exclude_self ? lst_ids : out_ids + o, exclude_self ? lst_scores : out_scores + o,
                         exclude_self ? lst_counts : out_counts + (i0 - q_row_lo), workspace, L.search_bytes, stream, nullptr,
                         L.search_path, &sq);
        if (rc) return rc;
        if (exclude_self) {
            rc = launch_knn_exclude(lst_ids, lst_scores, lst_counts, nb, k, sq.row0, sq.rows, q_id_offset, out_ids + o,
                                    out_scores + o, out_counts + (i0 - q_row_lo), stream);
            if (rc) return rc;
        }
    }
    return RVO_OK;
}

int rvo_knn_exclude_self(const int64_t* ids, const float* scores, const int32_t* counts, int32_t nq, int32_t k, int64_t q_row_lo,
                         const int64_t* q_rows, int64_t q_id_offset, int64_t* out_ids, float* out_scores, int32_t* out_counts,
                         void* stream) {
    DeviceGuard device_guard;
    RVO_REQUIRE(ids && scores && counts && out_ids && out_scores && out_counts, "knn exclude self: null pointer");
    RVO_REQUIRE(nq >= 0 && k >= 1 && k < RVO_MAX_K, "knn exclude self: nq=%d k=%d (k outside 1..%d)", nq, k, RVO_MAX_K - 1);
    RVO_REQUIRE((void*)ids != (void*)out_ids && (const void*)scores != (void*)out_scores, "knn exclude self: in place");
    int rc = select_device_of(ids, nullptr);
    if (rc) return rc;
    return launch_knn_exclude(ids, scores, counts, nq, k, q_row_lo, q_rows, q_id_offset, out_ids, out_scores, out_counts,
                              (cudaStream_t)stream);
}

// ---- spherical k-means update (kmeans.cu) ------------------------------------------------------------------------------

size_t rvo_kmeans_update_workspace_bytes(int64_t n_rows, int32_t n_clusters) {
    if (n_rows < 0 || n_rows >= (1ll << 31) || n_clusters < 1 || n_clusters > RVO_KMEANS_MAX_CLUSTERS) return 0;
    return kmeans_update_workspace_bytes(n_rows, n_clusters);
}

int rvo_kmeans_update(const uint16_t* db, int64_t row_lo, int64_t row_hi, int32_t d, int64_t d_pad_in, const int64_t* ids,
                      int64_t id_offset, int32_t n_clusters, const int32_t* prev_labels, int32_t* labels, int64_t* sums,
                      int64_t* counts, int64_t* changed, void* workspace, size_t workspace_bytes, void* stream) {
    DeviceGuard device_guard;
    RVO_REQUIRE(db && ids && labels && sums && counts && changed && workspace, "kmeans update: null pointer");
    RVO_REQUIRE(n_clusters >= 1 && n_clusters <= RVO_KMEANS_MAX_CLUSTERS, "kmeans update: n_clusters=%d outside 1..%d", n_clusters,
                RVO_KMEANS_MAX_CLUSTERS);
    RVO_REQUIRE(d > 0 && row_lo >= 0 && row_lo <= row_hi && row_hi - row_lo < (1ll << 31),
                "kmeans update: bad shape d=%d rows [%lld,%lld) (fewer than 2^31 rows)", d, (long long)row_lo, (long long)row_hi);
    RVO_REQUIRE(d_pad_in == (d + kBlockK - 1) / kBlockK * kBlockK, "kmeans update: d_pad must be d rounded up to 64");
    RVO_REQUIRE(((uintptr_t)db & 15) == 0 && ((uintptr_t)sums & 7) == 0 && ((uintptr_t)counts & 7) == 0 &&
                    ((uintptr_t)changed & 7) == 0 && ((uintptr_t)workspace & 255) == 0,
                "kmeans update: alignment");
    const long long n = row_hi - row_lo;
    if (workspace_bytes < kmeans_update_workspace_bytes(n, n_clusters)) {
        set_error("kmeans update workspace too small: %zu bytes given, %zu needed", workspace_bytes,
                  kmeans_update_workspace_bytes(n, n_clusters));
        return RVO_E_WORKSPACE;
    }
    int sm = 0;
    int rc = select_device_of(db, &sm);
    if (rc) return rc;
    int ddev = -1, sdev = -1;
    RVO_CUDA(cudaGetDevice(&ddev));
    rc = select_device_of(sums, nullptr);
    if (rc) return rc;
    RVO_CUDA(cudaGetDevice(&sdev));
    RVO_REQUIRE(ddev == sdev, "kmeans update: rows on device %d, sums on device %d", ddev, sdev);
    return launch_kmeans_update(db, row_lo, n, d, (int)d_pad_in, ids, id_offset, n_clusters, prev_labels, labels, sums, counts,
                                changed, workspace, sm, (cudaStream_t)stream);
}

int rvo_kmeans_finalize(const int64_t* sums, const int64_t* counts, int32_t n_clusters, int32_t d, float* scratch_f32,
                        uint16_t* centroids, int32_t* out_empty, int64_t* n_empty, void* stream) {
    DeviceGuard device_guard;
    RVO_REQUIRE(sums && counts && scratch_f32 && centroids && out_empty && n_empty, "kmeans finalize: null pointer");
    RVO_REQUIRE(n_clusters >= 1 && n_clusters <= RVO_KMEANS_MAX_CLUSTERS && d > 0, "kmeans finalize: n_clusters=%d d=%d",
                n_clusters, d);
    RVO_REQUIRE(((uintptr_t)centroids & 15) == 0 && ((uintptr_t)n_empty & 7) == 0, "kmeans finalize: alignment");
    int rc = select_device_of(sums, nullptr);
    if (rc) return rc;
    rc = launch_kmeans_finalize(sums, counts, n_clusters, d, scratch_f32, out_empty, n_empty, (cudaStream_t)stream);
    if (rc) return rc;
    const long long d_pad = (d + kBlockK - 1) / kBlockK * kBlockK;
    return launch_normalize_rows(scratch_f32, n_clusters, d, d, centroids, d_pad, 0, nullptr, d, (cudaStream_t)stream);
}

// ---- peer-memory exchange (DESIGN.md §5) ------------------------------------------------------------------------------
// Region of one rank: [4 slot sets][world slots of slot_bytes] | flags u64 [4][world] | done u32 [4].  Slot g of set (epoch % 4)
// receives rank g's packed result blob [ids | scores | counts] of search `epoch`; flag g its epoch.  FOUR sets let a rank enqueue
// the scan of search e+1 BEFORE the merge of search e (ShardedIndex.submit / collect): its push of search e+4 reuses set e % 4 only
// after its own merge of e+2, which waited for every peer's push of e+2, which every peer enqueued after its merge of e.
constexpr int kExchangeSlots = 4;
// Behind it, for the FUSED exchange (rvo_search_topk_fused): [4 slot sets][world ranks][nq_max queries] records of rec_bytes
// ([k ids | k scores | count]) | per-(rank, query) epoch flags u64 [4][world][nq_max].
struct ExchangeLayout {
    size_t slot_bytes, flags_off, done_off, bytes;
    size_t rec_bytes, lists_off, lists_set_bytes, qflags_off, qflags_set_bytes;
};
static ExchangeLayout exchange_layout(int world, int nq_max, int k_max) {
    ExchangeLayout L;
    L.slot_bytes = align_up(rvo_packed_result_bytes(nq_max, k_max), 256);
    L.flags_off = kExchangeSlots * (size_t)world * L.slot_bytes;
    L.done_off = L.flags_off + kExchangeSlots * (size_t)world * 8;
    L.rec_bytes = align_up((size_t)k_max * 12 + 4, 16);
    L.lists_off = align_up(L.done_off + 64, 256);
    L.lists_set_bytes = (size_t)world * nq_max * L.rec_bytes;
    L.qflags_off = L.lists_off + kExchangeSlots * L.lists_set_bytes;
    L.qflags_set_bytes = (size_t)world * nq_max * 8;
    L.bytes = L.qflags_off + kExchangeSlots * L.qflags_set_bytes;
    return L;
}

size_t rvo_exchange_bytes(int32_t world, int32_t nq_max, int32_t k_max) {
    if (world < 1 || world > kMaxPeers || nq_max <= 0 || k_max <= 0 || k_max > RVO_MAX_K) return 0;
    return exchange_layout(world, nq_max, k_max).bytes;
}

int rvo_exchange_alloc(size_t bytes, void** out_region) {
    RVO_REQUIRE(out_region && bytes > 0, "exchange_alloc: bad argument");
    void* p = nullptr;
    RVO_CUDA(cudaMalloc(&p, bytes));       // a plain cudaMalloc allocation: the unit cudaIpcGetMemHandle exports
    RVO_CUDA(cudaMemset(p, 0, bytes));
    RVO_CUDA(cudaDeviceSynchronize());
    *out_region = p;
    return RVO_OK;
}

int rvo_exchange_free(void* region) {
    if (region) RVO_CUDA(cudaFree(region));
    return RVO_OK;
}

int rvo_exchange_export(void* region, void* out_handle64) {
    RVO_REQUIRE(region && out_handle64, "exchange_export: null pointer");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t h;
    RVO_CUDA(cudaIpcGetMemHandle(&h, region));
    memcpy(out_handle64, &h, 64);
    return RVO_OK;
}

int rvo_exchange_import(const void* handle64, void** out_region) {
    RVO_REQUIRE(handle64 && out_region, "exchange_import: null pointer");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    void* p = nullptr;
    RVO_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    *out_region = p;
    return RVO_OK;
}

int rvo_exchange_unimport(void* region) {
    if (region) RVO_CUDA(cudaIpcCloseMemHandle(region));
    return RVO_OK;
}

int rvo_search_topk_push(const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad, const float* queries, int32_t nq,
                         int32_t k, float score_threshold, int64_t id_offset, void* const* regions, int32_t world,
                         int32_t rank, int32_t nq_max, int32_t k_max, uint64_t epoch, void* workspace,
                         size_t workspace_bytes, void* stream) {
    RVO_REQUIRE(regions && world >= 2 && world <= kMaxPeers && rank >= 0 && rank < world, "search_topk_push: bad world/rank");
    RVO_REQUIRE(nq > 0 && nq <= nq_max && k > 0 && k <= k_max && epoch > 0, "search_topk_push: nq/k beyond the region's maxima");
    for (int g = 0; g < world; ++g) RVO_REQUIRE(regions[g], "search_topk_push: null region %d", g);
    const ExchangeLayout L = exchange_layout(world, nq_max, k_max);
    const int par = (int)(epoch & (kExchangeSlots - 1));
    PushArgs pa;
    memset(&pa, 0, sizeof(pa));
    pa.world = world;
    pa.rank = rank;
    pa.nq = nq;
    pa.k = k;
    pa.epoch = epoch;
    for (int g = 0; g < world; ++g) {
        unsigned char* base = (unsigned char*)regions[g];
        pa.peer_slot[g] = base + ((size_t)par * world + rank) * L.slot_bytes;
        pa.peer_flag[g] = (unsigned long long*)(base + L.flags_off) + (size_t)par * world + rank;
    }
    unsigned char* local = (unsigned char*)regions[rank];
    pa.done = (unsigned int*)(local + L.done_off) + par;
    unsigned char* slot = pa.peer_slot[rank];
    int64_t* out_ids = (int64_t*)slot;
    float* out_scores = (float*)(slot + (size_t)nq * k * 8);
    int32_t* out_counts = (int32_t*)(slot + (size_t)nq * k * 12);
    return search_impl(db, n_rows, d, d_pad, queries, nq, k, score_threshold, id_offset, out_ids, out_scores, out_counts,
                       workspace, workspace_bytes, stream, &pa);
}

int rvo_search_topk_fused(const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad, const float* queries, int32_t nq,
                          int32_t k, float score_threshold, int64_t id_offset, void* const* regions, int32_t world,
                          int32_t rank, int32_t nq_max, int32_t k_max, uint64_t epoch, int64_t* out_ids, float* out_scores,
                          int32_t* out_counts, void* workspace, size_t workspace_bytes, void* stream) {
    RVO_REQUIRE(regions && world >= 2 && world <= kMaxPeers && rank >= 0 && rank < world, "search_topk_fused: bad world/rank");
    RVO_REQUIRE(nq > 0 && nq <= nq_max && k > 0 && k <= k_max && epoch > 0, "search_topk_fused: nq/k beyond the region's maxima");
    for (int g = 0; g < world; ++g) RVO_REQUIRE(regions[g], "search_topk_fused: null region %d", g);
    if ((long long)world * k > 2048 || k > 512) {
        set_error("search_topk_fused: world * k = %lld beyond the in-kernel merge (2048): use rvo_search_topk_push + "
                  "rvo_merge_topk_exchange", (long long)world * k);
        return RVO_E_UNSUPPORTED;
    }
    const ExchangeLayout L = exchange_layout(world, nq_max, k_max);
    const int par = (int)(epoch & (kExchangeSlots - 1));
    PushArgs pa;
    memset(&pa, 0, sizeof(pa));
    pa.world = world;
    pa.rank = rank;
    pa.nq = nq;
    pa.k = k;
    pa.epoch = epoch;
    pa.fused = 1;
    pa.nq_max = nq_max;
    pa.rec_bytes = (unsigned int)L.rec_bytes;
    pa.timeout_ns = (unsigned long long)g_exchange_timeout_ms.load() * 1000000ull;
    for (int g = 0; g < world; ++g) {
        unsigned char* base = (unsigned char*)regions[g];
        pa.lists[g] = base + L.lists_off + (size_t)par * L.lists_set_bytes;
        pa.qflags[g] = (unsigned long long*)(base + L.qflags_off + (size_t)par * L.qflags_set_bytes);
    }
    return search_impl(db, n_rows, d, d_pad, queries, nq, k, score_threshold, id_offset, out_ids, out_scores, out_counts,
                       workspace, workspace_bytes, stream, &pa);
}

int rvo_merge_topk_exchange(const void* local_region, int32_t world, int32_t nq, int32_t k, int32_t nq_max, int32_t k_max,
                            uint64_t epoch, int64_t* out_ids, float* out_scores, int32_t* out_counts, void* stream) {
    DeviceGuard device_guard;
    RVO_REQUIRE(local_region && out_ids && out_scores && out_counts, "merge_topk_exchange: null pointer");
    RVO_REQUIRE(world >= 2 && world <= kMaxPeers && nq > 0 && nq <= nq_max && k > 0 && k <= k_max && (long long)world * k <= 4096,
                "merge_topk_exchange: bad shape");
    int rc = select_device_of(local_region, nullptr);
    if (rc) return rc;
    const ExchangeLayout L = exchange_layout(world, nq_max, k_max);
    const int par = (int)(epoch & (kExchangeSlots - 1));
    const unsigned char* base = (const unsigned char*)local_region + (size_t)par * world * L.slot_bytes;
    const unsigned long long* flags = (const unsigned long long*)((const unsigned char*)local_region + L.flags_off) + (size_t)par * world;
    return launch_merge((const int64_t*)base, (const float*)(base + (size_t)nq * k * 8), (const int32_t*)(base + (size_t)nq * k * 12),
                        (long long)(L.slot_bytes / 8), (long long)(L.slot_bytes / 4), (long long)(L.slot_bytes / 4), world, nq, k,
                        out_ids, out_scores, out_counts, (cudaStream_t)stream, flags, epoch);
}

int rvo_padded_queries(int32_t nq, int32_t d) {
    TcPlan tc;
    if (nq <= 0 || d <= 0) return RVO_E_INVALID;
    int rc = plan_scan_tc(nq, (d + kBlockK - 1) / kBlockK * kBlockK, (int)opt_m_sub.load(), &tc);
    return rc ? rc : tc.nq_pad;
}

int rvo_scan_tile_rows(int32_t nq, int32_t d) {
    TcPlan tc;
    if (nq <= 0 || d <= 0) return RVO_E_INVALID;
    int rc = plan_scan_tc(nq, (d + kBlockK - 1) / kBlockK * kBlockK, (int)opt_m_sub.load(), &tc);
    return rc ? rc : kBlockM * tc.m_sub;
}

int rvo_scores_dense(const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad_in, const float* queries, int32_t nq,
                     int64_t tile_stride, float* out, int64_t out_ld, void* workspace, size_t workspace_bytes,
                     void* stream_) {
    DeviceGuard device_guard;
    cudaStream_t stream = (cudaStream_t)stream_;
    RVO_REQUIRE(db && queries && out && workspace, "scores_dense: null pointer");
    RVO_REQUIRE(n_rows > 0 && d > 0 && nq > 0 && tile_stride >= 1, "scores_dense: bad shape");
    RVO_REQUIRE(d_pad_in == (d + kBlockK - 1) / kBlockK * kBlockK, "scores_dense: d_pad must be d rounded up to 64");
    RVO_REQUIRE(((uintptr_t)workspace & 1023) == 0, "scores_dense: workspace must be 1024-byte aligned");
    int sm = 0;
    int rc = select_device_of(db, &sm);
    if (rc) return rc;
    const int d_pad = (d + kBlockK - 1) / kBlockK * kBlockK;
    TcPlan tc;
    rc = plan_scan_tc(nq, d_pad, (int)opt_m_sub.load(), &tc);
    if (rc) return rc;
    RVO_REQUIRE(out_ld >= scan_tc_sample_rows(n_rows, tc, tile_stride), "scores_dense: out_ld=%lld too small",
                (long long)out_ld);
    Arena ar(workspace, workspace_bytes);
    uint16_t* qb = ar.take<uint16_t>((size_t)tc.nq_pad * d_pad, 1024);
    if (!ar.ok()) {
        set_error("scores_dense: workspace too small (%zu needed)", ar.off);
        return RVO_E_WORKSPACE;
    }
    RVO_CUDA(cudaMemsetAsync(qb, 0, (size_t)tc.nq_pad * d_pad * 2, stream));
    rc = launch_normalize_rows(queries, nq, d, d, qb, d_pad, -1, nullptr, 0, stream);
    if (rc) return rc;
    return launch_scan_tc(kModeDense, db, n_rows, tile_stride, d_pad, qb, tc, nullptr, nullptr, nullptr, 0, out, out_ld, sm,
                          stream);
}

size_t rvo_selfjoin_workspace_bytes(int32_t d) { return rvo_selfjoin_workspace_bytes_ex(d, opt_cand_cap.load()); }

size_t rvo_selfjoin_workspace_bytes_ex(int32_t d, int64_t cand_cap) {
    if (d <= 0 || cand_cap <= 0) return 0;
    return selfjoin_workspace_bytes(d, cand_cap);
}

int rvo_selfjoin_threshold(const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad_in, int64_t row_lo, int64_t row_hi,
                           float threshold, int64_t id_offset, int64_t* out_pairs, float* out_scores, int64_t out_cap,
                           uint64_t* out_count, int32_t* out_overflowed, void* workspace, size_t workspace_bytes,
                           void* stream) {
    return rvo_selfjoin_threshold_ex(db, n_rows, d, d_pad_in, row_lo, row_hi, threshold, id_offset, opt_cand_cap.load(), out_pairs,
                                     out_scores, out_cap, out_count, out_overflowed, workspace, workspace_bytes, stream);
}

int rvo_selfjoin_threshold_ex(const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad_in, int64_t row_lo, int64_t row_hi,
                              float threshold, int64_t id_offset, int64_t cand_cap, int64_t* out_pairs, float* out_scores,
                              int64_t out_cap, uint64_t* out_count, int32_t* out_overflowed, void* workspace,
                              size_t workspace_bytes, void* stream) {
    DeviceGuard device_guard;
    RVO_REQUIRE(db && out_pairs && out_scores && out_count && workspace, "selfjoin: null pointer");
    RVO_REQUIRE(n_rows > 0 && d > 0 && row_lo >= 0 && row_lo <= row_hi && row_hi <= n_rows && out_cap >= 0 && cand_cap > 0,
                "selfjoin: bad shape n_rows=%lld rows [%lld,%lld)", (long long)n_rows, (long long)row_lo, (long long)row_hi);
    RVO_REQUIRE(d_pad_in == (d + kBlockK - 1) / kBlockK * kBlockK, "selfjoin: d_pad must be d rounded up to 64");
    RVO_REQUIRE(((uintptr_t)workspace & 1023) == 0 && ((uintptr_t)db & 15) == 0, "selfjoin: alignment");
    RVO_REQUIRE(n_rows < (1ll << 31), "selfjoin: too many rows");
    int sm = 0;
    int rc = select_device_of(db, &sm);
    if (rc) return rc;
    return launch_selfjoin(db, row_lo, row_hi, id_offset, db, n_rows, d, threshold, id_offset, cand_cap, (long long*)out_pairs,
                           out_scores, out_cap, nullptr, (unsigned long long*)out_count, out_overflowed, kJoinTriangle, false, workspace,
                           workspace_bytes, sm, (cudaStream_t)stream);
}

size_t rvo_join_workspace_bytes(int32_t d, int64_t cand_cap) { return rvo_selfjoin_workspace_bytes_ex(d, cand_cap); }

// The row-set checks of rvo_join_threshold and rvo_join_components; *triangle: qdb == db with equal id offsets.  Selects the
// target rows' device and sets *sm to its SM count.
static int check_join_rows(const char* what, const uint16_t* qdb, int64_t q_row_lo, int64_t q_row_hi, int64_t q_id_offset,
                           const uint16_t* db, int64_t n_rows, int32_t d, int64_t d_pad_in, int64_t id_offset, int64_t cand_cap,
                           const void* workspace, bool* triangle, int* sm) {
    RVO_REQUIRE(n_rows > 0 && n_rows < (1ll << 31) && d > 0 && q_row_lo >= 0 && q_row_lo <= q_row_hi && cand_cap > 0,
                "%s: bad shape n_rows=%lld query rows [%lld,%lld)", what, (long long)n_rows, (long long)q_row_lo,
                (long long)q_row_hi);
    RVO_REQUIRE(d_pad_in == (d + kBlockK - 1) / kBlockK * kBlockK, "%s: d_pad must be d rounded up to 64", what);
    RVO_REQUIRE(((uintptr_t)workspace & 1023) == 0 && ((uintptr_t)db & 15) == 0 && ((uintptr_t)qdb & 15) == 0,
                "%s: alignment", what);
    *triangle = qdb == db && q_id_offset == id_offset;
    if (*triangle) {
        RVO_REQUIRE(q_row_hi <= n_rows, "%s: query rows [%lld,%lld) outside the %lld rows of the DB", what, (long long)q_row_lo,
                    (long long)q_row_hi, (long long)n_rows);
    } else {
        // rectangle: the two row sets must be disjoint, by id and in memory (a pair would otherwise be found twice or
        // paired with itself)
        RVO_REQUIRE(qdb != db, "%s: qdb == db with different id offsets", what);
        RVO_REQUIRE(q_id_offset + q_row_hi <= id_offset || id_offset + n_rows <= q_id_offset + q_row_lo,
                    "%s: query ids [%lld,%lld) overlap target ids [%lld,%lld)", what, (long long)(q_id_offset + q_row_lo),
                    (long long)(q_id_offset + q_row_hi), (long long)id_offset, (long long)(id_offset + n_rows));
        const size_t blk = (size_t)(d_pad_in / kTileCols) * kTileRows * kTileCols;   // bf16 elements per 128-row block
        const uint16_t *q0 = qdb + (size_t)(q_row_lo / kTileRows) * blk,
                       *q1 = qdb + (size_t)((q_row_hi + kTileRows - 1) / kTileRows) * blk,
                       *t1 = db + (size_t)((n_rows + kTileRows - 1) / kTileRows) * blk;
        RVO_REQUIRE(q_row_lo == q_row_hi || q1 <= db || t1 <= q0, "%s: query rows and target rows overlap in memory", what);
        int qdev = -1, tdev = -1;
        int rc = select_device_of(qdb, nullptr);
        if (rc) return rc;
        RVO_CUDA(cudaGetDevice(&qdev));
        rc = select_device_of(db, nullptr);
        if (rc) return rc;
        RVO_CUDA(cudaGetDevice(&tdev));
        RVO_REQUIRE(qdev == tdev, "%s: query rows on device %d, target rows on device %d", what, qdev, tdev);
    }
    return select_device_of(db, sm);
}

int rvo_join_threshold(const uint16_t* qdb, int64_t q_row_lo, int64_t q_row_hi, int64_t q_id_offset, const uint16_t* db,
                       int64_t n_rows, int32_t d, int64_t d_pad_in, float threshold, int64_t id_offset, int64_t cand_cap,
                       int64_t* out_pairs, float* out_scores, int64_t out_cap, uint64_t* out_count, int32_t* out_overflowed,
                       void* workspace, size_t workspace_bytes, void* stream) {
    DeviceGuard device_guard;
    RVO_REQUIRE(qdb && db && out_pairs && out_scores && out_count && out_overflowed && workspace, "join: null pointer");
    RVO_REQUIRE(out_cap >= 0, "join: out_cap %lld < 0", (long long)out_cap);
    bool triangle = false;
    int sm = 0;
    int rc = check_join_rows("join", qdb, q_row_lo, q_row_hi, q_id_offset, db, n_rows, d, d_pad_in, id_offset, cand_cap, workspace,
                             &triangle, &sm);
    if (rc) return rc;
    return launch_selfjoin(qdb, q_row_lo, q_row_hi, q_id_offset, db, n_rows, d, threshold, id_offset, cand_cap,
                           (long long*)out_pairs, out_scores, out_cap, nullptr, (unsigned long long*)out_count, out_overflowed,
                           triangle ? kJoinTriangle : kJoinRectangle, true, workspace, workspace_bytes, sm, (cudaStream_t)stream);
}

int rvo_join_components(const uint16_t* qdb, int64_t q_row_lo, int64_t q_row_hi, int64_t q_id_offset, const uint16_t* db,
                        int64_t n_rows, int32_t d, int64_t d_pad_in, float threshold, int64_t id_offset, int64_t cand_cap,
                        int32_t* parent, int64_t n_labels, uint64_t* hit_count, int32_t* out_overflowed, void* workspace,
                        size_t workspace_bytes, void* stream) {
    DeviceGuard device_guard;
    RVO_REQUIRE(qdb && db && parent && hit_count && out_overflowed && workspace, "join components: null pointer");
    RVO_REQUIRE(n_labels > 0 && n_labels < (1ll << 31), "join components: %lld labels: the forest holds fewer than 2^31 rows",
                (long long)n_labels);
    RVO_REQUIRE(q_id_offset + q_row_lo >= 0 && q_id_offset + q_row_hi <= n_labels && id_offset >= 0 && id_offset + n_rows <= n_labels,
                "join components: query ids [%lld,%lld) or target ids [%lld,%lld) outside the %lld rows of the forest",
                (long long)(q_id_offset + q_row_lo), (long long)(q_id_offset + q_row_hi), (long long)id_offset,
                (long long)(id_offset + n_rows), (long long)n_labels);
    RVO_REQUIRE(((uintptr_t)parent & 3) == 0, "join components: alignment");
    bool triangle = false;
    int sm = 0;
    int rc = check_join_rows("join components", qdb, q_row_lo, q_row_hi, q_id_offset, db, n_rows, d, d_pad_in, id_offset,
                             cand_cap, workspace, &triangle, &sm);
    if (rc) return rc;
    int tdev = -1, pdev = -1;
    RVO_CUDA(cudaGetDevice(&tdev));
    rc = select_device_of(parent, nullptr);
    if (rc) return rc;
    RVO_CUDA(cudaGetDevice(&pdev));
    RVO_REQUIRE(pdev == tdev, "join components: forest on device %d, target rows on device %d", pdev, tdev);
    return launch_selfjoin(qdb, q_row_lo, q_row_hi, q_id_offset, db, n_rows, d, threshold, id_offset, cand_cap, nullptr, nullptr,
                           0, parent, (unsigned long long*)hit_count, out_overflowed, triangle ? kJoinTriangle : kJoinRectangle,
                           true, workspace, workspace_bytes, sm, (cudaStream_t)stream);
}

int rvo_components_flatten(int32_t* parent, int64_t n, int32_t* labels_out, void* stream) {
    DeviceGuard device_guard;
    RVO_REQUIRE(parent && labels_out, "components flatten: null pointer");
    RVO_REQUIRE(n > 0 && n < (1ll << 31), "components flatten: n=%lld outside [1, 2^31)", (long long)n);
    int sm = 0;
    int rc = select_device_of(parent, &sm);
    if (rc) return rc;
    return launch_components_flatten(parent, (int)n, labels_out, sm, (cudaStream_t)stream);
}

int rvo_components_merge(int32_t* parent, const int32_t* labels_src, int64_t n, void* stream) {
    DeviceGuard device_guard;
    RVO_REQUIRE(parent && labels_src, "components merge: null pointer");
    RVO_REQUIRE(n > 0 && n < (1ll << 31), "components merge: n=%lld outside [1, 2^31)", (long long)n);
    int sm = 0;
    int rc = select_device_of(parent, &sm);
    if (rc) return rc;
    return launch_components_merge(parent, labels_src, (int)n, sm, (cudaStream_t)stream);
}

int rvo_cross_join_threshold(const uint16_t* qdb, int64_t q_row_lo, int64_t q_row_hi, int64_t q_id_offset, const uint16_t* db,
                             int64_t n_rows, int32_t d, int64_t d_pad_in, float threshold, int64_t id_offset,
                             int32_t query_is_right, int64_t cand_cap, int64_t* out_pairs, float* out_scores, int64_t out_cap,
                             uint64_t* out_count, int32_t* out_overflowed, void* workspace, size_t workspace_bytes,
                             void* stream) {
    DeviceGuard device_guard;
    RVO_REQUIRE(qdb && db && out_pairs && out_scores && out_count && out_overflowed && workspace, "cross join: null pointer");
    RVO_REQUIRE(n_rows > 0 && n_rows < (1ll << 31) && d > 0 && q_row_lo >= 0 && q_row_lo <= q_row_hi && out_cap >= 0 &&
                    cand_cap > 0,
                "cross join: bad shape n_rows=%lld query rows [%lld,%lld)", (long long)n_rows, (long long)q_row_lo,
                (long long)q_row_hi);
    RVO_REQUIRE(query_is_right == 0 || query_is_right == 1, "cross join: query_is_right must be 0 or 1, got %d",
                (int)query_is_right);
    RVO_REQUIRE(d_pad_in == (d + kBlockK - 1) / kBlockK * kBlockK, "cross join: d_pad must be d rounded up to 64");
    RVO_REQUIRE(((uintptr_t)workspace & 1023) == 0 && ((uintptr_t)db & 15) == 0 && ((uintptr_t)qdb & 15) == 0,
                "cross join: alignment");
    // the two row sets belong to two collections: their ids may overlap, and qdb == db is the full ordered join of one row set
    // with itself (self pairs included)
    if (qdb == db)
        RVO_REQUIRE(q_row_hi <= n_rows, "cross join: query rows [%lld,%lld) outside the %lld rows of the DB",
                    (long long)q_row_lo, (long long)q_row_hi, (long long)n_rows);
    int qdev = -1, tdev = -1;
    int rc = select_device_of(qdb, nullptr);
    if (rc) return rc;
    RVO_CUDA(cudaGetDevice(&qdev));
    int sm = 0;
    rc = select_device_of(db, &sm);
    if (rc) return rc;
    RVO_CUDA(cudaGetDevice(&tdev));
    RVO_REQUIRE(qdev == tdev, "cross join: query rows on device %d, target rows on device %d", qdev, tdev);
    return launch_selfjoin(qdb, q_row_lo, q_row_hi, q_id_offset, db, n_rows, d, threshold, id_offset, cand_cap,
                           (long long*)out_pairs, out_scores, out_cap, nullptr, (unsigned long long*)out_count, out_overflowed,
                           query_is_right ? kJoinCrossRight : kJoinCrossLeft, true, workspace, workspace_bytes, sm,
                           (cudaStream_t)stream);
}

int rvo_merge_topk(const int64_t* ids, const float* scores, const int32_t* counts, int32_t G, int32_t nq, int32_t k,
                   int64_t* out_ids, float* out_scores, int32_t* out_counts, void* stream) {
    DeviceGuard device_guard;
    RVO_REQUIRE(ids && scores && counts && out_ids && out_scores && out_counts, "merge_topk: null pointer");
    RVO_REQUIRE(G >= 1 && nq >= 1 && k >= 1 && (long long)G * k <= 4096, "merge_topk: need G*k <= 4096 (G=%d k=%d)", G, k);
    int rc = select_device_of(ids, nullptr);
    if (rc) return rc;
    return launch_merge(ids, scores, counts, (long long)nq * k, (long long)nq * k, nq, G, nq, k, out_ids, out_scores,
                        out_counts, (cudaStream_t)stream);
}

size_t rvo_packed_result_bytes(int32_t nq, int32_t k) {
    if (nq <= 0 || k <= 0) return 0;
    return align_up((size_t)nq * k * 12 + (size_t)nq * 4, 8);
}

int rvo_merge_topk_packed(const void* gathered, int64_t rank_stride_bytes, int32_t G, int32_t nq, int32_t k,
                          int64_t* out_ids, float* out_scores, int32_t* out_counts, void* stream) {
    DeviceGuard device_guard;
    RVO_REQUIRE(gathered && out_ids && out_scores && out_counts, "merge_topk_packed: null pointer");
    RVO_REQUIRE(G >= 1 && nq >= 1 && k >= 1 && (long long)G * k <= 4096, "merge_topk_packed: need G*k <= 4096 (G=%d k=%d)",
                G, k);
    RVO_REQUIRE(rank_stride_bytes >= (int64_t)rvo_packed_result_bytes(nq, k) && rank_stride_bytes % 8 == 0 &&
                    ((uintptr_t)gathered & 7) == 0,
                "merge_topk_packed: bad stride/alignment");
    int rc = select_device_of(gathered, nullptr);
    if (rc) return rc;
    const char* base = (const char*)gathered;
    const int64_t* ids = (const int64_t*)base;
    const float* scores = (const float*)(base + (size_t)nq * k * 8);
    const int32_t* counts = (const int32_t*)(base + (size_t)nq * k * 12);
    return launch_merge(ids, scores, counts, rank_stride_bytes / 8, rank_stride_bytes / 4, rank_stride_bytes / 4, G, nq, k,
                        out_ids, out_scores, out_counts, (cudaStream_t)stream);
}

}  // extern "C"
