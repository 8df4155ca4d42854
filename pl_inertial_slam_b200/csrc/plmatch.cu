// C ABI of the B200 descriptor-matching path (include/plmatch.h): contexts, staging, launches.
// Built for sm_100a only; there is no CPU code path behind any compute entry point.
#include "../../include/plmatch.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <thread>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "plm_bow.cuh"
#include "plm_common.cuh"
#include "plm_frames.cuh"
#include "plm_frame_fused.cuh"
#include "plm_grid.cuh"
#include "plm_knn2.cuh"
#include "plm_knn2_umma.cuh"
#include "plm_map.cuh"
#include "plm_reproj.cuh"
#include "plm_micro.cuh"
#include "plm_peer.cuh"
#include "plm_stereo.cuh"

#define PLM_API extern "C" __attribute__((visibility("default")))

namespace {

thread_local std::string g_last_error;

int fail(int status, const std::string &msg) {
    g_last_error = msg;
    return status;
}

#define CU_TRY(expr)                                                                              \
    do {                                                                                          \
        cudaError_t e_ = (expr);                                                                  \
        if (e_ != cudaSuccess) {                                                                  \
            return fail(e_ == cudaErrorMemoryAllocation ? PLM_E_NOMEM : PLM_E_CUDA,               \
                        std::string(#expr) + ": " + cudaGetErrorString(e_));                      \
        }                                                                                         \
    } while (0)

inline size_t align_up(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }

// Accumulates a block layout (offsets first, pointers once the block exists).
struct Layout {
    size_t total = 0;
    size_t add(size_t bytes) {
        const size_t off = total;
        total = align_up(total + bytes);
        return off;
    }
};

} // namespace

struct plm_ctx {
    int device = 0;
    int sm_count = 148;
    size_t smem_optin = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    char *d_buf = nullptr;
    size_t d_cap = 0;
    char *h_buf = nullptr; // pinned
    char *h_buf_dev = nullptr; // the same block as the device addresses it (zero-copy result stores of the frame kernel)
    size_t h_cap = 0;
    char *d_aux = nullptr; // second device scratch: survives the ensure_device of nested entry points
    size_t aux_cap = 0;
    uint64_t launches = 0;
    bool fused_attr_set = false;
    bool cluster_attr_set = false;
    int knn_occ[2][7] = {{0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0}};
    bool umma_attr_set = false;
    // set by knn2_umma_kernel / mma_i8_rate_kernel when an MMA completion wait timed out (mapped pinned word)
    int32_t *umma_err_host = nullptr, *umma_err_dev = nullptr;
    size_t chunked_attr[2] = {0, 0};
    bool rows_attr_set = false;
    bool frame_fused_attr_set = false;
    // frame session: the calls recorded between plm_frame_begin and plm_frame_end
    struct FrameCall {
        int kind = 0; // 0 match / matchNNR, 1 matchGrid
        int is_lines = 0, n1 = 0, n2 = 0, grid_rows = 0, grid_cols = 0, best_lr = 0;
        const uint8_t *d1 = nullptr, *d2 = nullptr;
        size_t step1 = 0, step2 = 0;
        const int32_t *coords = nullptr, *cell_start = nullptr, *cell_items = nullptr;
        const double *dirs2 = nullptr;
        double line_sim_th = 0.0, ratio = 0.0;
        float nnr = 0.f;
        int32_t win[4] = {0, 0, 0, 0};
        int32_t *m12 = nullptr;
        int *n_matches = nullptr;
    };
    bool in_frame = false;
    std::vector<FrameCall> frame_calls;
    cudaStream_t frame_streams[3] = {nullptr, nullptr, nullptr};
    cudaEvent_t frame_events[4] = {nullptr, nullptr, nullptr, nullptr};
    // optional per-launch timing of the brute-force slice kernel (bench.py's roofline)
    bool profiling = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_free;

    int ensure_device(size_t bytes) {
        if (bytes <= d_cap) return PLM_OK;
        CU_TRY(cudaStreamSynchronize(stream));
        if (d_buf) CU_TRY(cudaFree(d_buf));
        d_buf = nullptr;
        d_cap = 0;
        const size_t cap = align_up(bytes + bytes / 4, 1 << 20);
        CU_TRY(cudaMalloc(reinterpret_cast<void **>(&d_buf), cap));
        d_cap = cap;
        return PLM_OK;
    }
    int ensure_aux(size_t bytes) {
        if (bytes <= aux_cap) return PLM_OK;
        CU_TRY(cudaStreamSynchronize(stream));
        if (d_aux) CU_TRY(cudaFree(d_aux));
        d_aux = nullptr;
        aux_cap = 0;
        const size_t cap = align_up(bytes + bytes / 4, 1 << 20);
        CU_TRY(cudaMalloc(reinterpret_cast<void **>(&d_aux), cap));
        aux_cap = cap;
        return PLM_OK;
    }
    int ensure_pinned(size_t bytes) {
        if (bytes <= h_cap) return PLM_OK;
        CU_TRY(cudaStreamSynchronize(stream));
        if (h_buf) CU_TRY(cudaFreeHost(h_buf));
        h_buf = nullptr;
        h_cap = 0;
        const size_t cap = align_up(bytes + bytes / 4, 1 << 16);
        CU_TRY(cudaHostAlloc(reinterpret_cast<void **>(&h_buf), cap, cudaHostAllocDefault));
        h_cap = cap;
        // the address kernels use for zero-copy stores into this block (equal to h_buf under unified addressing)
        void *dp = nullptr;
        h_buf_dev = (cudaHostGetDevicePointer(&dp, h_buf, 0) == cudaSuccess && dp) ? static_cast<char *>(dp) : nullptr;
        if (!h_buf_dev) (void)cudaGetLastError();
        return PLM_OK;
    }
};

// How one host-buffer call is executed.  A stand-alone call runs every phase at once on the context's buffers; inside
// a frame session (plm_frame_begin / plm_frame_end) the call is recorded and its phases run later, interleaved with the
// other calls of the frame: SIZE (layout only), PACK (inputs into the shared pinned block), LAUNCH (H2D of this call's
// inputs, kernels, D2H of its outputs -- all asynchronous on the current stream), UNPACK (after the one sync).
enum ExecPhase { EXEC_ALL = 0, EXEC_SIZE = 1, EXEC_PACK = 2, EXEC_LAUNCH = 3, EXEC_UNPACK = 4 };
struct Exec {
    int phase = EXEC_ALL;
    char *h_base = nullptr, *d_base = nullptr; // this call's sub-blocks (phases PACK .. UNPACK)
    size_t h_bytes = 0, d_bytes = 0;            // reported by phase SIZE
};

namespace {
int frame_end_fused(plm_ctx *ctx, const plm_ctx::FrameCall *calls, int n, bool *done);
}

struct plm_db {
    plm_ctx *ctx = nullptr;
    uint4 *rows = nullptr;
    int64_t capacity = 0;
    int64_t size = 0;
};

namespace {

struct TlsCtx {
    plm_ctx *ctx = nullptr;
    ~TlsCtx() {
        if (ctx) plm_ctx_destroy(ctx);
    }
};
thread_local TlsCtx g_tls;

// Makes the context's device current for the calling thread.  NOTE: like cudaSetDevice itself this is sticky -- a call
// with an explicit context on another GPU leaves that GPU current afterwards (documented in include/plmatch.h).
int resolve_ctx(plm_ctx *&ctx) {
    if (ctx) {
        int cur = -1;
        if (cudaGetDevice(&cur) != cudaSuccess || cur != ctx->device) CU_TRY(cudaSetDevice(ctx->device));
        return PLM_OK;
    }
    if (!g_tls.ctx) {
        int dev = 0;
        CU_TRY(cudaGetDevice(&dev));
        const int st = plm_ctx_create(dev, &g_tls.ctx);
        if (st != PLM_OK) return st;
    }
    ctx = g_tls.ctx;
    CU_TRY(cudaSetDevice(ctx->device));
    return PLM_OK;
}

// Packs n rows of 32 bytes, `step` bytes apart, into a contiguous block.
void pack_rows(void *dst, const uint8_t *src, int64_t n, size_t step) {
    if (n <= 0) return;
    if (step == 32) {
        std::memcpy(dst, src, static_cast<size_t>(n) * 32);
    } else {
        uint8_t *d = static_cast<uint8_t *>(dst);
        for (int64_t i = 0; i < n; ++i) std::memcpy(d + i * 32, src + static_cast<size_t>(i) * step, 32);
    }
}

struct KnnPlan {
    int threads = 128;
    int unit_rows = plm::KNN_STAGE_ROWS;
    int n_units = 1;
    int n_workers = 1;
    int qpb = 128;        // queries per CTA (threads, or 2 x threads in the two-queries-per-thread form)
    int extra_qb = 0;     // query blocks with n_workers + 1 workers (fills the last resident CTA slots)
    bool share_thr = false; // long scans: the workers of a query share their second-best bound
};

// frame pipeline: candidate slots per query row the pair-list form is sized for (points, lines); options
// "frames_pairs_p" / "frames_pairs_l", 0 = chunk phases only.  Lines default to the chunk phases: a segment
// sits in ~8 cells, so a row holds ~20 slots for ~6 distinct candidates, the slot arrays push the CTA to one
// per SM and the measured stereo-lines stage is 6x slower than with the chunk phases (profiles/r1_frames.md).
int g_frames_pairs_per_row[2] = {8, 0};
int g_frames_out_group = 2;  // plm_frames_process: chunks per device -> host copy group (option "frames_out_group")
int g_frames_threads_l = 256; // threads per CTA of the line chain of the frame pipeline (128 or 256; measurement knob)
int g_frames_threads_p = 512; // ... of the point chain (256 or 512)
int g_grid_cluster = 2; // single matchGrid calls: 2 = row-parallel kernel on one cluster, 1 = chunk kernel on an 8-CTA cluster, 0 = one CTA
long long g_peer_spin_ticks = 4000000000ll; // bounded spin of the peer-memory kernels (~2 s of SM clock); option "peer_spin_ms"
int g_knn_qpt = 1;      // 2: long scans with >= 4096 queries keep two queries per thread (variant 6); option "knn_qpt"
int g_knn_fill = 1;     // long brute-force scans: uneven workers fill every CTA slot + shared second-best bound (0: off, measurement)
int g_frame_fused = 1;  // frame sessions run as ONE launch (frame_fused_kernel) when every recorded call fits (0: one lane per call)
int g_grid_head = 1;    // map-sized matchGrid: short CTAs at the start of the map (0: uniform rows per CTA, measurement / tests)
int g_grid_rows = 1;    // map-sized matchGrid uses the row-parallel kernels (0: warp-per-chunk kernels, measurement / tests)

// -1 = automatic (the tensor-core kernel for long scans with many queries, variant 3 for other long slices, 1 otherwise);
// 0..5 force an integer variant, 7 the tensor-core kernel wherever a launch could take it (measurement and tests)
int g_knn_variant = -2;
// fewest queries for which a long scan (>= 65 536 train rows) runs on the tensor cores: a group of 256 queries costs the
// tensor kernel the same whether it is full or not, and at 256 queries it is already 3.1 x faster (DESIGN K1b)
constexpr int KNN_UMMA_MIN_QUERIES = 256;
int knn_variant_for(int slice_rows) {
    if (g_knn_variant == -2) {
        const char *e = std::getenv("PLM_KNN_VARIANT");
        g_knn_variant = -1;
        if (e && std::strcmp(e, "popc8") == 0) g_knn_variant = 0;
        if (e && std::strcmp(e, "csa5") == 0) g_knn_variant = 1;
        if (e && std::strcmp(e, "csa4") == 0) g_knn_variant = 2;
        if (e && std::strcmp(e, "t13") == 0) g_knn_variant = 3;
        if (e && std::strcmp(e, "mix") == 0) g_knn_variant = 4;
        if (e && std::strcmp(e, "t13s") == 0) g_knn_variant = 5;
        if (e && std::strcmp(e, "umma") == 0) g_knn_variant = 7;
        const char *f = std::getenv("PLM_KNN_FILL"); // measurement knob, same as option "knn_fill"
        if (f) g_knn_fill = std::atoi(f) ? 1 : 0;
        const char *q2 = std::getenv("PLM_KNN_QPT");
        if (q2) g_knn_qpt = std::atoi(q2) == 2 ? 2 : 1;
    }
    if (g_knn_variant >= 0 && g_knn_variant != 7) return g_knn_variant;
    return slice_rows >= 2048 ? 3 : 1;
}

// Single-direction launches (allow_two) of a long scan take the tensor-core kernel (variant 7).
bool knn_use_umma(int n1, long long n2, bool allow_two) {
    (void)knn_variant_for(0); // reads PLM_KNN_VARIANT on first use
    if (!allow_two || n2 <= 0) return false;
    if (g_knn_variant == 7) return true;
    return g_knn_variant < 0 && n2 >= 65536 && n1 >= KNN_UMMA_MIN_QUERIES;
}

// CTAs of the brute-force kernel that are resident on one SM (per CTA width and variant).
int knn_ctas_per_sm(plm_ctx *ctx, int threads, int variant) {
    int &cached = ctx->knn_occ[threads == 128 ? 1 : 0][variant];
    if (cached > 0) return cached;
    int nb = 0;
    cudaError_t e = cudaErrorUnknown;
#define PLM_KNN_OCC(T, V) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, plm::knn2_slice_kernel<T, V>, T, 0)
    if (threads == 128) {
        if (variant == 6) PLM_KNN_OCC(128, 6);
        else if (variant == 5) PLM_KNN_OCC(128, 5);
        else if (variant == 4) PLM_KNN_OCC(128, 4);
        else if (variant == 3) PLM_KNN_OCC(128, 3);
        else if (variant == 2) PLM_KNN_OCC(128, 2);
        else if (variant == 1) PLM_KNN_OCC(128, 1);
        else PLM_KNN_OCC(128, 0);
    } else {
        if (variant == 5) PLM_KNN_OCC(64, 5);
        else if (variant == 4) PLM_KNN_OCC(64, 4);
        else if (variant == 3) PLM_KNN_OCC(64, 3);
        else if (variant == 2) PLM_KNN_OCC(64, 2);
        else if (variant == 1) PLM_KNN_OCC(64, 1);
        else PLM_KNN_OCC(64, 0);
    }
#undef PLM_KNN_OCC
    cached = (e == cudaSuccess && nb > 0) ? nb : 8;
    return cached;
}

// The train set is cut into units of <= 256 rows (one shared-memory stage) dealt round-robin to as many
// workers per query block as fit on the chip at once: one wave of co-resident CTAs, no last-wave tail,
// W partials per query.  Frame-sized problems get narrow CTAs and small units so that a single call
// still spreads over the whole chip.
KnnPlan plan_knn(plm_ctx *ctx, int n1, long long n2, bool allow_two = false) {
    KnnPlan p;
    if (knn_use_umma(n1, n2, allow_two)) {
        // one CTA per SM, each owning an equal contiguous share of the (query group, 128-row unit) list; n_workers =
        // the most CTAs any query group is spread over (knn2_umma_kernel writes the slots a group does not use)
        p.threads = p.qpb = plm::KNN_UMMA_THREADS;
        p.unit_rows = plm::KNN_UMMA_ROWS;
        const long long groups = std::max(1, (n1 + p.qpb - 1) / p.qpb), units = (n2 + p.unit_rows - 1) / p.unit_rows;
        const long long total = groups * units, ctas = std::min<long long>(ctx->sm_count, total);
        p.n_units = static_cast<int>(units);
        p.n_workers = 1;
        for (long long g = 0; g < groups; ++g)
            p.n_workers = static_cast<int>(std::max<long long>(p.n_workers, plm::umma_cta_of(g * units + units - 1, total, ctas) -
                                                                                  plm::umma_cta_of(g * units, total, ctas) + 1));
        p.share_thr = true;
        return p;
    }
    p.threads = (n1 >= 4096) ? 128 : 64;
    int variant = knn_variant_for(n2 >= 65536 ? 4096 : 64);
    // a short train side with a lot of work is launched with variant 5 (launch_knn_slices): plan the workers for it
    if (variant == 1 && (g_knn_variant < 0 || g_knn_variant == 7) && n2 >= 64 && static_cast<long long>(n1) * n2 >= (1ll << 26)) variant = 5;
    // long scans with many queries: two queries per thread (variant 6), single-direction launches only
    if (allow_two && variant == 3 && g_knn_qpt == 2 && p.threads == 128) variant = 6;
    p.qpb = (variant == 6) ? 2 * p.threads : p.threads;
    const long long qblocks = std::max<long long>(1, (n1 + p.qpb - 1) / p.qpb);
    const long long capacity = static_cast<long long>(ctx->sm_count) * knn_ctas_per_sm(ctx, p.threads, variant);
    const long long want = std::max<long long>(1, capacity / qblocks); // workers per query block
    long long rows = (n2 + want - 1) / want;
    rows = std::min<long long>(plm::KNN_STAGE_ROWS, std::max<long long>(64, (rows + 63) / 64 * 64));
    p.unit_rows = static_cast<int>(rows);
    p.n_units = static_cast<int>(std::max<long long>(1, (n2 + rows - 1) / rows));
    p.n_workers = static_cast<int>(std::min<long long>(p.n_units, want));
    if (variant >= 2 && g_knn_fill) {
        // long scans: qblocks x workers rarely divides the resident CTA slots (50 x 26 = 1300 of 1332): the first
        // `extra_qb` query blocks get one more worker, so that a launch fills every slot
        if (p.n_workers == want && p.n_units > want && qblocks * want < capacity) p.extra_qb = static_cast<int>(std::min<long long>(qblocks, capacity - qblocks * want));
        p.share_thr = true;
    }
    return p;
}

// The mapped pinned word the tensor-core kernels raise when an MMA completion wait runs past the spin limit (option
// "peer_spin_ms").  Such a launch's results are undefined, so from then on every tensor-core launch of the context fails
// instead of returning them.
int umma_error_word(plm_ctx *ctx) {
    if (!ctx->umma_err_host) {
        int32_t *h = nullptr;
        void *d = nullptr;
        CU_TRY(cudaHostAlloc(reinterpret_cast<void **>(&h), sizeof(int32_t), cudaHostAllocMapped));
        *h = 0;
        const cudaError_t e = cudaHostGetDevicePointer(&d, h, 0);
        if (e != cudaSuccess) {
            cudaFreeHost(h);
            return fail(PLM_E_CUDA, std::string("cudaHostGetDevicePointer: ") + cudaGetErrorString(e));
        }
        ctx->umma_err_host = h;
        ctx->umma_err_dev = static_cast<int32_t *>(d);
    }
    if (*reinterpret_cast<volatile int32_t *>(ctx->umma_err_host) != 0)
        return fail(PLM_E_CUDA, "tensor-core brute force: an MMA completion wait timed out in an earlier launch on this context "
                                "(its results are undefined); destroy the context");
    return PLM_OK;
}

int launch_knn_slices(plm_ctx *ctx, plm::KnnTaskPair &tp, int n_tasks, int threads) {
    long long total = 0;
    for (int i = 0; i < n_tasks; ++i) {
        const int qpb = tp.t[i].threads > 0 ? tp.t[i].threads : threads; // queries per CTA of this task
        const long long c = static_cast<long long>((tp.t[i].n1 + qpb - 1) / qpb) * tp.t[i].n_workers + tp.t[i].extra_qb;
        if (i == 0) tp.cta_split = static_cast<int>(c);
        total += c;
    }
    if (n_tasks == 1) tp.cta_split = static_cast<int>(total);
    // planned for the tensor-core kernel (plan_knn: single task, 256 queries per CTA)
    const bool umma = n_tasks == 1 && threads == plm::KNN_UMMA_THREADS;
    if (umma) {
        const long long units = tp.t[0].n_units, groups = (tp.t[0].n1 + threads - 1) / threads;
        total = std::min<long long>(ctx->sm_count, groups * units);
        tp.cta_split = static_cast<int>(total);
    }
    if (total == 0) return PLM_OK;
    if (total > INT_MAX) return fail(PLM_E_UNSUPPORTED, "too many query blocks");
    const dim3 grid(static_cast<unsigned>(total), 1, 1);
    int min_rows = INT_MAX;
    for (int i = 0; i < n_tasks; ++i) min_rows = std::min<long long>(min_rows, std::min<long long>(tp.t[i].n2, INT_MAX));
    int variant = knn_variant_for(min_rows >= 65536 ? 4096 : 64);
    if (variant == 1 && (g_knn_variant < 0 || g_knn_variant == 7) && min_rows >= 64) {
        // a short train side but a lot of work (the match fallback of the local map, 200 000 x 600 in both directions):
        // the 13-LOP3 distance with the per-pair update (variant 5) -- a few per cent there (0.369 -> 0.356 ms, plan_knn sizes the workers for it); frame-sized calls keep
        // variant 1, whose stages need no in-place transform
        long long pairs = 0;
        for (int i = 0; i < n_tasks; ++i) pairs = std::max(pairs, static_cast<long long>(tp.t[i].n1) * tp.t[i].n2);
        if (pairs >= (1ll << 26)) variant = 5;
    }
    if (n_tasks == 1 && tp.t[0].threads == 2 * threads) variant = 6; // planned with two queries per thread
    if (umma) {
        if (!ctx->umma_attr_set) {
            CU_TRY(cudaFuncSetAttribute(plm::knn2_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, plm::KNN_UMMA_SMEM));
            ctx->umma_attr_set = true;
        }
        const int st = umma_error_word(ctx);
        if (st != PLM_OK) return st;
    }
    if (umma || (variant >= 2 && g_knn_fill)) {
        // the shared second-best bounds live behind each task's partial results (build_knn_task reserved the room)
        for (int i = 0; i < n_tasks; ++i) {
            plm::KnnTask &t = tp.t[i];
            if (!t.part || t.n1 <= 0) continue;
            t.gthr = reinterpret_cast<uint32_t *>(t.part + size_t(t.n_workers + (t.extra_qb ? 1 : 0)) * size_t(t.n1));
            CU_TRY(cudaMemsetAsync(t.gthr, 0xFF, size_t(t.n1) * 4, ctx->stream));
        }
    }
    std::pair<cudaEvent_t, cudaEvent_t> ev{nullptr, nullptr};
    if (ctx->profiling) {
        if (!ctx->prof_free.empty()) {
            ev = ctx->prof_free.back();
            ctx->prof_free.pop_back();
        } else {
            CU_TRY(cudaEventCreate(&ev.first));
            CU_TRY(cudaEventCreate(&ev.second));
        }
        CU_TRY(cudaEventRecord(ev.first, ctx->stream));
    }
#define PLM_KNN_LAUNCH(T, V) plm::knn2_slice_kernel<T, V><<<grid, T, 0, ctx->stream>>>(tp)
    if (umma) {
        plm::knn2_umma_kernel<<<grid, plm::KNN_UMMA_CTA_THREADS, plm::KNN_UMMA_SMEM, ctx->stream>>>(tp.t[0], ctx->umma_err_dev, g_peer_spin_ticks);
    } else if (threads == 128) {
        if (variant == 6) PLM_KNN_LAUNCH(128, 6);
        else if (variant == 5) PLM_KNN_LAUNCH(128, 5);
        else if (variant == 4) PLM_KNN_LAUNCH(128, 4);
        else if (variant == 3) PLM_KNN_LAUNCH(128, 3);
        else if (variant == 2) PLM_KNN_LAUNCH(128, 2);
        else if (variant == 1) PLM_KNN_LAUNCH(128, 1);
        else PLM_KNN_LAUNCH(128, 0);
    } else {
        if (variant == 5) PLM_KNN_LAUNCH(64, 5);
        else if (variant == 4) PLM_KNN_LAUNCH(64, 4);
        else if (variant == 3) PLM_KNN_LAUNCH(64, 3);
        else if (variant == 2) PLM_KNN_LAUNCH(64, 2);
        else if (variant == 1) PLM_KNN_LAUNCH(64, 1);
        else PLM_KNN_LAUNCH(64, 0);
    }
#undef PLM_KNN_LAUNCH
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    if (ctx->profiling) {
        CU_TRY(cudaEventRecord(ev.second, ctx->stream));
        ctx->prof_events.push_back(ev);
    }
    return PLM_OK;
}

int launch_knn_merge(plm_ctx *ctx, const plm::KnnTaskPair &tp, int n_tasks, float nnr, int do_accept) {
    // few queries with many partials each (a short query side against a long train side) get one warp per
    // query; the two directions of match() can differ, so the choice is per task
    auto wide = [&](int i) { return tp.t[i].n_workers >= 32 && tp.t[i].n1 <= 16384; };
    const bool split = n_tasks == 2 && wide(0) != wide(1);
    for (int first = 0; first < n_tasks; first += split ? 1 : n_tasks) {
        const int cnt = split ? 1 : n_tasks;
        int n = 0;
        for (int i = first; i < first + cnt; ++i) n = std::max(n, tp.t[i].n1);
        if (n == 0) continue;
        if (wide(first)) {
            const dim3 grid((n + 3) / 4, cnt);
            plm::knn2_merge_wide_kernel<<<grid, 128, 0, ctx->stream>>>(tp, first, nnr, do_accept);
        } else {
            const dim3 grid((n + 127) / 128, cnt);
            plm::knn2_merge_kernel<<<grid, 128, 0, ctx->stream>>>(tp, first, nnr, do_accept);
        }
        ctx->launches++;
        CU_TRY(cudaGetLastError());
    }
    return PLM_OK;
}

int check_desc(const uint8_t *d, int n, size_t step) {
    if (n < 0) return fail(PLM_E_INVALID, "negative row count");
    if (n > 0 && !d) return fail(PLM_E_INVALID, "null descriptor pointer");
    if (n > 0 && step < 32) return fail(PLM_E_INVALID, "descriptor step < 32 bytes");
    return PLM_OK;
}

} // namespace

// ---------------------------------------------------------------------------------------------
PLM_API int plm_set_option(const char *key, int value) {
    if (!key) return fail(PLM_E_INVALID, "null key");
    if (std::strcmp(key, "knn_variant") == 0) {
        g_knn_variant = ((value >= 0 && value <= 5) || value == 7) ? value : -1;
        return PLM_OK;
    }
    if (std::strcmp(key, "peer_spin_ms") == 0) {
        g_peer_spin_ticks = static_cast<long long>(std::max(1, value)) * 2000000ll; // ~2 GHz SM clock
        return PLM_OK;
    }
    if (std::strcmp(key, "knn_qpt") == 0) {
        g_knn_qpt = value == 2 ? 2 : 1;
        return PLM_OK;
    }
    if (std::strcmp(key, "knn_fill") == 0) {
        g_knn_fill = value ? 1 : 0;
        return PLM_OK;
    }
    if (std::strcmp(key, "grid_head") == 0) {
        g_grid_head = value ? 1 : 0;
        return PLM_OK;
    }
    if (std::strcmp(key, "grid_rows") == 0) {
        g_grid_rows = value ? 1 : 0;
        return PLM_OK;
    }
    if (std::strcmp(key, "frame_fused") == 0) {
        g_frame_fused = value ? 1 : 0;
        return PLM_OK;
    }
    if (std::strcmp(key, "grid_cluster") == 0) {
        g_grid_cluster = std::max(0, std::min(value, 2));
        return PLM_OK;
    }
    if (std::strcmp(key, "frames_out_group") == 0) {
        g_frames_out_group = std::max(1, std::min(value, 64));
        return PLM_OK;
    }
    if (std::strcmp(key, "frames_threads_l") == 0) {
        g_frames_threads_l = value >= 256 ? 256 : 128;
        return PLM_OK;
    }
    if (std::strcmp(key, "frames_threads_p") == 0) {
        g_frames_threads_p = value >= 512 ? 512 : 256;
        return PLM_OK;
    }
    if (std::strcmp(key, "frames_pairs_p") == 0 || std::strcmp(key, "frames_pairs_l") == 0) {
        g_frames_pairs_per_row[key[13] == 'l' ? 1 : 0] = std::max(0, std::min(value, 64));
        return PLM_OK;
    }
    return fail(PLM_E_INVALID, std::string("unknown option ") + key);
}

PLM_API int plm_version(void) { return PLM_VERSION; }

PLM_API const char *plm_status_string(int status) {
    switch (status) {
    case PLM_OK: return "ok";
    case PLM_E_INVALID: return "invalid argument";
    case PLM_E_SIZE: return "size mismatch between features and descriptors";
    case PLM_E_TRAIN: return "fewer than two train descriptors";
    case PLM_E_GRID: return "[GridStructure] invalid dimension";
    case PLM_E_RATIO: return "matchGrid ratio must be <= 1";
    case PLM_E_CUDA: return "CUDA failure";
    case PLM_E_NOMEM: return "out of memory";
    case PLM_E_UNSUPPORTED: return "unsupported size";
    case PLM_E_PEER: return "peer-memory exchange timed out";
    default: return "unknown status";
    }
}

PLM_API const char *plm_last_error(void) { return g_last_error.c_str(); }

PLM_API int plm_device_count(int *count) {
    if (!count) return fail(PLM_E_INVALID, "null count");
    *count = 0;
    CU_TRY(cudaGetDeviceCount(count));
    return PLM_OK;
}

PLM_API int plm_ctx_create(int device, plm_ctx **out) {
    if (!out) return fail(PLM_E_INVALID, "null out");
    *out = nullptr;
    int n = 0;
    CU_TRY(cudaGetDeviceCount(&n));
    if (device < 0 || device >= n) return fail(PLM_E_CUDA, "no such CUDA device");
    CU_TRY(cudaSetDevice(device));
    plm_ctx *c = new (std::nothrow) plm_ctx();
    if (!c) return fail(PLM_E_NOMEM, "host allocation failed");
    c->device = device;
    cudaDeviceProp prop;
    cudaError_t e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) {
        delete c;
        return fail(PLM_E_CUDA, cudaGetErrorString(e));
    }
    c->sm_count = prop.multiProcessorCount;
    c->smem_optin = prop.sharedMemPerBlockOptin;
    e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete c;
        return fail(PLM_E_CUDA, cudaGetErrorString(e));
    }
    c->stream = c->own_stream;
    *out = c;
    return PLM_OK;
}

PLM_API int plm_ctx_destroy(plm_ctx *ctx) {
    if (!ctx) return PLM_OK;
    cudaSetDevice(ctx->device);
    if (ctx->own_stream) {
        cudaStreamSynchronize(ctx->own_stream);
        cudaStreamDestroy(ctx->own_stream);
    }
    for (int i = 0; i < 3; ++i)
        if (ctx->frame_streams[i]) cudaStreamDestroy(ctx->frame_streams[i]);
    for (int i = 0; i < 4; ++i)
        if (ctx->frame_events[i]) cudaEventDestroy(ctx->frame_events[i]);
    if (ctx->d_buf) cudaFree(ctx->d_buf);
    if (ctx->d_aux) cudaFree(ctx->d_aux);
    if (ctx->h_buf) cudaFreeHost(ctx->h_buf);
    if (ctx->umma_err_host) cudaFreeHost(ctx->umma_err_host);
    if (g_tls.ctx == ctx) g_tls.ctx = nullptr;
    delete ctx;
    return PLM_OK;
}

PLM_API void *plm_ctx_stream(plm_ctx *ctx) { return ctx ? static_cast<void *>(ctx->stream) : nullptr; }

PLM_API int plm_ctx_set_stream(plm_ctx *ctx, void *cuda_stream, int external) {
    if (!ctx) return fail(PLM_E_INVALID, "null ctx");
    ctx->stream = external ? static_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
    return PLM_OK;
}

PLM_API int plm_ctx_synchronize(plm_ctx *ctx) {
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    return PLM_OK;
}

PLM_API int plm_ctx_set_profiling(plm_ctx *ctx, int on) {
    if (!ctx) return fail(PLM_E_INVALID, "null ctx");
    ctx->profiling = on != 0;
    return PLM_OK;
}

PLM_API int plm_ctx_read_profile(plm_ctx *ctx, double *knn2_slice_ms, int *n_launches) {
    if (!ctx) return fail(PLM_E_INVALID, "null ctx");
    CU_TRY(cudaSetDevice(ctx->device));
    double total = 0.0;
    int n = 0;
    for (auto &ev : ctx->prof_events) {
        CU_TRY(cudaEventSynchronize(ev.second));
        float ms = 0.f;
        CU_TRY(cudaEventElapsedTime(&ms, ev.first, ev.second));
        total += ms;
        ++n;
        ctx->prof_free.push_back(ev);
    }
    ctx->prof_events.clear();
    if (knn2_slice_ms) *knn2_slice_ms = total;
    if (n_launches) *n_launches = n;
    return PLM_OK;
}

PLM_API uint64_t plm_ctx_launch_count(plm_ctx *ctx) {
    if (!ctx) ctx = g_tls.ctx;
    return ctx ? ctx->launches : 0;
}

// ---------------------------------------------------------------------------------------------
PLM_API int plm_hamming256(plm_ctx *ctx, const uint8_t *a, size_t step_a, const uint8_t *b, size_t step_b,
                           int n, int32_t *dist) {
    int st = check_desc(a, n, step_a);
    if (st == PLM_OK) st = check_desc(b, n, step_b);
    if (st != PLM_OK) return st;
    if (n > 0 && !dist) return fail(PLM_E_INVALID, "null dist");
    if (n == 0) return PLM_OK;
    if ((st = resolve_ctx(ctx)) != PLM_OK) return st;
    Layout L;
    const size_t o_a = L.add(size_t(n) * 32), o_b = L.add(size_t(n) * 32);
    const size_t in_bytes = L.total;
    const size_t o_d = L.add(size_t(n) * 4);
    if ((st = ctx->ensure_pinned(L.total)) != PLM_OK) return st;
    if ((st = ctx->ensure_device(L.total)) != PLM_OK) return st;
    pack_rows(ctx->h_buf + o_a, a, n, step_a);
    pack_rows(ctx->h_buf + o_b, b, n, step_b);
    CU_TRY(cudaMemcpyAsync(ctx->d_buf, ctx->h_buf, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    plm::hamming_pairs_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(
        reinterpret_cast<const uint4 *>(ctx->d_buf + o_a), reinterpret_cast<const uint4 *>(ctx->d_buf + o_b), n,
        reinterpret_cast<int32_t *>(ctx->d_buf + o_d));
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(ctx->h_buf + o_d, ctx->d_buf + o_d, size_t(n) * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    std::memcpy(dist, ctx->h_buf + o_d, size_t(n) * 4);
    return PLM_OK;
}

// ---------------------------------------------------------------------------------------------
// Brute force on device-resident rows; partial buffers come from the context scratch AFTER
// `reserved` bytes (which the caller is using for its own staged data).
namespace {

struct KnnScratch {
    size_t part_off[2] = {0, 0};
};

int build_knn_task(plm_ctx *ctx, Layout &L, plm::KnnTask &t, KnnPlan &plan, const uint4 *q, int n1, const uint4 *db,
                   long long n2, unsigned long long idx_base, size_t &part_off, bool allow_two = false) {
    plan = plan_knn(ctx, n1, n2, allow_two);
    t.q = q;
    t.db = db;
    t.n1 = n1;
    t.n2 = n2;
    t.idx_base = idx_base;
    t.unit_rows = plan.unit_rows;
    t.n_units = plan.n_units;
    t.n_workers = plan.n_workers;
    t.extra_qb = plan.extra_qb;
    t.threads = plan.qpb;
    t.part = nullptr;
    t.top2 = nullptr;
    t.m = nullptr;
    t.count = nullptr;
    t.gthr = nullptr;
    // behind the partial results: room for the per-query bound the workers of a launch share (launch_knn_slices)
    part_off = L.add(size_t(plan.n_workers + (plan.extra_qb ? 1 : 0)) * size_t(std::max(n1, 1)) * sizeof(ulonglong2) +
                     align_up(size_t(std::max(n1, 1)) * 4));
    return PLM_OK;
}

} // namespace

PLM_API int plm_dev_knn2(plm_ctx *ctx, const void *d1_dev, int n1, const void *d2_dev, int64_t n2, uint64_t idx_base,
                         uint64_t *top2_dev) {
    if (n1 < 0 || n2 < 0) return fail(PLM_E_INVALID, "negative row count");
    if ((n1 > 0 && !d1_dev) || (n2 > 0 && !d2_dev) || (n1 > 0 && !top2_dev)) return fail(PLM_E_INVALID, "null pointer");
    if ((reinterpret_cast<uintptr_t>(d1_dev) | reinterpret_cast<uintptr_t>(d2_dev) | reinterpret_cast<uintptr_t>(top2_dev)) & 15)
        return fail(PLM_E_INVALID, "device pointers must be 16-byte aligned");
    if (idx_base + static_cast<uint64_t>(n2) > (1ull << 32)) return fail(PLM_E_UNSUPPORTED, "train index does not fit 32 bits");
    if (n1 == 0) return PLM_OK;
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    Layout L;
    plm::KnnTaskPair tp;
    std::memset(&tp, 0, sizeof(tp));
    KnnPlan plan;
    size_t part_off = 0;
    build_knn_task(ctx, L, tp.t[0], plan, static_cast<const uint4 *>(d1_dev), n1, static_cast<const uint4 *>(d2_dev), n2,
                   idx_base, part_off, true);
    if ((st = ctx->ensure_device(L.total)) != PLM_OK) return st;
    tp.t[0].part = reinterpret_cast<ulonglong2 *>(ctx->d_buf + part_off);
    tp.t[0].top2 = reinterpret_cast<ulonglong2 *>(top2_dev);
    if ((st = launch_knn_slices(ctx, tp, 1, plan.threads)) != PLM_OK) return st;
    return launch_knn_merge(ctx, tp, 1, 0.f, 0);
}

PLM_API int plm_dev_top2_merge(plm_ctx *ctx, const uint64_t *parts_dev, int n_parts, int n1, uint64_t *top2_out_dev) {
    if (n_parts < 0 || n1 < 0) return fail(PLM_E_INVALID, "negative size");
    if (n1 > 0 && (!parts_dev || !top2_out_dev)) return fail(PLM_E_INVALID, "null pointer");
    if (n1 == 0) return PLM_OK;
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    plm::top2_merge_kernel<<<(n1 + 127) / 128, 128, 0, ctx->stream>>>(reinterpret_cast<const ulonglong2 *>(parts_dev), n_parts, n1,
                                                                     reinterpret_cast<ulonglong2 *>(top2_out_dev));
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    return PLM_OK;
}

PLM_API int plm_dev_nnr_accept(plm_ctx *ctx, const uint64_t *top2_dev, int n1, float nnr, int32_t *m12_dev_inout,
                               int32_t *count_dev) {
    if (n1 < 0) return fail(PLM_E_INVALID, "negative size");
    if (n1 > 0 && (!top2_dev || !m12_dev_inout)) return fail(PLM_E_INVALID, "null pointer");
    if (n1 == 0) return PLM_OK;
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    plm::nnr_accept_kernel<<<(n1 + 127) / 128, 128, 0, ctx->stream>>>(reinterpret_cast<const ulonglong2 *>(top2_dev), n1, nnr,
                                                                     m12_dev_inout, count_dev);
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    return PLM_OK;
}

PLM_API int plm_dev_cross_check(plm_ctx *ctx, int32_t *m12_dev_inout, int n1, int64_t i1_base, const int32_t *m21_dev,
                                int64_t n2, int32_t *count_dev) {
    if (n1 < 0 || n2 < 0) return fail(PLM_E_INVALID, "negative size");
    if (n1 > 0 && (!m12_dev_inout || !count_dev || (n2 > 0 && !m21_dev))) return fail(PLM_E_INVALID, "null pointer");
    if (n1 == 0) return PLM_OK;
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    plm::cross_check_kernel<<<(n1 + 127) / 128, 128, 0, ctx->stream>>>(m12_dev_inout, n1, i1_base, m21_dev, n2, count_dev);
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    return PLM_OK;
}

// ---------------------------------------------------------------------------------------------
PLM_API int plm_knn2(plm_ctx *ctx, const uint8_t *d1, int n1, size_t step1, const uint8_t *d2, int n2, size_t step2,
                     uint64_t idx_base, uint64_t *top2) {
    int st = check_desc(d1, n1, step1);
    if (st == PLM_OK) st = check_desc(d2, n2, step2);
    if (st != PLM_OK) return st;
    if (n1 > 0 && !top2) return fail(PLM_E_INVALID, "null top2");
    if (idx_base + static_cast<uint64_t>(n2) > (1ull << 32)) return fail(PLM_E_UNSUPPORTED, "train index does not fit 32 bits");
    if (n1 == 0) return PLM_OK;
    if ((st = resolve_ctx(ctx)) != PLM_OK) return st;

    Layout L;
    const size_t o_d1 = L.add(size_t(n1) * 32), o_d2 = L.add(size_t(n2) * 32);
    const size_t in_bytes = L.total;
    const size_t o_top2 = L.add(size_t(n1) * 16);
    const size_t staged = L.total;
    plm::KnnTaskPair tp;
    std::memset(&tp, 0, sizeof(tp));
    KnnPlan plan;
    size_t part_off = 0;
    build_knn_task(ctx, L, tp.t[0], plan, nullptr, n1, nullptr, n2, idx_base, part_off, true);
    if ((st = ctx->ensure_pinned(staged)) != PLM_OK) return st;
    if ((st = ctx->ensure_device(L.total)) != PLM_OK) return st;
    pack_rows(ctx->h_buf + o_d1, d1, n1, step1);
    pack_rows(ctx->h_buf + o_d2, d2, n2, step2);
    CU_TRY(cudaMemcpyAsync(ctx->d_buf, ctx->h_buf, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    tp.t[0].q = reinterpret_cast<const uint4 *>(ctx->d_buf + o_d1);
    tp.t[0].db = reinterpret_cast<const uint4 *>(ctx->d_buf + o_d2);
    tp.t[0].part = reinterpret_cast<ulonglong2 *>(ctx->d_buf + part_off);
    tp.t[0].top2 = reinterpret_cast<ulonglong2 *>(ctx->d_buf + o_top2);
    if ((st = launch_knn_slices(ctx, tp, 1, plan.threads)) != PLM_OK) return st;
    if ((st = launch_knn_merge(ctx, tp, 1, 0.f, 0)) != PLM_OK) return st;
    CU_TRY(cudaMemcpyAsync(ctx->h_buf + o_top2, ctx->d_buf + o_top2, size_t(n1) * 16, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    std::memcpy(top2, ctx->h_buf + o_top2, size_t(n1) * 16);
    return PLM_OK;
}

// StVO::matchNNR / StVO::match share one implementation: direction 21 + mutual check are added
// when best_lr is set.
static int match_impl(plm_ctx *ctx, const uint8_t *d1, int n1, size_t step1, const uint8_t *d2, int n2, size_t step2,
                      float nnr, int best_lr, int32_t *m12_inout, int *n_matches, Exec *ex = nullptr) {
    int st = check_desc(d1, n1, step1);
    if (st == PLM_OK) st = check_desc(d2, n2, step2);
    if (st != PLM_OK) return st;
    if (!n_matches) return fail(PLM_E_INVALID, "null n_matches");
    if (n1 > 0 && !m12_inout) return fail(PLM_E_INVALID, "null m12");
    *n_matches = 0;
    // Degenerate sizes (sparse frames).  The reference: an empty query matches nothing and returns 0 (knnMatch yields no
    // rows, matching.cpp:50 holds; the throw of the 21 direction is swallowed by future::wait, :74); an empty train set
    // with a non-empty query throws (:50-51) -> PLM_E_TRAIN; a SINGLE train row makes it read matches_[idx][1] out of
    // bounds (:54, UB, it does not throw).  Here a row without a second neighbour is simply not accepted (the merge
    // kernels require both keys), so one-row inputs leave m12 untouched in that direction and the mutual check culls.
    if (n1 == 0) return PLM_OK;
    if (n2 == 0) return fail(PLM_E_TRAIN, "matchNNR: empty train set");
    if ((st = resolve_ctx(ctx)) != PLM_OK) return st;
    if (!ex) { // frame session: record, run at plm_frame_end; a stand-alone frame-sized call is a session of one call
        plm_ctx::FrameCall c;
        c.kind = 0; c.d1 = d1; c.n1 = n1; c.step1 = step1; c.d2 = d2; c.n2 = n2; c.step2 = step2; c.nnr = nnr; c.best_lr = best_lr;
        c.m12 = m12_inout; c.n_matches = n_matches;
        if (ctx->in_frame) {
            ctx->frame_calls.push_back(c);
            return PLM_OK;
        }
        bool done = false;
        if ((st = frame_end_fused(ctx, &c, 1, &done)) != PLM_OK || done) return st;
    }
    const int phase = ex ? ex->phase : EXEC_ALL;

    Layout L;
    const size_t o_d1 = L.add(size_t(n1) * 32), o_d2 = L.add(size_t(n2) * 32);
    const size_t o_m12 = L.add(size_t(n1) * 4 + 4); // m12 followed by the counter
    const size_t in_bytes = L.total;
    const size_t o_m21 = L.add(size_t(n2) * 4);
    const size_t staged = L.total;
    plm::KnnTaskPair tp;
    std::memset(&tp, 0, sizeof(tp));
    KnnPlan plan[2];
    size_t part_off[2] = {0, 0};
    build_knn_task(ctx, L, tp.t[0], plan[0], nullptr, n1, nullptr, n2, 0, part_off[0], !best_lr);
    if (best_lr) build_knn_task(ctx, L, tp.t[1], plan[1], nullptr, n2, nullptr, n1, 0, part_off[1]);
    (void)staged;
    if (phase == EXEC_SIZE) {
        ex->h_bytes = in_bytes;
        ex->d_bytes = L.total;
        return PLM_OK;
    }
    if (phase == EXEC_ALL) {
        if ((st = ctx->ensure_pinned(in_bytes)) != PLM_OK) return st;
        if ((st = ctx->ensure_device(L.total)) != PLM_OK) return st;
    }
    char *HB = ex && phase != EXEC_ALL ? ex->h_base : ctx->h_buf, *DB = ex && phase != EXEC_ALL ? ex->d_base : ctx->d_buf;
    if (phase == EXEC_ALL || phase == EXEC_PACK) {
        pack_rows(HB + o_d1, d1, n1, step1);
        pack_rows(HB + o_d2, d2, n2, step2);
        std::memcpy(HB + o_m12, m12_inout, size_t(n1) * 4);
        std::memset(HB + o_m12 + size_t(n1) * 4, 0, 4);
        if (phase == EXEC_PACK) return PLM_OK;
    }
    if (phase == EXEC_UNPACK) {
        std::memcpy(m12_inout, HB + o_m12, size_t(n1) * 4);
        int32_t cnt_u;
        std::memcpy(&cnt_u, HB + o_m12 + size_t(n1) * 4, 4);
        *n_matches = cnt_u;
        return PLM_OK;
    }
    CU_TRY(cudaMemcpyAsync(DB, HB, in_bytes, cudaMemcpyHostToDevice, ctx->stream));

    const uint4 *dd1 = reinterpret_cast<const uint4 *>(DB + o_d1);
    const uint4 *dd2 = reinterpret_cast<const uint4 *>(DB + o_d2);
    int32_t *dm12 = reinterpret_cast<int32_t *>(DB + o_m12);
    int32_t *dcount = dm12 + n1;
    int32_t *dm21 = reinterpret_cast<int32_t *>(DB + o_m21);
    tp.t[0].q = dd1;
    tp.t[0].db = dd2;
    tp.t[0].part = reinterpret_cast<ulonglong2 *>(DB + part_off[0]);
    tp.t[0].m = dm12;
    tp.t[0].count = dcount;
    int n_tasks = 1;
    if (best_lr) {
        CU_TRY(cudaMemsetAsync(dm21, 0xFF, size_t(n2) * 4, ctx->stream));
        tp.t[1].q = dd2;
        tp.t[1].db = dd1;
        tp.t[1].part = reinterpret_cast<ulonglong2 *>(DB + part_off[1]);
        tp.t[1].m = dm21;
        tp.t[1].count = nullptr; // the reference ignores the 21 count (matching.cpp:72,77)
        n_tasks = 2;
    }
    const int threads = std::max(plan[0].threads, best_lr ? plan[1].threads : 0);
    // both directions share one launch and therefore one CTA width; the slice plans stay valid
    if ((st = launch_knn_slices(ctx, tp, n_tasks, threads)) != PLM_OK) return st;
    if ((st = launch_knn_merge(ctx, tp, n_tasks, nnr, 1)) != PLM_OK) return st;
    if (best_lr) {
        plm::cross_check_kernel<<<(n1 + 127) / 128, 128, 0, ctx->stream>>>(dm12, n1, 0, dm21, n2, dcount);
        ctx->launches++;
        CU_TRY(cudaGetLastError());
    }
    CU_TRY(cudaMemcpyAsync(HB + o_m12, DB + o_m12, size_t(n1) * 4 + 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (phase == EXEC_LAUNCH) return PLM_OK;
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    std::memcpy(m12_inout, HB + o_m12, size_t(n1) * 4);
    int32_t cnt;
    std::memcpy(&cnt, HB + o_m12 + size_t(n1) * 4, 4);
    *n_matches = cnt;
    return PLM_OK;
}

PLM_API int plm_match_nnr(plm_ctx *ctx, const uint8_t *d1, int n1, size_t step1, const uint8_t *d2, int n2, size_t step2,
                          float nnr, int32_t *m12_inout, int *n_matches) {
    return match_impl(ctx, d1, n1, step1, d2, n2, step2, nnr, 0, m12_inout, n_matches);
}

PLM_API int plm_match(plm_ctx *ctx, const uint8_t *d1, int n1, size_t step1, const uint8_t *d2, int n2, size_t step2,
                      float nnr, int best_lr, int32_t *m12_inout, int *n_matches) {
    return match_impl(ctx, d1, n1, step1, d2, n2, step2, nnr, best_lr ? 1 : 0, m12_inout, n_matches);
}

// ---------------------------------------------------------------------------------------------
// matchGrid
namespace {

constexpr int GRID_N2_MAX = 32768;
constexpr int GRID_CHUNK_ROWS_PER_WARP = 32;
constexpr int GRID_FUSED_MAX_ROWS = 4096;

struct FusedShape {
    int warps;
    int staged;
    size_t smem;
};

// Shape of the fused kernel: stage the job's inputs in shared memory when they fit next to at least
// 8 chunk arrays, then as many warps (chunks) as the remaining shared memory allows, >= ~4 rows each.
FusedShape fused_shape(const plm_ctx *ctx, int n1_max, int n2_max, int items_max, int n_cells, bool any_lines) {
    const size_t budget = ctx->smem_optin - 2048;
    const int want = std::min(32, std::max(1, (n1_max + 3) / 4));
    for (int staged = 1; staged >= 0; --staged) {
        int w = want;
        while (w > 1 && plm::grid_fused_smem(w, n2_max, staged, n1_max, items_max, n_cells, any_lines) > budget) --w;
        const size_t need = plm::grid_fused_smem(w, n2_max, staged, n1_max, items_max, n_cells, any_lines);
        if (need <= budget && (!staged || w >= std::min(want, 8))) return {w, staged, need};
    }
    return {1, 0, plm::grid_fused_smem(1, n2_max, 0, n1_max, items_max, n_cells, any_lines)};
}

int validate_grid(const int32_t *cell_start, const int32_t *cell_items, int grid_rows, int grid_cols, int *n_items) {
    if (grid_rows <= 0 || grid_cols <= 0) return fail(PLM_E_GRID, "[GridStructure] invalid dimension");
    if (static_cast<long long>(grid_rows) * grid_cols > (1 << 24)) return fail(PLM_E_UNSUPPORTED, "grid too large");
    if (!cell_start) return fail(PLM_E_INVALID, "null cell_start");
    const int n_cells = grid_rows * grid_cols;
    if (cell_start[0] != 0) return fail(PLM_E_GRID, "cell_start[0] must be 0");
    for (int c = 0; c < n_cells; ++c)
        if (cell_start[c + 1] < cell_start[c]) return fail(PLM_E_GRID, "cell_start must be non-decreasing");
    *n_items = cell_start[n_cells];
    if (*n_items > 0 && !cell_items) return fail(PLM_E_INVALID, "null cell_items");
    return PLM_OK;
}

int launch_grid_fused(plm_ctx *ctx, const plm::GridJob *jobs_dev, int n_jobs, plm::GridParams gp, int n1_max,
                      int n2_max, int items_max, bool any_lines) {
    const FusedShape fs = fused_shape(ctx, n1_max, n2_max, items_max, gp.grid_rows * gp.grid_cols, any_lines);
    if (fs.smem > ctx->smem_optin - 2048) return fail(PLM_E_UNSUPPORTED, "matchGrid: train set too large for shared memory");
    gp.staged = fs.staged;
    gp.cap_n1 = n1_max;
    gp.cap_items = items_max;
    if (!ctx->fused_attr_set) {
        CU_TRY(cudaFuncSetAttribute(plm::grid_match_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    static_cast<int>(ctx->smem_optin - 2048)));
        ctx->fused_attr_set = true;
    }
    plm::grid_match_fused_kernel<<<n_jobs, fs.warps * 32, fs.smem, ctx->stream>>>(jobs_dev, gp, n2_max);
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    return PLM_OK;
}

// One frame-sized job on a cluster of 8 CTAs (8 SMs) -- the single-call path.
constexpr int GRID_CLUSTER = 8;

int launch_grid_cluster(plm_ctx *ctx, const plm::GridJob *jobs_dev, int n_jobs, plm::GridParams gp, int n1_max, int n2_max,
                        int items_max, bool any_lines) {
    const size_t budget = ctx->smem_optin - 2048;
    const int n_cells = gp.grid_rows * gp.grid_cols;
    int warps = 16, staged = 1;
    size_t smem = 0;
    for (;;) {
        const int rpw = (n1_max + GRID_CLUSTER * warps - 1) / (GRID_CLUSTER * warps);
        smem = plm::grid_cluster_smem(warps, n2_max, staged, warps * rpw, items_max, n_cells, any_lines);
        if (smem <= budget) {
            gp.cap_n1 = warps * rpw;
            break;
        }
        if (staged) staged = 0;
        else if (warps > 1) warps >>= 1;
        else return fail(PLM_E_UNSUPPORTED, "matchGrid: train set too large for shared memory");
    }
    gp.staged = staged;
    gp.cap_items = items_max;
    if (!ctx->cluster_attr_set) {
        CU_TRY(cudaFuncSetAttribute(plm::grid_match_cluster_kernel<GRID_CLUSTER>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    static_cast<int>(ctx->smem_optin - 2048)));
        ctx->cluster_attr_set = true;
    }
    cudaLaunchConfig_t cfg;
    std::memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(GRID_CLUSTER * n_jobs, 1, 1);
    cfg.blockDim = dim3(warps * 32, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = GRID_CLUSTER;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    CU_TRY(cudaLaunchKernelEx(&cfg, plm::grid_match_cluster_kernel<GRID_CLUSTER>, jobs_dev, gp, n2_max));
    ctx->launches++;
    return PLM_OK;
}


// Map-sized jobs.  Row-parallel kernels (one thread per row, csrc/plm_grid.cuh grid_rows_kernel) whenever their
// per-column work arrays fit shared memory, else the warp-per-chunk kernels.  warps == 0 selects the row-parallel
// form; n_cta is sized so that the whole launch is one wave of co-resident CTAs.

// Shared-memory plan of the row-parallel kernels (grid_rows_device): per-column work arrays + block arrays are fixed;
// the frame side is staged when everything stays under ~72 KB (3 CTAs per SM); the pair list takes what is left, at
// least 2048 entries.  false = the work arrays do not fit (the warp-per-chunk kernels take the job).
bool plan_grid_rows_smem(plm_ctx *ctx, int n2c, int n_cells, bool is_lines, plm::GridParams &gp, size_t &smem) {
    const size_t optin = ctx->smem_optin - 2048;
    const size_t fixed = plm::grid_rows_layout(n2c, is_lines, 0, n_cells, 0, 0).total;
    if (!(g_grid_rows && n2c <= 0xFFFF && fixed + 2048 * 4 <= std::min<size_t>(optin, 160 * 1024))) return false;
    const size_t target = 72 * 1024;
    const size_t frame = plm::grid_rows_layout(n2c, is_lines, 0, n_cells, 0, 1).total - fixed;
    gp.staged = (fixed + frame + 3072 * 4 <= target) ? 1 : 0;
    size_t room = std::max<size_t>(target, fixed + 2048 * 4 + 64) - fixed - (gp.staged ? frame : 0);
    gp.cap_items = gp.staged ? static_cast<int>(std::min<size_t>(room / 4 / 4, 8192)) : 0; // <= a quarter of the room
    room -= plm::grid_align16(size_t(gp.cap_items) * 4);
    gp.cap_pairs = static_cast<int>(std::min<size_t>(room / 4 - 8, 16384));
    smem = plm::grid_rows_layout(n2c, is_lines, gp.cap_pairs, n_cells, gp.cap_items, gp.staged).total;
    return true;
}

int plan_map_grid(plm_ctx *ctx, long long n1, int n2, int n_cells, bool is_lines, plm::GridParams &gp, int &warps, int &n_cta,
                  size_t &smem) {
    const size_t optin = ctx->smem_optin - 2048;
    const int n2c = std::max(n2, 1);
    if (plan_grid_rows_smem(ctx, n2c, n_cells, is_lines, gp, smem)) {
        warps = 0;
        if (!ctx->rows_attr_set) {
            CU_TRY(cudaFuncSetAttribute(plm::grid_rows_kernel<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(optin)));
            CU_TRY(cudaFuncSetAttribute(plm::grid_rows_kernel<0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(optin)));
            CU_TRY(cudaFuncSetAttribute(plm::grid_rows_kernel<1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(optin)));
            CU_TRY(cudaFuncSetAttribute(plm::grid_rows_kernel<1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(optin)));
            CU_TRY(cudaFuncSetAttribute(plm::grid_rows_cluster_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(optin)));
            CU_TRY(cudaFuncSetAttribute(plm::grid_rows_cluster_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(optin)));
            ctx->rows_attr_set = true;
        }
        int per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, plm::grid_rows_kernel<1, 1>, plm::GRID_ROW_THREADS, smem) != cudaSuccess || per_sm < 1)
            per_sm = 1;
        const long long resident = static_cast<long long>(ctx->sm_count) * per_sm;
        const long long blocks = (n1 + plm::GRID_ROW_THREADS - 1) / plm::GRID_ROW_THREADS;
        if (blocks >= resident) {
            const long long per_cta = (blocks + resident - 1) / resident; // whole blocks of rows per CTA
            gp.rows_per_cta = static_cast<int>(per_cta * plm::GRID_ROW_THREADS);
        } else {
            // fewer rows than one wave of full blocks: spread them over every resident slot (>= 64 rows per CTA, whole
            // warps) -- the pair-list phases use all 256 threads of a CTA whatever its row count, and dense windows
            // (lines: ~50 slots per row) make those phases the bulk of the work
            const long long per = (n1 + resident - 1) / resident;
            gp.rows_per_cta = static_cast<int>(std::min<long long>(plm::GRID_ROW_THREADS, std::max<long long>(64, (per + 31) / 32 * 32)));
        }
        n_cta = static_cast<int>((n1 + gp.rows_per_cta - 1) / gp.rows_per_cta);
        // spare slots of the wave go to short CTAs at the start of the map (GridParams::head_ctas)
        gp.head_ctas = 0;
        gp.head_rows = 0;
        const int head_rows = 64;
        for (long long h = g_grid_head ? std::min<long long>(64, resident - n_cta) : 0; h >= 8; --h) {
            const long long covered = h * head_rows;
            if (covered >= n1) continue;
            const long long rest = (n1 - covered + gp.rows_per_cta - 1) / gp.rows_per_cta;
            if (h + rest <= resident) {
                gp.head_ctas = static_cast<int>(h);
                gp.head_rows = head_rows;
                n_cta = static_cast<int>(h + rest);
                break;
            }
        }
        return PLM_OK;
    }
    const size_t budget = std::min<size_t>(optin, 200 * 1024);
    warps = 16;
    while (warps > 1 && size_t(warps) * n2c * 2 > budget) warps >>= 1;
    const long long rows_per_cta = static_cast<long long>(warps) * GRID_CHUNK_ROWS_PER_WARP;
    n_cta = static_cast<int>((n1 + rows_per_cta - 1) / rows_per_cta);
    smem = size_t(warps) * n2c * 2;
    gp.rows_per_warp = GRID_CHUNK_ROWS_PER_WARP;
    for (int pass = 0; pass < 2; ++pass) {
        if (ctx->chunked_attr[pass] < smem) {
            if (pass == 0)
                CU_TRY(cudaFuncSetAttribute(plm::grid_match_chunked_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(optin)));
            else
                CU_TRY(cudaFuncSetAttribute(plm::grid_match_chunked_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(optin)));
            ctx->chunked_attr[pass] = optin;
        }
    }
    return PLM_OK;
}

// Hand-over scratch of the row-parallel launch (pass 0 -> pass 1): [seg_tab][seg_cnt][ent_g]
size_t map_grid_handover_bytes(int warps, int n_cta, int rows_per_cta) {
    if (warps != 0 || n_cta <= 0) return 0;
    return align_up(size_t(n_cta) * plm::GRID_SEG_TAB * sizeof(int4)) + align_up(size_t(n_cta) * 4) +
           align_up(size_t(n_cta) * rows_per_cta * plm::GRID_ENT_PER_ROW * 4);
}
void map_grid_handover_bind(plm::GridParams &gp, char *base, int warps, int n_cta, bool best_lr) {
    gp.ent_g = nullptr;
    gp.seg_tab = nullptr;
    gp.seg_cnt = nullptr;
    gp.ent_per_cta = 0;
    if (warps != 0 || n_cta <= 0 || !best_lr || !base) return;
    gp.seg_tab = reinterpret_cast<int4 *>(base);
    base += align_up(size_t(n_cta) * plm::GRID_SEG_TAB * sizeof(int4));
    gp.seg_cnt = reinterpret_cast<int32_t *>(base);
    base += align_up(size_t(n_cta) * 4);
    gp.ent_g = reinterpret_cast<uint32_t *>(base);
    gp.ent_per_cta = gp.rows_per_cta * plm::GRID_ENT_PER_ROW;
}

int launch_map_grid(plm_ctx *ctx, int pass, const plm::GridJob &job, const plm::GridParams &gp, int warps, int n_cta, size_t smem) {
    if (n_cta <= 0) return PLM_OK;
    if (warps == 0) {
        if (pass == 0 && gp.staged) plm::grid_rows_kernel<0, 1><<<n_cta, plm::GRID_ROW_THREADS, smem, ctx->stream>>>(job, gp);
        else if (pass == 0) plm::grid_rows_kernel<0, 0><<<n_cta, plm::GRID_ROW_THREADS, smem, ctx->stream>>>(job, gp);
        else if (gp.staged) plm::grid_rows_kernel<1, 1><<<n_cta, plm::GRID_ROW_THREADS, smem, ctx->stream>>>(job, gp);
        else plm::grid_rows_kernel<1, 0><<<n_cta, plm::GRID_ROW_THREADS, smem, ctx->stream>>>(job, gp);
    } else {
        if (pass == 0) plm::grid_match_chunked_kernel<0><<<n_cta, warps * 32, smem, ctx->stream>>>(job, gp);
        else plm::grid_match_chunked_kernel<1><<<n_cta, warps * 32, smem, ctx->stream>>>(job, gp);
    }
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    return PLM_OK;
}

// Frame-sized job (<= 8 x 256 rows) as ONE launch: the row-parallel kernel on one thread-block cluster.
constexpr int GRID_ROWS_CLUSTER_MAX = 8;
int launch_grid_rows_cluster(plm_ctx *ctx, const plm::GridJob &job, const plm::GridParams &gp, int n_cta, size_t smem) {
    cudaLaunchConfig_t cfg;
    std::memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(n_cta, 1, 1);
    cfg.blockDim = dim3(plm::GRID_ROW_THREADS, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = n_cta;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (gp.staged) CU_TRY(cudaLaunchKernelEx(&cfg, plm::grid_rows_cluster_kernel<1>, job, gp));
    else CU_TRY(cudaLaunchKernelEx(&cfg, plm::grid_rows_cluster_kernel<0>, job, gp));
    ctx->launches++;
    return PLM_OK;
}

// Map-sized job: pass 0 (per-CTA minima) -> scan -> pass 1 (match) -> mutual check.
// scratch: cta_min [n_cta][n2] u16, m21key [n2] u64, m21 [n2] i32 -- offsets into ctx->d_buf.
int launch_grid_chunked(plm_ctx *ctx, char *DB, const plm::GridJob &job, plm::GridParams gp, size_t off_cta_min, size_t off_m21key,
                        size_t off_m21, int warps, int n_cta, size_t smem) {
    int st;
    gp.cta_min = reinterpret_cast<uint16_t *>(DB + off_cta_min);
    gp.m21key = reinterpret_cast<unsigned long long *>(DB + off_m21key);
    int32_t *m21 = reinterpret_cast<int32_t *>(DB + off_m21);
    if (gp.best_lr) {
        CU_TRY(cudaMemsetAsync(gp.m21key, 0xFF, size_t(job.n2) * 8, ctx->stream));
        if ((st = launch_map_grid(ctx, 0, job, gp, warps, n_cta, smem)) != PLM_OK) return st;
        plm::grid_scan_kernel<<<(job.n2 + 3) / 4, 128, 0, ctx->stream>>>(gp.cta_min, n_cta, job.n2, nullptr, nullptr);
        ctx->launches++;
        CU_TRY(cudaGetLastError());
    }
    if ((st = launch_map_grid(ctx, 1, job, gp, warps, n_cta, smem)) != PLM_OK) return st;
    if (gp.best_lr) {
        (void)m21;
        plm::cross_check_keys_kernel<<<(job.n1 + 255) / 256, 256, 0, ctx->stream>>>(job.m12, job.n1, job.i1_base, gp.m21key, job.n2,
                                                                                   job.count);
        ctx->launches++;
        CU_TRY(cudaGetLastError());
    }
    return PLM_OK;
}

int match_grid_impl(plm_ctx *ctx, int is_lines, const int32_t *coords, const uint8_t *d1, int n1, size_t step1,
                    const int32_t *cell_start, const int32_t *cell_items, int grid_rows, int grid_cols, const uint8_t *d2,
                    int n2, size_t step2, const double *dirs2, double line_sim_th, const int32_t win[4], double ratio,
                    int best_lr, int32_t *m12_inout, int *n_matches, Exec *ex = nullptr) {
    int st = check_desc(d1, n1, step1);
    if (st == PLM_OK) st = check_desc(d2, n2, step2);
    if (st != PLM_OK) return st;
    if (!n_matches || !win) return fail(PLM_E_INVALID, "null n_matches / win");
    if (n1 > 0 && (!coords || !m12_inout)) return fail(PLM_E_INVALID, "null coords / m12");
    if (is_lines && n2 > 0 && !dirs2) return fail(PLM_E_INVALID, "null dirs2");
    *n_matches = 0;
    if (ratio > 1.0) return fail(PLM_E_RATIO, plm_status_string(PLM_E_RATIO));
    int n_items = 0;
    if ((st = validate_grid(cell_start, cell_items, grid_rows, grid_cols, &n_items)) != PLM_OK) return st;
    if (n2 > GRID_N2_MAX) return fail(PLM_E_UNSUPPORTED, "matchGrid supports at most 32768 train features");
    if (n1 == 0) return PLM_OK;
    if ((st = resolve_ctx(ctx)) != PLM_OK) return st;
    if (!ex) { // frame session: record, run at plm_frame_end; a stand-alone frame-sized call is a session of one call
        plm_ctx::FrameCall c;
        c.kind = 1; c.is_lines = is_lines; c.coords = coords; c.d1 = d1; c.n1 = n1; c.step1 = step1; c.cell_start = cell_start;
        c.cell_items = cell_items; c.grid_rows = grid_rows; c.grid_cols = grid_cols; c.d2 = d2; c.n2 = n2; c.step2 = step2; c.dirs2 = dirs2;
        c.line_sim_th = line_sim_th; c.ratio = ratio; c.best_lr = best_lr; c.m12 = m12_inout; c.n_matches = n_matches;
        for (int i = 0; i < 4; ++i) c.win[i] = win[i];
        if (ctx->in_frame) {
            ctx->frame_calls.push_back(c);
            return PLM_OK;
        }
        bool done = false;
        if ((st = frame_end_fused(ctx, &c, 1, &done)) != PLM_OK || done) return st;
    }
    const int phase = ex ? ex->phase : EXEC_ALL;

    const int n_cells = grid_rows * grid_cols;
    const int cpq = is_lines ? 4 : 2;
    Layout L;
    const size_t o_d1 = L.add(size_t(n1) * 32), o_d2 = L.add(size_t(std::max(n2, 1)) * 32);
    const size_t o_xy = L.add(size_t(n1) * cpq * 4);
    const size_t o_cs = L.add(size_t(n_cells + 1) * 4), o_ci = L.add(size_t(std::max(n_items, 1)) * 4);
    const size_t o_dir = L.add(is_lines ? size_t(std::max(n2, 1)) * 16 : 0);
    const size_t o_job = L.add(sizeof(plm::GridJob));
    const size_t o_m12 = L.add(size_t(n1) * 4 + 4);
    const size_t in_bytes = L.total;
    const size_t staged = L.total;

    // single-launch kernels: the per-column arrays of at least one chunk (8 bytes per train feature) must fit shared memory;
    // wider train sides take the multi-launch kernels whatever the number of rows
    const bool fused = n1 <= GRID_FUSED_MAX_ROWS && n1 < (1 << plm::GRID_KEY_BITS) &&
                       size_t(8) * size_t(std::max(n2, 1)) + 1024 <= ctx->smem_optin - 2048;
    int warps = 0, n_cta = 0;
    size_t map_smem = 0;
    size_t o_cta_min = 0, o_m21key = 0, o_m21 = 0, o_handover = 0;
    plm::GridParams gp;
    std::memset(&gp, 0, sizeof(gp));
    // frame-sized single calls: the row-parallel kernel on one cluster (one launch) when its work arrays fit
    bool rows_cluster = fused && n1 >= 64 && n1 <= GRID_ROWS_CLUSTER_MAX * plm::GRID_ROW_THREADS && g_grid_cluster >= 2;
    if (rows_cluster) {
        if ((st = plan_map_grid(ctx, n1, n2, n_cells, is_lines != 0, gp, warps, n_cta, map_smem)) != PLM_OK) return st;
        if (warps != 0) {
            rows_cluster = false; // frame wider than the shared-memory work arrays: chunk kernels
        } else {
            // spread the rows over all 8 CTAs of the cluster (a CTA always has 256 threads: the rows of its block feed
            // phase A, all threads share the flat pair list of phase B)
            int rpc = ((n1 + GRID_ROWS_CLUSTER_MAX - 1) / GRID_ROWS_CLUSTER_MAX + 31) / 32 * 32;
            rpc = std::min(rpc, plm::GRID_ROW_THREADS);
            gp.rows_per_cta = rpc;
            gp.head_ctas = 0; // uniform rows: the CTA index is the cluster rank
            gp.head_rows = 0;
            n_cta = (n1 + rpc - 1) / rpc;
            o_m21key = L.add(size_t(std::max(n2, 1)) * 8);
        }
    }
    if (!fused) {
        if ((st = plan_map_grid(ctx, n1, n2, n_cells, is_lines != 0, gp, warps, n_cta, map_smem)) != PLM_OK) return st;
        o_cta_min = L.add(size_t(n_cta) * std::max(n2, 1) * 2);
        o_handover = L.add(map_grid_handover_bytes(warps, n_cta, gp.rows_per_cta));
        o_m21key = L.add(size_t(std::max(n2, 1)) * 8);
        o_m21 = L.add(size_t(std::max(n2, 1)) * 4);
    }
    if (phase == EXEC_SIZE) {
        ex->h_bytes = staged;
        ex->d_bytes = L.total;
        return PLM_OK;
    }
    if (phase == EXEC_ALL) {
        if ((st = ctx->ensure_pinned(staged)) != PLM_OK) return st;
        if ((st = ctx->ensure_device(L.total)) != PLM_OK) return st;
    }
    char *HB = ex && phase != EXEC_ALL ? ex->h_base : ctx->h_buf, *DB = ex && phase != EXEC_ALL ? ex->d_base : ctx->d_buf;
    if (phase == EXEC_UNPACK) {
        std::memcpy(m12_inout, HB + o_m12, size_t(n1) * 4);
        int32_t cnt_u;
        std::memcpy(&cnt_u, HB + o_m12 + size_t(n1) * 4, 4);
        *n_matches = cnt_u;
        return PLM_OK;
    }

    plm::GridJob job;
    std::memset(&job, 0, sizeof(job));
    job.coords = reinterpret_cast<const int32_t *>(DB + o_xy);
    job.d1 = reinterpret_cast<const uint4 *>(DB + o_d1);
    job.cell_start = reinterpret_cast<const int32_t *>(DB + o_cs);
    job.cell_items = reinterpret_cast<const int32_t *>(DB + o_ci);
    job.d2 = reinterpret_cast<const uint4 *>(DB + o_d2);
    job.dirs2 = reinterpret_cast<const double *>(DB + o_dir);
    job.m12 = reinterpret_cast<int32_t *>(DB + o_m12);
    job.count = job.m12 + n1;
    job.n1 = n1;
    job.n2 = n2;
    job.is_lines = is_lines;
    for (int i = 0; i < 4; ++i) job.win[i] = win[i];
    job.i1_base = 0;
    if (phase == EXEC_ALL || phase == EXEC_PACK) {
        pack_rows(HB + o_d1, d1, n1, step1);
        pack_rows(HB + o_d2, d2, n2, step2);
        std::memcpy(HB + o_xy, coords, size_t(n1) * cpq * 4);
        std::memcpy(HB + o_cs, cell_start, size_t(n_cells + 1) * 4);
        if (n_items > 0) std::memcpy(HB + o_ci, cell_items, size_t(n_items) * 4);
        if (is_lines && n2 > 0) std::memcpy(HB + o_dir, dirs2, size_t(n2) * 16);
        std::memcpy(HB + o_m12, m12_inout, size_t(n1) * 4);
        std::memset(HB + o_m12 + size_t(n1) * 4, 0, 4);
        std::memcpy(HB + o_job, &job, sizeof(job));
        if (phase == EXEC_PACK) return PLM_OK;
    }

    CU_TRY(cudaMemcpyAsync(DB, HB, in_bytes, cudaMemcpyHostToDevice, ctx->stream));

    gp.grid_rows = grid_rows;
    gp.grid_cols = grid_cols;
    gp.best_lr = best_lr ? 1 : 0;
    gp.ratio = ratio;
    gp.line_sim_th = line_sim_th;
    if (rows_cluster) {
        gp.m21key = reinterpret_cast<unsigned long long *>(DB + o_m21key);
        st = launch_grid_rows_cluster(ctx, job, gp, n_cta, map_smem);
    } else if (fused && n1 >= 64 && g_grid_cluster) {
        st = launch_grid_cluster(ctx, reinterpret_cast<const plm::GridJob *>(DB + o_job), 1, gp, n1, std::max(n2, 1),
                                 std::max(n_items, 1), is_lines != 0);
    } else if (fused) {
        st = launch_grid_fused(ctx, reinterpret_cast<const plm::GridJob *>(DB + o_job), 1, gp, n1, std::max(n2, 1), std::max(n_items, 1), is_lines != 0);
    } else {
        map_grid_handover_bind(gp, DB + o_handover, warps, n_cta, best_lr != 0);
        st = launch_grid_chunked(ctx, DB, job, gp, o_cta_min, o_m21key, o_m21, warps, n_cta, map_smem);
    }
    if (st != PLM_OK) return st;
    CU_TRY(cudaMemcpyAsync(HB + o_m12, DB + o_m12, size_t(n1) * 4 + 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (phase == EXEC_LAUNCH) return PLM_OK;
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    std::memcpy(m12_inout, HB + o_m12, size_t(n1) * 4);
    int32_t cnt;
    std::memcpy(&cnt, HB + o_m12 + size_t(n1) * 4, 4);
    *n_matches = cnt;
    return PLM_OK;
}

} // namespace

PLM_API int plm_match_grid_points(plm_ctx *ctx, const int32_t *xy, const uint8_t *d1, int n1, size_t step1,
                                  const int32_t *cell_start, const int32_t *cell_items, int grid_rows, int grid_cols,
                                  const uint8_t *d2, int n2, size_t step2, const int32_t win[4], double ratio, int best_lr,
                                  int32_t *m12_inout, int *n_matches) {
    return match_grid_impl(ctx, 0, xy, d1, n1, step1, cell_start, cell_items, grid_rows, grid_cols, d2, n2, step2, nullptr,
                           0.0, win, ratio, best_lr, m12_inout, n_matches);
}

PLM_API int plm_match_grid_lines(plm_ctx *ctx, const int32_t *xyxy, const uint8_t *d1, int n1, size_t step1,
                                 const int32_t *cell_start, const int32_t *cell_items, int grid_rows, int grid_cols,
                                 const uint8_t *d2, int n2, size_t step2, const double *dirs2, double line_sim_th,
                                 const int32_t win[4], double ratio, int best_lr, int32_t *m12_inout, int *n_matches) {
    return match_grid_impl(ctx, 1, xyxy, d1, n1, step1, cell_start, cell_items, grid_rows, grid_cols, d2, n2, step2, dirs2,
                           line_sim_th, win, ratio, best_lr, m12_inout, n_matches);
}

// ---------------------------------------------------------------------------------------------
// Row-sharded matchGrid on device-resident data
namespace {

int dev_grid_setup(plm_ctx *&ctx, const plm_dev_grid_args *a, plm::GridJob &job, plm::GridParams &gp, int &warps, int &n_cta,
                   size_t &smem, size_t extra_bytes = 0, char **extra = nullptr) {
    if (!a) return fail(PLM_E_INVALID, "null args");
    if (a->n1 < 0 || a->n2 < 0) return fail(PLM_E_INVALID, "negative size");
    if (a->grid_rows <= 0 || a->grid_cols <= 0) return fail(PLM_E_GRID, "[GridStructure] invalid dimension");
    if (a->ratio > 1.0) return fail(PLM_E_RATIO, plm_status_string(PLM_E_RATIO));
    if (a->n2 > GRID_N2_MAX) return fail(PLM_E_UNSUPPORTED, "matchGrid supports at most 32768 train features");
    if (a->n1 > 0 && (!a->coords || !a->d1 || !a->m12_inout || !a->count)) return fail(PLM_E_INVALID, "null pointer");
    if (!a->cell_start || (a->n2 > 0 && !a->d2) || (a->is_lines && a->n2 > 0 && !a->dirs2)) return fail(PLM_E_INVALID, "null pointer");
    if ((reinterpret_cast<uintptr_t>(a->d1) | reinterpret_cast<uintptr_t>(a->d2)) & 15)
        return fail(PLM_E_INVALID, "device descriptor pointers must be 16-byte aligned");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    std::memset(&job, 0, sizeof(job));
    job.coords = a->coords;
    job.d1 = static_cast<const uint4 *>(a->d1);
    job.cell_start = a->cell_start;
    job.cell_items = a->cell_items;
    job.d2 = static_cast<const uint4 *>(a->d2);
    job.dirs2 = a->dirs2;
    job.m12 = a->m12_inout;
    job.count = a->count;
    job.n1 = a->n1;
    job.n2 = a->n2;
    job.is_lines = a->is_lines ? 1 : 0;
    for (int i = 0; i < 4; ++i) job.win[i] = a->win[i];
    job.i1_base = a->i1_base;
    std::memset(&gp, 0, sizeof(gp));
    gp.grid_rows = a->grid_rows;
    gp.grid_cols = a->grid_cols;
    gp.best_lr = a->best_lr ? 1 : 0;
    gp.ratio = a->ratio;
    gp.line_sim_th = a->line_sim_th;
    if ((st = plan_map_grid(ctx, a->n1, a->n2, a->grid_rows * a->grid_cols, a->is_lines != 0, gp, warps, n_cta, smem)) != PLM_OK) return st;
    const size_t cta_min_bytes = align_up(size_t(std::max(n_cta, 1)) * std::max(a->n2, 1) * 2);
    const size_t handover = map_grid_handover_bytes(warps, n_cta, gp.rows_per_cta);
    st = ctx->ensure_device(cta_min_bytes + handover + extra_bytes);
    if (st != PLM_OK) return st;
    gp.cta_min = reinterpret_cast<uint16_t *>(ctx->d_buf);
    map_grid_handover_bind(gp, ctx->d_buf + cta_min_bytes, warps, n_cta, gp.best_lr != 0);
    if (extra) *extra = ctx->d_buf + cta_min_bytes + handover;
    return PLM_OK;
}

} // namespace

PLM_API int plm_dev_grid_colmin(plm_ctx *ctx, const plm_dev_grid_args *a, uint16_t *col_min_dev) {
    plm::GridJob job;
    plm::GridParams gp;
    int warps = 0, n_cta = 0;
    size_t smem = 0;
    int st = dev_grid_setup(ctx, a, job, gp, warps, n_cta, smem);
    if (st != PLM_OK) return st;
    if (a->n2 == 0) return PLM_OK;
    if (!col_min_dev) return fail(PLM_E_INVALID, "null col_min");
    if (!gp.best_lr || n_cta == 0) {
        CU_TRY(cudaMemsetAsync(col_min_dev, 0xFF, size_t(a->n2) * 2, ctx->stream));
        return PLM_OK;
    }
    if ((st = launch_map_grid(ctx, 0, job, gp, warps, n_cta, smem)) != PLM_OK) return st;
    plm::grid_scan_kernel<<<(a->n2 + 3) / 4, 128, 0, ctx->stream>>>(gp.cta_min, n_cta, a->n2, nullptr, col_min_dev);
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    return PLM_OK;
}

PLM_API int plm_dev_grid_match(plm_ctx *ctx, const plm_dev_grid_args *a, const uint16_t *seed_dev, uint64_t *m21key_dev) {
    plm::GridJob job;
    plm::GridParams gp;
    int warps = 0, n_cta = 0;
    size_t smem = 0;
    int st = dev_grid_setup(ctx, a, job, gp, warps, n_cta, smem);
    if (st != PLM_OK) return st;
    if (gp.best_lr && a->n2 > 0 && !m21key_dev) return fail(PLM_E_INVALID, "null m21key");
    gp.m21key = reinterpret_cast<unsigned long long *>(m21key_dev);
    if (gp.best_lr && a->n2 > 0) CU_TRY(cudaMemsetAsync(m21key_dev, 0xFF, size_t(a->n2) * 8, ctx->stream));
    if (n_cta == 0 || a->n2 == 0) return PLM_OK;
    if (gp.best_lr) {
        if ((st = launch_map_grid(ctx, 0, job, gp, warps, n_cta, smem)) != PLM_OK) return st;
        plm::grid_scan_kernel<<<(a->n2 + 3) / 4, 128, 0, ctx->stream>>>(gp.cta_min, n_cta, a->n2, seed_dev, nullptr);
        ctx->launches++;
        CU_TRY(cudaGetLastError());
    }
    return launch_map_grid(ctx, 1, job, gp, warps, n_cta, smem);
}

// The complete matchGrid of device-resident rows against one frame on ONE device, as one call: pass 0 (which also
// initialises the fresh match vector, the count and the per-column keys), scan, pass 1, mutual check from the keys --
// four launches back to back, nothing else on the stream.
PLM_API int plm_dev_match_grid(plm_ctx *ctx, const plm_dev_grid_args *a, int fresh) {
    plm::GridJob job;
    plm::GridParams gp;
    int warps = 0, n_cta = 0;
    size_t smem = 0;
    char *X = nullptr;
    int st = dev_grid_setup(ctx, a, job, gp, warps, n_cta, smem, align_up(size_t(std::max(a ? a->n2 : 0, 1)) * 8), &X);
    if (st != PLM_OK) return st;
    if (a->n1 == 0) {
        if (fresh && a->count) CU_TRY(cudaMemsetAsync(a->count, 0, 4, ctx->stream));
        return PLM_OK;
    }
    gp.m21key = reinterpret_cast<unsigned long long *>(X);
    const bool two_pass = gp.best_lr && a->n2 > 0 && n_cta > 0;
    if (two_pass && warps == 0) {
        gp.init_flags = 4 | (fresh ? 3 : 0);
    } else {
        if (fresh) {
            CU_TRY(cudaMemsetAsync(a->m12_inout, 0xFF, size_t(a->n1) * 4, ctx->stream));
            CU_TRY(cudaMemsetAsync(a->count, 0, 4, ctx->stream));
        }
        if (two_pass) CU_TRY(cudaMemsetAsync(gp.m21key, 0xFF, size_t(a->n2) * 8, ctx->stream));
    }
    if (n_cta == 0) return PLM_OK;
    if (a->n2 > 0) {
        if (two_pass) {
            if ((st = launch_map_grid(ctx, 0, job, gp, warps, n_cta, smem)) != PLM_OK) return st;
            plm::grid_scan_kernel<<<(a->n2 + 3) / 4, 128, 0, ctx->stream>>>(gp.cta_min, n_cta, a->n2, nullptr, nullptr);
            ctx->launches++;
            CU_TRY(cudaGetLastError());
        }
        if ((st = launch_map_grid(ctx, 1, job, gp, warps, n_cta, smem)) != PLM_OK) return st;
    }
    if (gp.best_lr) { // mutual check (matching.cpp:166-174), stale entries included
        plm::cross_check_keys_kernel<<<(a->n1 + 127) / 128, 128, 0, ctx->stream>>>(a->m12_inout, a->n1, a->i1_base, gp.m21key, a->n2, a->count);
        ctx->launches++;
        CU_TRY(cudaGetLastError());
    }
    return PLM_OK;
}

namespace {

size_t sharded_grid_extra_bytes(int n2) {
    const size_t n2p8 = (size_t(n2) + 7) / 8 * 8, n2p2 = (size_t(n2) + 1) / 2 * 2;
    Layout L;
    L.add(n2p8 * 2); L.add(n2p8 * 2); L.add(n2p2 * 8); L.add(n2p2 * 8); L.add(size_t(std::max(n2, 1)) * 4);
    return L.total;
}

// Everything plm_dev_sharded_match_grid / plm_dev_sharded_match may allocate, done up front: an in-process caller
// driving several devices (plm_shard_*) sizes every context before the first kernel that waits for a peer is enqueued.
int plm_dev_sharded_match_grid_prepare(plm_ctx *ctx, const plm_dev_grid_args *a) {
    plm::GridJob job;
    plm::GridParams gp;
    int warps = 0, n_cta = 0;
    size_t smem = 0;
    char *X = nullptr;
    return dev_grid_setup(ctx, a, job, gp, warps, n_cta, smem, sharded_grid_extra_bytes(a ? std::max(a->n2, 0) : 0), &X);
}

int plm_dev_sharded_match_prepare(plm_ctx *ctx, int n1, int n2) {
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    Layout A;
    A.add(size_t(std::max(n1, 1)) * 16); A.add(size_t(n2) * 16); A.add(size_t(n2) * 4); A.add(16);
    if ((st = ctx->ensure_aux(A.total)) != PLM_OK) return st;
    size_t need = 0;
    for (int dir = 0; dir < 2; ++dir) {
        Layout L;
        plm::KnnTask t;
        KnnPlan plan;
        size_t off = 0;
        build_knn_task(ctx, L, t, plan, nullptr, dir ? n2 : n1, nullptr, dir ? n1 : n2, 0, off);
        need = std::max(need, L.total);
    }
    return ctx->ensure_device(need);
}

} // namespace

// The whole row-sharded matchGrid of one rank, launched back to back from C: minima pass, the two peer-memory
// reductions around the match pass, mutual check and the peer-memory all-gather of the match vectors.
PLM_API int plm_dev_sharded_match_grid(plm_ctx *ctx, const plm_dev_grid_args *a, const plm_peer_group *g, int64_t n_rows_total,
                                       int32_t *m12_global_dev, int32_t *count_global_dev, int32_t *error_dev) {
    if (!g || !g->xchg || !g->gather || !m12_global_dev || !count_global_dev || !error_dev) return fail(PLM_E_INVALID, "null pointer");
    if (g->world < 2 || g->world > PLM_PEER_MAX_RANKS || g->rank < 0 || g->rank >= g->world) return fail(PLM_E_INVALID, "bad rank / world");
    plm::GridJob job;
    plm::GridParams gp;
    int warps = 0, n_cta = 0;
    size_t smem = 0;
    const int n2 = a ? std::max(a->n2, 0) : 0;
    const size_t n2p8 = (size_t(n2) + 7) / 8 * 8, n2p2 = (size_t(n2) + 1) / 2 * 2;
    Layout L;
    const size_t o_colmin = L.add(n2p8 * 2), o_seed = L.add(n2p8 * 2), o_key = L.add(n2p2 * 8), o_keyg = L.add(n2p2 * 8),
                 o_m21 = L.add(size_t(std::max(n2, 1)) * 4);
    char *X = nullptr;
    int st = dev_grid_setup(ctx, a, job, gp, warps, n_cta, smem, L.total, &X);
    if (st != PLM_OK) return st;
    if (n_rows_total > g->n_rows_cap || a->i1_base < 0 || a->i1_base + a->n1 > n_rows_total) return fail(PLM_E_INVALID, "rows outside the gather buffers");
    if (n2 > 0 && (n2p8 / 8 > size_t(g->q_cap) || n2p2 / 2 > size_t(g->q_cap))) return fail(PLM_E_UNSUPPORTED, "frame too large for the exchange buffers");
    uint16_t *col_min = reinterpret_cast<uint16_t *>(X + o_colmin), *seed = reinterpret_cast<uint16_t *>(X + o_seed);
    uint64_t *key = reinterpret_cast<uint64_t *>(X + o_key), *key_g = reinterpret_cast<uint64_t *>(X + o_keyg);
    int32_t *m21 = reinterpret_cast<int32_t *>(X + o_m21);
    uint32_t epoch = g->xchg_epoch;
    if (gp.best_lr && n2 > 0) {
        CU_TRY(cudaMemsetAsync(X, 0xFF, L.total, ctx->stream)); // identities of both reductions, absent keys, m21 = -1
        if (n_cta > 0) {
            if ((st = launch_map_grid(ctx, 0, job, gp, warps, n_cta, smem)) != PLM_OK) return st;
            plm::grid_scan_kernel<<<(n2 + 3) / 4, 128, 0, ctx->stream>>>(gp.cta_min, n_cta, n2, nullptr, col_min);
            ctx->launches++;
            CU_TRY(cudaGetLastError());
        }
        // running column minima of the lower-ranked shards
        if ((st = plm_dev_peer_reduce(ctx, g->xchg, g->rank, g->world, g->q_cap, epoch++, PLM_PEER_PREFIX_MIN_U16, col_min,
                                      static_cast<int>(n2p8 / 8), seed, error_dev)) != PLM_OK)
            return st;
        if (n_cta > 0) {
            const long long cells = static_cast<long long>(n_cta) * n2;
            plm::grid_seed_kernel<<<static_cast<int>((cells + 255) / 256), 256, 0, ctx->stream>>>(gp.cta_min, n_cta, n2, seed);
            ctx->launches++;
            CU_TRY(cudaGetLastError());
        }
    }
    gp.m21key = reinterpret_cast<unsigned long long *>(key);
    if (n_cta > 0 && n2 > 0 && (st = launch_map_grid(ctx, 1, job, gp, warps, n_cta, smem)) != PLM_OK) return st;
    if (gp.best_lr && n2 > 0) {
        // per-column best pairs over all shards, then the mutual check on this shard's rows
        if ((st = plm_dev_peer_reduce(ctx, g->xchg, g->rank, g->world, g->q_cap, epoch++, PLM_PEER_MIN_U64, key,
                                      static_cast<int>(n2p2 / 2), key_g, error_dev)) != PLM_OK)
            return st;
        (void)m21;
        if (a->n1 > 0) {
            plm::cross_check_keys_kernel<<<(a->n1 + 255) / 256, 256, 0, ctx->stream>>>(a->m12_inout, a->n1, a->i1_base, reinterpret_cast<const unsigned long long *>(key_g), n2, a->count);
            ctx->launches++;
            CU_TRY(cudaGetLastError());
        }
    }
    return plm_dev_peer_allgather_i32(ctx, g->gather, g->rank, g->world, g->n_rows_cap, g->gather_epoch, a->m12_inout, a->i1_base,
                                      a->n1, n_rows_total, a->count, m12_global_dev, count_global_dev, error_dev);
}

// The row-sharded StVO::match of one rank (the brute-force fallback of matchMap2KF*, mapHandler.cpp:645-650) in one
// call: 12 direction local, 21 direction through the peer-memory top-2 exchange, mutual check, all-gather.
PLM_API int plm_dev_sharded_match(plm_ctx *ctx, const void *d1_shard_dev, int n1, int64_t i1_base, const void *d2_dev, int n2,
                                  float nnr, int best_lr, int32_t *m12_local_inout_dev, const plm_peer_group *g,
                                  int64_t n_rows_total, int32_t *m12_global_dev, int32_t *count_global_dev, int32_t *error_dev) {
    if (!g || !g->xchg || !g->gather || !m12_global_dev || !count_global_dev || !error_dev) return fail(PLM_E_INVALID, "null pointer");
    if (g->world < 2 || g->world > PLM_PEER_MAX_RANKS || g->rank < 0 || g->rank >= g->world) return fail(PLM_E_INVALID, "bad rank / world");
    if (n1 < 0 || n2 < 0 || i1_base < 0 || i1_base + n1 > n_rows_total || n_rows_total > g->n_rows_cap)
        return fail(PLM_E_INVALID, "rows outside the gather buffers");
    if (n1 > 0 && (!d1_shard_dev || !m12_local_inout_dev)) return fail(PLM_E_INVALID, "null pointer");
    if (n2 < 1) return fail(PLM_E_TRAIN, plm_status_string(PLM_E_TRAIN)); // empty train set: the reference throws (matching.cpp:50-51)
    if (n2 > g->q_cap) return fail(PLM_E_UNSUPPORTED, "frame too large for the exchange buffers");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    Layout L;
    const size_t o_top12 = L.add(size_t(std::max(n1, 1)) * 16), o_part = L.add(size_t(n2) * 16), o_m21 = L.add(size_t(n2) * 4),
                 o_cnt = L.add(16);
    if ((st = ctx->ensure_aux(L.total)) != PLM_OK) return st;
    char *X = ctx->d_aux;
    uint64_t *top12 = reinterpret_cast<uint64_t *>(X + o_top12), *part = reinterpret_cast<uint64_t *>(X + o_part);
    int32_t *m21 = reinterpret_cast<int32_t *>(X + o_m21), *cnt = reinterpret_cast<int32_t *>(X + o_cnt);
    CU_TRY(cudaMemsetAsync(cnt, 0, 4, ctx->stream));
    // direction 12: this shard's rows against the whole frame are final locally
    if (n1 > 0) {
        if ((st = plm_dev_knn2(ctx, d1_shard_dev, n1, d2_dev, n2, 0, top12)) != PLM_OK) return st;
        if ((st = plm_dev_nnr_accept(ctx, top12, n1, nnr, m12_local_inout_dev, cnt)) != PLM_OK) return st;
    }
    if (best_lr) {
        // direction 21: per-shard top-2 with global map indices -> push / wait / merge / ratio test in one kernel
        CU_TRY(cudaMemsetAsync(part, 0xFF, size_t(n2) * 16, ctx->stream)); // an empty shard contributes absent keys
        CU_TRY(cudaMemsetAsync(m21, 0xFF, size_t(n2) * 4, ctx->stream));
        if (n1 > 0 && (st = plm_dev_knn2(ctx, d2_dev, n2, d1_shard_dev, n1, static_cast<uint64_t>(i1_base), part)) != PLM_OK) return st;
        if ((st = plm_dev_top2_exchange(ctx, g->xchg, g->rank, g->world, g->q_cap, g->xchg_epoch, part, n2, nullptr, nnr, m21, nullptr,
                                        error_dev)) != PLM_OK)
            return st;
        if (n1 > 0 && (st = plm_dev_cross_check(ctx, m12_local_inout_dev, n1, i1_base, m21, n2, cnt)) != PLM_OK) return st;
    }
    return plm_dev_peer_allgather_i32(ctx, g->gather, g->rank, g->world, g->n_rows_cap, g->gather_epoch, m12_local_inout_dev, i1_base,
                                      n1, n_rows_total, cnt, m12_global_dev, count_global_dev, error_dev);
}

PLM_API int plm_dev_m21_from_keys(plm_ctx *ctx, const uint64_t *m21key_dev, int n2, int32_t *m21_dev) {
    if (n2 < 0) return fail(PLM_E_INVALID, "negative size");
    if (n2 == 0) return PLM_OK;
    if (!m21key_dev || !m21_dev) return fail(PLM_E_INVALID, "null pointer");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    plm::m21_from_keys_kernel<<<(n2 + 127) / 128, 128, 0, ctx->stream>>>(reinterpret_cast<const unsigned long long *>(m21key_dev), n2, m21_dev);
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    return PLM_OK;
}

PLM_API int plm_line_pair_filter(plm_ctx *ctx, const float *ln1, int n1, const float *ln2, int n2, const int32_t *m12,
                                 double overlap_th, double line_sim_th, uint8_t *keep, double *overlap, double *sim, int *n_kept) {
    if (n1 < 0 || n2 < 0) return fail(PLM_E_INVALID, "negative size");
    if (!n_kept) return fail(PLM_E_INVALID, "null n_kept");
    *n_kept = 0;
    if (n1 == 0) return PLM_OK;
    if (!ln1 || !m12 || !keep || !overlap || !sim || (n2 > 0 && !ln2)) return fail(PLM_E_INVALID, "null pointer");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    Layout L;
    const size_t o_l1 = L.add(size_t(n1) * 16), o_l2 = L.add(size_t(std::max(n2, 1)) * 16), o_m = L.add(size_t(n1) * 4);
    const size_t in_bytes = L.total;
    const size_t o_ov = L.add(size_t(n1) * 8), o_sim = L.add(size_t(n1) * 8), o_keep = L.add(size_t(n1)), o_cnt = L.add(4);
    if ((st = ctx->ensure_pinned(L.total)) != PLM_OK) return st;
    if ((st = ctx->ensure_device(L.total)) != PLM_OK) return st;
    char *H = ctx->h_buf, *D = ctx->d_buf;
    std::memcpy(H + o_l1, ln1, size_t(n1) * 16);
    if (n2 > 0) std::memcpy(H + o_l2, ln2, size_t(n2) * 16);
    std::memcpy(H + o_m, m12, size_t(n1) * 4);
    CU_TRY(cudaMemcpyAsync(D, H, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(cudaMemsetAsync(D + o_cnt, 0, 4, ctx->stream));
    plm::line_pair_filter_kernel<<<(n1 + 127) / 128, 128, 0, ctx->stream>>>(
        reinterpret_cast<const float4 *>(D + o_l1), n1, reinterpret_cast<const float4 *>(D + o_l2), n2,
        reinterpret_cast<const int32_t *>(D + o_m), overlap_th, line_sim_th, reinterpret_cast<uint8_t *>(D + o_keep),
        reinterpret_cast<double *>(D + o_ov), reinterpret_cast<double *>(D + o_sim), reinterpret_cast<int32_t *>(D + o_cnt));
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(H + o_ov, D + o_ov, L.total - o_ov, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    std::memcpy(overlap, H + o_ov, size_t(n1) * 8);
    std::memcpy(sim, H + o_sim, size_t(n1) * 8);
    std::memcpy(keep, H + o_keep, size_t(n1));
    int32_t cnt;
    std::memcpy(&cnt, H + o_cnt, 4);
    *n_kept = cnt;
    return PLM_OK;
}

// ---------------------------------------------------------------------------------------------
// Map landmarks: MapPoint / MapLine::updateAverageDescDir (src/mapFeatures.cpp:51-93, :121-163)
namespace {

// Both launches of a batch; `work` (1 + n_lm int32) is scratch for the list of long observation lists.
int launch_med_desc(plm_ctx *ctx, plm::MedArgs a) {
    CU_TRY(cudaMemsetAsync(a.work, 0, 4, ctx->stream));
    const int per_cta = 32 * plm::MED_WARPS; // a warp takes a chunk of 32 landmarks at a time
    const int ctas = std::min((a.n_lm + per_cta - 1) / per_cta, ctx->sm_count * 32);
    plm::med_desc_warp_kernel<<<ctas, 32 * plm::MED_WARPS, 0, ctx->stream>>>(a);
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    plm::med_desc_cta_kernel<<<ctx->sm_count * 2, plm::MED_CTA_THREADS, 0, ctx->stream>>>(a);
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    return PLM_OK;
}

} // namespace

PLM_API int plm_dev_med_desc(plm_ctx *ctx, const void *desc_obs_dev, int64_t n_obs, const double *dir_obs_dev,
                             const int32_t *obs_start_dev, int n_lm, int32_t *med_idx_dev, void *med_desc_dev,
                             const int32_t *dst_rows_dev, double *med_dir_dev) {
    if (n_lm < 0 || n_obs < 0) return fail(PLM_E_INVALID, "negative size");
    if (n_lm == 0) return PLM_OK;
    if (!obs_start_dev || !med_idx_dev || (n_obs > 0 && !desc_obs_dev)) return fail(PLM_E_INVALID, "null pointer");
    if ((reinterpret_cast<uintptr_t>(desc_obs_dev) | reinterpret_cast<uintptr_t>(med_desc_dev)) & 15)
        return fail(PLM_E_INVALID, "descriptor rows must be 16-byte aligned");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    if ((st = ctx->ensure_device(size_t(n_lm + 1) * 4)) != PLM_OK) return st;
    plm::MedArgs a{};
    a.desc = static_cast<const uint4 *>(desc_obs_dev);
    a.dirs = dir_obs_dev;
    a.obs_start = obs_start_dev;
    a.n_obs = n_obs;
    a.n_lm = n_lm;
    a.med_idx = med_idx_dev;
    a.med_desc = static_cast<uint4 *>(med_desc_dev);
    a.dst_rows = dst_rows_dev;
    a.med_dir = med_dir_dev;
    a.work = reinterpret_cast<int32_t *>(ctx->d_buf);
    return launch_med_desc(ctx, a);
}

PLM_API int plm_med_desc(plm_ctx *ctx, const uint8_t *desc_obs, int64_t n_obs, size_t step, const double *dir_obs,
                         const int32_t *obs_start, int n_lm, int32_t *med_idx, uint8_t *med_desc, double *med_dir) {
    if (n_lm < 0 || n_obs < 0) return fail(PLM_E_INVALID, "negative size");
    if (n_lm == 0) return PLM_OK;
    if (!obs_start || !med_idx || (n_obs > 0 && !desc_obs)) return fail(PLM_E_INVALID, "null pointer");
    if (step < 32) return fail(PLM_E_INVALID, "step < 32");
    if (n_obs > INT32_MAX) return fail(PLM_E_UNSUPPORTED, "more than 2^31 - 1 observations in one call");
    if (obs_start[0] < 0 || obs_start[n_lm] > n_obs) return fail(PLM_E_INVALID, "obs_start outside [0, n_obs]");
    for (int l = 0; l < n_lm; ++l)
        if (obs_start[l + 1] < obs_start[l]) return fail(PLM_E_INVALID, "obs_start must be non-decreasing");
    const bool want_dir = med_dir != nullptr && dir_obs != nullptr;
    if (med_dir && !dir_obs) return fail(PLM_E_INVALID, "med_dir requested without dir_obs");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    Layout L;
    const size_t o_start = L.add(size_t(n_lm + 1) * 4);
    const size_t o_desc = L.add(size_t(n_obs) * 32);
    const size_t o_dirs = L.add(want_dir ? size_t(n_obs) * 24 : 0);
    const size_t in_bytes = L.total;
    const size_t o_idx = L.add(size_t(n_lm) * 4);
    const size_t o_med = L.add(med_desc ? size_t(n_lm) * 32 : 0);
    const size_t o_mdir = L.add(want_dir ? size_t(n_lm) * 24 : 0);
    const size_t out_end = L.total;
    const size_t o_work = L.add(size_t(n_lm + 1) * 4);
    if ((st = ctx->ensure_pinned(out_end)) != PLM_OK) return st;
    if ((st = ctx->ensure_device(L.total)) != PLM_OK) return st;
    std::memcpy(ctx->h_buf + o_start, obs_start, size_t(n_lm + 1) * 4);
    pack_rows(ctx->h_buf + o_desc, desc_obs, n_obs, step);
    if (want_dir) std::memcpy(ctx->h_buf + o_dirs, dir_obs, size_t(n_obs) * 24);
    CU_TRY(cudaMemcpyAsync(ctx->d_buf, ctx->h_buf, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    plm::MedArgs a{};
    a.desc = reinterpret_cast<const uint4 *>(ctx->d_buf + o_desc);
    a.dirs = want_dir ? reinterpret_cast<const double *>(ctx->d_buf + o_dirs) : nullptr;
    a.obs_start = reinterpret_cast<const int32_t *>(ctx->d_buf + o_start);
    a.n_obs = n_obs;
    a.n_lm = n_lm;
    a.med_idx = reinterpret_cast<int32_t *>(ctx->d_buf + o_idx);
    a.med_desc = med_desc ? reinterpret_cast<uint4 *>(ctx->d_buf + o_med) : nullptr;
    a.dst_rows = nullptr;
    a.med_dir = want_dir ? reinterpret_cast<double *>(ctx->d_buf + o_mdir) : nullptr;
    a.work = reinterpret_cast<int32_t *>(ctx->d_buf + o_work);
    if ((st = launch_med_desc(ctx, a)) != PLM_OK) return st;
    CU_TRY(cudaMemcpyAsync(ctx->h_buf + o_idx, ctx->d_buf + o_idx, out_end - o_idx, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    std::memcpy(med_idx, ctx->h_buf + o_idx, size_t(n_lm) * 4);
    if (med_desc) std::memcpy(med_desc, ctx->h_buf + o_med, size_t(n_lm) * 32);
    if (want_dir) std::memcpy(med_dir, ctx->h_buf + o_mdir, size_t(n_lm) * 24);
    return PLM_OK;
}

// ---------------------------------------------------------------------------------------------
// Top-2 exchange over NVLink peer memory (csrc/plm_peer.cuh)
namespace {
inline int peer_blocks_cap(int q_cap) { return (q_cap + plm::PEER_THREADS - 1) / plm::PEER_THREADS; }
} // namespace

PLM_API size_t plm_peer_buffer_bytes(int world, int q_cap) {
    if (world <= 0 || q_cap <= 0) return 0;
    return plm::peer_buffer_bytes(world, q_cap, peer_blocks_cap(q_cap));
}

PLM_API size_t plm_peer_gather_bytes(int world, int64_t n_rows_cap) {
    if (world <= 0 || n_rows_cap <= 0) return 0;
    return plm::peer_gather_bytes(world, n_rows_cap);
}

PLM_API int plm_peer_alloc(plm_ctx *ctx, int world, int q_cap, void **buf_dev, uint8_t handle[PLM_PEER_HANDLE_BYTES]) {
    if (world <= 0 || world > PLM_PEER_MAX_RANKS || q_cap <= 0) return fail(PLM_E_INVALID, "world in 1..16 and q_cap > 0 required");
    return plm_peer_alloc_bytes(ctx, plm_peer_buffer_bytes(world, q_cap), buf_dev, handle);
}

PLM_API int plm_peer_alloc_bytes(plm_ctx *ctx, size_t bytes, void **buf_dev, uint8_t handle[PLM_PEER_HANDLE_BYTES]) {
    static_assert(sizeof(cudaIpcMemHandle_t) == PLM_PEER_HANDLE_BYTES, "IPC handle size");
    if (!buf_dev || !handle) return fail(PLM_E_INVALID, "null pointer");
    *buf_dev = nullptr;
    if (bytes == 0) return fail(PLM_E_INVALID, "empty buffer");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    void *p = nullptr;
    CU_TRY(cudaMalloc(&p, bytes));
    cudaError_t e = cudaMemsetAsync(p, 0, bytes, ctx->stream); // flags start at epoch 0 = "nothing arrived"
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        cudaFree(p);
        return fail(PLM_E_CUDA, std::string("plm_peer_alloc: ") + cudaGetErrorString(e));
    }
    std::memcpy(handle, &h, sizeof(h));
    *buf_dev = p;
    return PLM_OK;
}

PLM_API int plm_peer_open(plm_ctx *ctx, const uint8_t handle[PLM_PEER_HANDLE_BYTES], void **buf_dev) {
    if (!buf_dev || !handle) return fail(PLM_E_INVALID, "null pointer");
    *buf_dev = nullptr;
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof(h));
    CU_TRY(cudaIpcOpenMemHandle(buf_dev, h, cudaIpcMemLazyEnablePeerAccess));
    return PLM_OK;
}

PLM_API int plm_peer_close(plm_ctx *ctx, void *buf_dev) {
    if (!buf_dev) return PLM_OK;
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    CU_TRY(cudaIpcCloseMemHandle(buf_dev));
    return PLM_OK;
}

PLM_API int plm_peer_free(plm_ctx *ctx, void *buf_dev) {
    if (!buf_dev) return PLM_OK;
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    CU_TRY(cudaFree(buf_dev));
    return PLM_OK;
}

// Single-GPU emulation of the peer kernels (see csrc/plm_peer.cuh): calls are recorded per thread, then run as ONE
// cooperative launch with blockIdx.y = rank.
namespace {
struct PeerEmu {
    int world = 0;   // > 0 while recording
    int kind = -1;   // 0 exchange, 1 min_u64, 2 prefix_min_u16, 3 gather
    int grid_x = 0;
    int n = 0;
    plm::PeerEmuExchange ex;
    plm::PeerEmuGather ga;
};
thread_local PeerEmu g_emu;

int emu_record_exchange(int kind, const plm::PeerExchangeArgs &a, int grid) {
    if (g_emu.n >= g_emu.world || g_emu.n >= plm::PEER_EMU_MAX_RANKS) return fail(PLM_E_INVALID, "peer emulation: more calls than ranks");
    if (g_emu.n > 0 && (g_emu.kind != kind || g_emu.grid_x != grid)) return fail(PLM_E_INVALID, "peer emulation: the recorded calls differ in kind or size");
    g_emu.kind = kind;
    g_emu.grid_x = grid;
    g_emu.ex.a[g_emu.n++] = a;
    return PLM_OK;
}
} // namespace

PLM_API int plm_peer_emulate_begin(int world) {
    if (world < 1 || world > plm::PEER_EMU_MAX_RANKS) return fail(PLM_E_INVALID, "peer emulation supports 1 .. 4 ranks");
    g_emu = PeerEmu();
    g_emu.world = world;
    return PLM_OK;
}

PLM_API int plm_peer_emulate_run(plm_ctx *ctx) {
    PeerEmu e = g_emu;
    g_emu = PeerEmu();
    if (e.world == 0) return fail(PLM_E_INVALID, "peer emulation: no recording in progress");
    if (e.n == 0) return PLM_OK;
    if (e.n != e.world) return fail(PLM_E_INVALID, "peer emulation: every rank must have recorded its call");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    const dim3 grid(e.grid_x, e.world, 1);
    void *params[1];
    cudaError_t err;
    if (e.kind == 3) {
        params[0] = &e.ga;
        err = cudaLaunchCooperativeKernel(reinterpret_cast<const void *>(plm::peer_emu_gather_kernel), grid, dim3(256), params, 0, ctx->stream);
    } else {
        params[0] = &e.ex;
        const void *fn = e.kind == 0 ? reinterpret_cast<const void *>(plm::peer_emu_exchange_kernel<0>)
                         : e.kind == 1 ? reinterpret_cast<const void *>(plm::peer_emu_exchange_kernel<1>)
                                       : reinterpret_cast<const void *>(plm::peer_emu_exchange_kernel<2>);
        err = cudaLaunchCooperativeKernel(fn, grid, dim3(plm::PEER_THREADS), params, 0, ctx->stream);
    }
    if (err != cudaSuccess) return fail(PLM_E_CUDA, std::string("peer emulation (cooperative launch): ") + cudaGetErrorString(err));
    ctx->launches++;
    return PLM_OK;
}

PLM_API int plm_dev_top2_exchange(plm_ctx *ctx, void *const *peers, int rank, int world, int q_cap, uint32_t epoch,
                                  const uint64_t *local_top2_dev, int n1, uint64_t *top2_out_dev, float nnr,
                                  int32_t *m12_dev_inout, int32_t *count_dev, int32_t *error_dev) {
    if (world <= 0 || world > PLM_PEER_MAX_RANKS || rank < 0 || rank >= world) return fail(PLM_E_INVALID, "bad rank / world");
    if (n1 < 0 || n1 > q_cap || epoch == 0) return fail(PLM_E_INVALID, "n1 outside [0, q_cap] or epoch == 0");
    if (!peers || !error_dev || (n1 > 0 && !local_top2_dev)) return fail(PLM_E_INVALID, "null pointer");
    for (int r = 0; r < world; ++r)
        if (!peers[r]) return fail(PLM_E_INVALID, "null peer buffer");
    if (n1 == 0) return PLM_OK;
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    plm::PeerExchangeArgs a{};
    for (int r = 0; r < world; ++r) a.peer[r] = static_cast<unsigned char *>(peers[r]);
    a.rank = rank;
    a.world = world;
    a.q_cap = q_cap;
    a.blocks_cap = peer_blocks_cap(q_cap);
    a.epoch = epoch;
    a.local = reinterpret_cast<const ulonglong2 *>(local_top2_dev);
    a.n1 = n1;
    a.out = reinterpret_cast<ulonglong2 *>(top2_out_dev);
    a.nnr = nnr;
    a.m12 = m12_dev_inout;
    a.count = count_dev;
    a.error = error_dev;
    a.spin_limit = g_peer_spin_ticks;
    if (g_emu.world > 0) return emu_record_exchange(0, a, (n1 + plm::PEER_THREADS - 1) / plm::PEER_THREADS);
    plm::top2_exchange_merge_kernel<<<(n1 + plm::PEER_THREADS - 1) / plm::PEER_THREADS, plm::PEER_THREADS, 0, ctx->stream>>>(a);
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    return PLM_OK;
}

PLM_API int plm_dev_peer_allgather_i32(plm_ctx *ctx, void *const *peers, int rank, int world, int64_t n_rows_cap, uint32_t epoch,
                                       const int32_t *local_dev, int64_t row_lo, int64_t n_local, int64_t n_rows,
                                       const int32_t *local_count_dev, int32_t *out_dev, int32_t *out_count_dev,
                                       int32_t *error_dev) {
    if (world <= 0 || world > PLM_PEER_MAX_RANKS || rank < 0 || rank >= world) return fail(PLM_E_INVALID, "bad rank / world");
    if (epoch == 0 || n_rows < 0 || n_rows > n_rows_cap || row_lo < 0 || n_local < 0 || row_lo + n_local > n_rows)
        return fail(PLM_E_INVALID, "rows outside [0, n_rows_cap] or epoch == 0");
    if (!peers || !error_dev || (n_local > 0 && !local_dev) || (n_rows > 0 && !out_dev)) return fail(PLM_E_INVALID, "null pointer");
    for (int r = 0; r < world; ++r)
        if (!peers[r]) return fail(PLM_E_INVALID, "null peer buffer");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    plm::PeerGatherArgs a{};
    for (int r = 0; r < world; ++r) a.peer[r] = static_cast<unsigned char *>(peers[r]);
    a.rank = rank;
    a.world = world;
    a.n_rows_cap = n_rows_cap;
    a.epoch = epoch;
    a.local = local_dev;
    a.row_lo = row_lo;
    a.n_local = n_local;
    a.n_rows = n_rows;
    a.local_count = local_count_dev;
    a.out = out_dev;
    a.out_count = out_count_dev;
    a.error = error_dev;
    a.spin_limit = g_peer_spin_ticks;
    // every rank must launch the SAME grid size is not required (flags are per rank), but the grid must fit the device at
    // once so that no block waits behind spinning ones: at most one CTA per SM
    const int64_t work = std::max<int64_t>(std::max<int64_t>(n_rows, n_local), 1);
    const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((work + 1023) / 1024, ctx->sm_count)));
    if (g_emu.world > 0) {
        const int eg = std::max(1, std::min(grid, ctx->sm_count / std::max(1, g_emu.world))); // all ranks' CTAs must be co-resident
        if (g_emu.n >= g_emu.world || g_emu.n >= plm::PEER_EMU_MAX_RANKS) return fail(PLM_E_INVALID, "peer emulation: more calls than ranks");
        if (g_emu.n > 0 && (g_emu.kind != 3 || g_emu.grid_x != eg)) return fail(PLM_E_INVALID, "peer emulation: the recorded calls differ in kind or size");
        g_emu.kind = 3;
        g_emu.grid_x = eg;
        g_emu.ga.a[g_emu.n++] = a;
        return PLM_OK;
    }
    plm::peer_allgather_kernel<<<grid, 256, 0, ctx->stream>>>(a);
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    return PLM_OK;
}

PLM_API int plm_dev_peer_reduce(plm_ctx *ctx, void *const *peers, int rank, int world, int q_cap, uint32_t epoch, int op,
                                const void *src_dev, int n_chunks, void *out_dev, int32_t *error_dev) {
    if (world <= 0 || world > PLM_PEER_MAX_RANKS || rank < 0 || rank >= world) return fail(PLM_E_INVALID, "bad rank / world");
    if (n_chunks < 0 || n_chunks > q_cap || epoch == 0) return fail(PLM_E_INVALID, "n_chunks outside [0, q_cap] or epoch == 0");
    if (op != PLM_PEER_MIN_U64 && op != PLM_PEER_PREFIX_MIN_U16) return fail(PLM_E_INVALID, "unknown reduction");
    if (!peers || !error_dev || (n_chunks > 0 && (!src_dev || !out_dev))) return fail(PLM_E_INVALID, "null pointer");
    if ((reinterpret_cast<uintptr_t>(src_dev) | reinterpret_cast<uintptr_t>(out_dev)) & 15) return fail(PLM_E_INVALID, "16-byte alignment required");
    for (int r = 0; r < world; ++r)
        if (!peers[r]) return fail(PLM_E_INVALID, "null peer buffer");
    if (n_chunks == 0) return PLM_OK;
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    plm::PeerExchangeArgs a{};
    for (int r = 0; r < world; ++r) a.peer[r] = static_cast<unsigned char *>(peers[r]);
    a.rank = rank;
    a.world = world;
    a.q_cap = q_cap;
    a.blocks_cap = peer_blocks_cap(q_cap);
    a.epoch = epoch;
    a.local = static_cast<const ulonglong2 *>(src_dev);
    a.n1 = n_chunks;
    a.out = static_cast<ulonglong2 *>(out_dev);
    a.error = error_dev;
    a.spin_limit = g_peer_spin_ticks;
    const int grid = (n_chunks + plm::PEER_THREADS - 1) / plm::PEER_THREADS;
    if (g_emu.world > 0) return emu_record_exchange(op == PLM_PEER_MIN_U64 ? 1 : 2, a, grid);
    if (op == PLM_PEER_MIN_U64) plm::peer_reduce_kernel<0><<<grid, plm::PEER_THREADS, 0, ctx->stream>>>(a);
    else plm::peer_reduce_kernel<1><<<grid, plm::PEER_THREADS, 0, ctx->stream>>>(a);
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    return PLM_OK;
}

// ---------------------------------------------------------------------------------------------
// Bag-of-words: DBoW2 vocabulary transform + L1 score (src/mapHandler.cpp:3116-3237)
struct plm_voc {
    plm_ctx *ctx = nullptr;
    char *d_buf = nullptr;
    plm::VocDev dev{};
    int n_words = 0;
    bool smem_attr_set = false;
};

namespace {

constexpr int BOW_MAX_SET = 8192;

int pow2_at_least(int n) {
    int p = 32;
    while (p < n) p <<= 1;
    return p;
}

int launch_bow_transform(plm_voc *voc, plm::BowTransformArgs a, int max_set) {
    plm_ctx *ctx = voc->ctx;
    a.voc = voc->dev;
    a.cap = pow2_at_least(std::max(max_set, 1));
    const size_t smem = plm::bow_transform_smem(a.cap);
    if (smem > 48 * 1024 || !voc->smem_attr_set) {
        CU_TRY(cudaFuncSetAttribute(plm::bow_transform_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    static_cast<int>(plm::bow_transform_smem(BOW_MAX_SET))));
        voc->smem_attr_set = true;
    }
    plm::bow_transform_kernel<<<std::min(a.n_sets, ctx->sm_count * 8), plm::BOW_THREADS, smem, ctx->stream>>>(a);
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    return PLM_OK;
}

int launch_bow_score(plm_ctx *ctx, plm::BowScoreArgs a, int max_q_len, int64_t n_words) {
    a.q_cap = std::max(max_q_len, 1);
    a.table_slots = pow2_at_least(2 * a.q_cap);
    // membership bitmap over word ids [0, n_words): as large as fits next to the staged query and its hash table;
    // word ids beyond it (or n_words unknown) go to the hash table directly
    const size_t budget = ctx->smem_optin > 2048 ? ctx->smem_optin - 2048 : 0;
    const size_t fixed = plm::bow_score_smem(a.q_cap, a.table_slots, 0);
    size_t words = n_words > 0 ? static_cast<size_t>((n_words + 31) / 32) : 0;
    if (fixed + words * 4 > budget) words = budget > fixed ? (budget - fixed) / 4 : 0;
    a.bitmap_words = static_cast<int>(words);
    const size_t smem = plm::bow_score_smem(a.q_cap, a.table_slots, a.bitmap_words);
    if (smem > budget) return fail(PLM_E_UNSUPPORTED, "query vector too long for shared memory");
    CU_TRY(cudaFuncSetAttribute(plm::bow_score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(budget)));
    // a large bitmap leaves room for few CTAs per SM: make them wide so that enough warps stream the database
    const int threads = smem > 24 * 1024 ? 512 : plm::BOW_THREADS;
    const int warps = threads / 32;
    // one resident wave: every CTA builds the query's bitmap and hash table once, its warps then loop over the database
    int per_sm = 0;
    CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, plm::bow_score_kernel, threads, smem));
    const int ctas = std::max(1, std::min((a.n_db + warps - 1) / warps, ctx->sm_count * std::max(per_sm, 1)));
    plm::bow_score_kernel<<<dim3(ctas, a.n_q), threads, smem, ctx->stream>>>(a);
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    return PLM_OK;
}

} // namespace

PLM_API int plm_voc_create(plm_ctx *ctx, int n_nodes, const int32_t *child_start, const int32_t *child_ids,
                           const uint8_t *node_desc, const double *node_weight, const int32_t *node_word, int weighting,
                           int scoring, plm_voc **out) {
    if (!out) return fail(PLM_E_INVALID, "null out");
    *out = nullptr;
    if (n_nodes < 1 || !child_start || !node_desc || !node_weight || !node_word) return fail(PLM_E_INVALID, "null pointer / empty tree");
    if (weighting < 0 || weighting > 3) return fail(PLM_E_INVALID, "unknown DBoW2 weighting type");
    if (scoring != 0) return fail(PLM_E_UNSUPPORTED, "only L1_NORM scoring (the DBoW2 default) is implemented");
    if (child_start[0] != 0) return fail(PLM_E_INVALID, "child_start[0] != 0");
    const int n_child = child_start[n_nodes];
    if (n_child != n_nodes - 1 || (n_child > 0 && !child_ids)) return fail(PLM_E_INVALID, "every node except the root must be a child exactly once");
    std::vector<char> seen(static_cast<size_t>(n_nodes), 0);
    int n_words = 0;
    for (int i = 0; i < n_nodes; ++i) {
        if (child_start[i + 1] < child_start[i] || child_start[i + 1] > n_child) return fail(PLM_E_INVALID, "child_start must be non-decreasing");
        for (int c = child_start[i]; c < child_start[i + 1]; ++c) {
            const int id = child_ids[c];
            if (id <= i || id >= n_nodes || seen[id]) return fail(PLM_E_INVALID, "child id outside (parent, n_nodes) or listed twice");
            seen[id] = 1;
        }
        const bool leaf = child_start[i + 1] == child_start[i];
        if (leaf && i > 0) {
            if (node_word[i] < 0) return fail(PLM_E_INVALID, "leaf without a word id");
            n_words = std::max(n_words, node_word[i] + 1);
        }
    }
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    plm_voc *v = new (std::nothrow) plm_voc();
    if (!v) return fail(PLM_E_NOMEM, "host allocation failed");
    v->ctx = ctx;
    v->n_words = n_words;
    Layout L;
    const size_t o_desc = L.add(size_t(n_nodes) * 32), o_w = L.add(size_t(n_nodes) * 8), o_cs = L.add(size_t(n_nodes + 1) * 4),
                 o_ci = L.add(size_t(std::max(n_child, 1)) * 4), o_word = L.add(size_t(n_nodes) * 4);
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&v->d_buf), L.total);
    if (e == cudaSuccess) e = cudaMemcpyAsync(v->d_buf + o_desc, node_desc, size_t(n_nodes) * 32, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(v->d_buf + o_w, node_weight, size_t(n_nodes) * 8, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(v->d_buf + o_cs, child_start, size_t(n_nodes + 1) * 4, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess && n_child > 0) e = cudaMemcpyAsync(v->d_buf + o_ci, child_ids, size_t(n_child) * 4, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(v->d_buf + o_word, node_word, size_t(n_nodes) * 4, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        if (v->d_buf) cudaFree(v->d_buf);
        delete v;
        return fail(e == cudaErrorMemoryAllocation ? PLM_E_NOMEM : PLM_E_CUDA, std::string("plm_voc_create: ") + cudaGetErrorString(e));
    }
    v->dev.node_desc = reinterpret_cast<const uint4 *>(v->d_buf + o_desc);
    v->dev.node_weight = reinterpret_cast<const double *>(v->d_buf + o_w);
    v->dev.child_start = reinterpret_cast<const int32_t *>(v->d_buf + o_cs);
    v->dev.child_ids = reinterpret_cast<const int32_t *>(v->d_buf + o_ci);
    v->dev.node_word = reinterpret_cast<const int32_t *>(v->d_buf + o_word);
    v->dev.n_nodes = n_nodes;
    v->dev.weighting = weighting;
    *out = v;
    return PLM_OK;
}

PLM_API int plm_voc_destroy(plm_voc *voc) {
    if (!voc) return PLM_OK;
    if (voc->ctx) {
        cudaSetDevice(voc->ctx->device);
        cudaStreamSynchronize(voc->ctx->stream);
    }
    if (voc->d_buf) cudaFree(voc->d_buf);
    delete voc;
    return PLM_OK;
}

PLM_API int plm_voc_words(const plm_voc *voc) { return voc ? voc->n_words : 0; }

PLM_API int plm_dev_bow_transform(plm_voc *voc, const void *desc_dev, int64_t n_rows, const int32_t *set_start_dev, int n_sets,
                                  int max_set, uint32_t *bow_ids_dev, double *bow_vals_dev, int32_t *bow_len_dev) {
    if (!voc) return fail(PLM_E_INVALID, "null vocabulary");
    if (n_sets < 0 || n_rows < 0 || max_set < 0) return fail(PLM_E_INVALID, "negative size");
    if (n_sets == 0) return PLM_OK;
    if (!set_start_dev || !bow_len_dev || (n_rows > 0 && (!desc_dev || !bow_ids_dev || !bow_vals_dev))) return fail(PLM_E_INVALID, "null pointer");
    if (reinterpret_cast<uintptr_t>(desc_dev) & 15) return fail(PLM_E_INVALID, "descriptor rows must be 16-byte aligned");
    if (max_set > BOW_MAX_SET) return fail(PLM_E_UNSUPPORTED, "more than 8192 features in one set");
    plm_ctx *ctx = voc->ctx;
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    plm::BowTransformArgs a{};
    a.desc = static_cast<const uint4 *>(desc_dev);
    a.set_start = set_start_dev;
    a.n_sets = n_sets;
    a.bow_ids = bow_ids_dev;
    a.bow_vals = bow_vals_dev;
    a.bow_len = bow_len_dev;
    return launch_bow_transform(voc, a, max_set);
}

PLM_API int plm_bow_transform(plm_voc *voc, const uint8_t *desc, int64_t n_rows, size_t step, const int32_t *set_start,
                              int n_sets, uint32_t *bow_ids, double *bow_vals, int32_t *bow_len) {
    if (!voc) return fail(PLM_E_INVALID, "null vocabulary");
    if (n_sets < 0 || n_rows < 0) return fail(PLM_E_INVALID, "negative size");
    if (n_sets == 0) return PLM_OK;
    if (!set_start || !bow_len || (n_rows > 0 && (!desc || !bow_ids || !bow_vals))) return fail(PLM_E_INVALID, "null pointer");
    if (step < 32) return fail(PLM_E_INVALID, "step < 32");
    if (n_rows > INT32_MAX) return fail(PLM_E_UNSUPPORTED, "more than 2^31 - 1 rows in one call");
    if (set_start[0] < 0 || set_start[n_sets] > n_rows) return fail(PLM_E_INVALID, "set_start outside [0, n_rows]");
    int max_set = 0;
    for (int s = 0; s < n_sets; ++s) {
        if (set_start[s + 1] < set_start[s]) return fail(PLM_E_INVALID, "set_start must be non-decreasing");
        max_set = std::max(max_set, set_start[s + 1] - set_start[s]);
    }
    if (max_set > BOW_MAX_SET) return fail(PLM_E_UNSUPPORTED, "more than 8192 features in one set");
    plm_ctx *ctx = voc->ctx;
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    Layout L;
    const size_t o_start = L.add(size_t(n_sets + 1) * 4), o_desc = L.add(size_t(n_rows) * 32);
    const size_t in_bytes = L.total;
    const size_t o_vals = L.add(size_t(n_rows) * 8), o_ids = L.add(size_t(n_rows) * 4), o_len = L.add(size_t(n_sets) * 4);
    if ((st = ctx->ensure_pinned(L.total)) != PLM_OK) return st;
    if ((st = ctx->ensure_device(L.total)) != PLM_OK) return st;
    std::memcpy(ctx->h_buf + o_start, set_start, size_t(n_sets + 1) * 4);
    pack_rows(ctx->h_buf + o_desc, desc, n_rows, step);
    CU_TRY(cudaMemcpyAsync(ctx->d_buf, ctx->h_buf, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    plm::BowTransformArgs a{};
    a.desc = reinterpret_cast<const uint4 *>(ctx->d_buf + o_desc);
    a.set_start = reinterpret_cast<const int32_t *>(ctx->d_buf + o_start);
    a.n_sets = n_sets;
    a.bow_vals = reinterpret_cast<double *>(ctx->d_buf + o_vals);
    a.bow_ids = reinterpret_cast<uint32_t *>(ctx->d_buf + o_ids);
    a.bow_len = reinterpret_cast<int32_t *>(ctx->d_buf + o_len);
    if ((st = launch_bow_transform(voc, a, max_set)) != PLM_OK) return st;
    CU_TRY(cudaMemcpyAsync(ctx->h_buf + o_vals, ctx->d_buf + o_vals, L.total - o_vals, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    std::memcpy(bow_len, ctx->h_buf + o_len, size_t(n_sets) * 4);
    // only the written slots of a set are defined on the device; copy those
    for (int s = 0; s < n_sets; ++s) {
        const size_t lo = size_t(set_start[s]), n = size_t(bow_len[s]);
        std::memcpy(bow_ids + lo, ctx->h_buf + o_ids + lo * 4, n * 4);
        std::memcpy(bow_vals + lo, ctx->h_buf + o_vals + lo * 8, n * 8);
    }
    return PLM_OK;
}

PLM_API int plm_dev_bow_score(plm_ctx *ctx, const uint32_t *q_ids_dev, const double *q_vals_dev, const int64_t *q_start_dev,
                              const int32_t *q_len_dev, int n_q, int max_q_len, int64_t n_words, const uint32_t *db_ids_dev,
                              const double *db_vals_dev, const int64_t *db_start_dev, const int32_t *db_len_dev, int n_db,
                              double *scores_dev) {
    if (n_q < 0 || n_db < 0 || max_q_len < 0) return fail(PLM_E_INVALID, "negative size");
    if (n_q == 0 || n_db == 0) return PLM_OK;
    if (!q_start_dev || !q_len_dev || !db_start_dev || !db_len_dev || !scores_dev) return fail(PLM_E_INVALID, "null pointer");
    if (max_q_len > BOW_MAX_SET) return fail(PLM_E_UNSUPPORTED, "more than 8192 entries in a query vector");
    if (n_q > 65535) return fail(PLM_E_UNSUPPORTED, "more than 65535 queries in one launch");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    plm::BowScoreArgs a{};
    a.q_ids = q_ids_dev;
    a.q_vals = q_vals_dev;
    a.q_start = reinterpret_cast<const long long *>(q_start_dev);
    a.q_len = q_len_dev;
    a.n_q = n_q;
    a.db_ids = db_ids_dev;
    a.db_vals = db_vals_dev;
    a.db_start = reinterpret_cast<const long long *>(db_start_dev);
    a.db_len = db_len_dev;
    a.n_db = n_db;
    a.scores = scores_dev;
    return launch_bow_score(ctx, a, max_q_len, n_words);
}

namespace {

// Extent (in entries) of a set of sparse vectors and their validity: every [start, start + len) inside [0, cap_hint].
int bow_vectors_extent(const int64_t *start, const int32_t *len, int n, int64_t *extent, int *max_len) {
    int64_t hi = 0;
    int ml = 0;
    for (int i = 0; i < n; ++i) {
        if (start[i] < 0 || len[i] < 0) return fail(PLM_E_INVALID, "negative vector start / length");
        hi = std::max<int64_t>(hi, start[i] + len[i]);
        ml = std::max(ml, len[i]);
    }
    *extent = hi;
    *max_len = ml;
    return PLM_OK;
}

} // namespace

PLM_API int plm_bow_score(plm_ctx *ctx, const uint32_t *q_ids, const double *q_vals, const int64_t *q_start,
                          const int32_t *q_len, int n_q, const uint32_t *db_ids, const double *db_vals,
                          const int64_t *db_start, const int32_t *db_len, int n_db, double *scores) {
    if (n_q < 0 || n_db < 0) return fail(PLM_E_INVALID, "negative size");
    if (n_q == 0 || n_db == 0) return PLM_OK;
    if (!q_start || !q_len || !db_start || !db_len || !scores) return fail(PLM_E_INVALID, "null pointer");
    int64_t q_ext = 0, db_ext = 0;
    int q_max = 0, db_max = 0;
    int st;
    if ((st = bow_vectors_extent(q_start, q_len, n_q, &q_ext, &q_max)) != PLM_OK) return st;
    if ((st = bow_vectors_extent(db_start, db_len, n_db, &db_ext, &db_max)) != PLM_OK) return st;
    if ((q_ext > 0 && (!q_ids || !q_vals)) || (db_ext > 0 && (!db_ids || !db_vals))) return fail(PLM_E_INVALID, "null pointer");
    if (q_max > BOW_MAX_SET) return fail(PLM_E_UNSUPPORTED, "more than 8192 entries in a query vector");
    if ((st = resolve_ctx(ctx)) != PLM_OK) return st;
    Layout L;
    const size_t o_qv = L.add(size_t(q_ext) * 8), o_dv = L.add(size_t(db_ext) * 8), o_qs = L.add(size_t(n_q) * 8),
                 o_ds = L.add(size_t(n_db) * 8), o_qi = L.add(size_t(q_ext) * 4), o_di = L.add(size_t(db_ext) * 4),
                 o_ql = L.add(size_t(n_q) * 4), o_dl = L.add(size_t(n_db) * 4);
    const size_t in_bytes = L.total;
    const size_t o_out = L.add(size_t(n_q) * size_t(n_db) * 8);
    if ((st = ctx->ensure_pinned(L.total)) != PLM_OK) return st;
    if ((st = ctx->ensure_device(L.total)) != PLM_OK) return st;
    char *H = ctx->h_buf, *D = ctx->d_buf;
    if (q_ext) std::memcpy(H + o_qv, q_vals, size_t(q_ext) * 8), std::memcpy(H + o_qi, q_ids, size_t(q_ext) * 4);
    if (db_ext) std::memcpy(H + o_dv, db_vals, size_t(db_ext) * 8), std::memcpy(H + o_di, db_ids, size_t(db_ext) * 4);
    std::memcpy(H + o_qs, q_start, size_t(n_q) * 8);
    std::memcpy(H + o_ds, db_start, size_t(n_db) * 8);
    std::memcpy(H + o_ql, q_len, size_t(n_q) * 4);
    std::memcpy(H + o_dl, db_len, size_t(n_db) * 4);
    CU_TRY(cudaMemcpyAsync(D, H, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    // word ids reach up to the largest query id: the bitmap covers [0, that]
    int64_t q_words = 0;
    for (int i = 0; i < n_q; ++i)
        if (q_len[i] > 0) q_words = std::max<int64_t>(q_words, int64_t(q_ids[q_start[i] + q_len[i] - 1]) + 1);
    if ((st = plm_dev_bow_score(ctx, reinterpret_cast<const uint32_t *>(D + o_qi), reinterpret_cast<const double *>(D + o_qv),
                                reinterpret_cast<const int64_t *>(D + o_qs), reinterpret_cast<const int32_t *>(D + o_ql), n_q, q_max, q_words,
                                reinterpret_cast<const uint32_t *>(D + o_di), reinterpret_cast<const double *>(D + o_dv),
                                reinterpret_cast<const int64_t *>(D + o_ds), reinterpret_cast<const int32_t *>(D + o_dl), n_db,
                                reinterpret_cast<double *>(D + o_out))) != PLM_OK)
        return st;
    CU_TRY(cudaMemcpyAsync(H + o_out, D + o_out, size_t(n_q) * size_t(n_db) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    std::memcpy(scores, H + o_out, size_t(n_q) * size_t(n_db) * 8);
    return PLM_OK;
}

// ---------------------------------------------------------------------------------------------
// Stereo post-filters
PLM_API int plm_stereo_filter_points(plm_ctx *ctx, const float *kp_l, int n1, const float *kp_r, int n2, const int32_t *m12,
                                     double max_dist_epip, double min_disp, uint8_t *keep, double *disp, int *n_kept) {
    if (n1 < 0 || n2 < 0) return fail(PLM_E_INVALID, "negative size");
    if (!n_kept) return fail(PLM_E_INVALID, "null n_kept");
    *n_kept = 0;
    if (n1 == 0) return PLM_OK;
    if (!kp_l || !m12 || !keep || !disp || (n2 > 0 && !kp_r)) return fail(PLM_E_INVALID, "null pointer");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    Layout L;
    const size_t o_l = L.add(size_t(n1) * 8), o_r = L.add(size_t(std::max(n2, 1)) * 8), o_m = L.add(size_t(n1) * 4);
    const size_t in_bytes = L.total;
    const size_t o_out = L.add(size_t(n1) * 8 + size_t(n1) + 8); // disp | keep | count
    if ((st = ctx->ensure_pinned(L.total)) != PLM_OK) return st;
    if ((st = ctx->ensure_device(L.total)) != PLM_OK) return st;
    std::memcpy(ctx->h_buf + o_l, kp_l, size_t(n1) * 8);
    if (n2 > 0) std::memcpy(ctx->h_buf + o_r, kp_r, size_t(n2) * 8);
    std::memcpy(ctx->h_buf + o_m, m12, size_t(n1) * 4);
    CU_TRY(cudaMemcpyAsync(ctx->d_buf, ctx->h_buf, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    double *d_disp = reinterpret_cast<double *>(ctx->d_buf + o_out);
    uint8_t *d_keep = reinterpret_cast<uint8_t *>(ctx->d_buf + o_out + size_t(n1) * 8);
    const size_t cnt_off = align_up(size_t(n1) * 8 + size_t(n1), 4);
    int32_t *d_cnt = reinterpret_cast<int32_t *>(ctx->d_buf + o_out + cnt_off);
    CU_TRY(cudaMemsetAsync(d_cnt, 0, 4, ctx->stream));
    plm::stereo_filter_points_kernel<<<(n1 + 127) / 128, 128, 0, ctx->stream>>>(
        reinterpret_cast<const float2 *>(ctx->d_buf + o_l), reinterpret_cast<const float2 *>(ctx->d_buf + o_r), n2,
        reinterpret_cast<const int32_t *>(ctx->d_buf + o_m), n1, max_dist_epip, min_disp, d_keep, d_disp, d_cnt);
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(ctx->h_buf + o_out, ctx->d_buf + o_out, cnt_off + 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    std::memcpy(disp, ctx->h_buf + o_out, size_t(n1) * 8);
    std::memcpy(keep, ctx->h_buf + o_out + size_t(n1) * 8, size_t(n1));
    int32_t cnt;
    std::memcpy(&cnt, ctx->h_buf + o_out + cnt_off, 4);
    *n_kept = cnt;
    return PLM_OK;
}

PLM_API int plm_stereo_filter_lines(plm_ctx *ctx, const float *ln_l, int n1, const float *ln_r, int n2, const int32_t *m12,
                                    double min_disp, double line_horiz_th, double stereo_overlap_th,
                                    double ls_min_disp_ratio, uint8_t *keep, double *disp_se, int *n_kept) {
    if (n1 < 0 || n2 < 0) return fail(PLM_E_INVALID, "negative size");
    if (!n_kept) return fail(PLM_E_INVALID, "null n_kept");
    *n_kept = 0;
    if (n1 == 0) return PLM_OK;
    if (!ln_l || !m12 || !keep || !disp_se || (n2 > 0 && !ln_r)) return fail(PLM_E_INVALID, "null pointer");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    Layout L;
    const size_t o_l = L.add(size_t(n1) * 16), o_r = L.add(size_t(std::max(n2, 1)) * 16), o_m = L.add(size_t(n1) * 4);
    const size_t in_bytes = L.total;
    const size_t o_out = L.add(size_t(n1) * 16 + size_t(n1) + 8);
    if ((st = ctx->ensure_pinned(L.total)) != PLM_OK) return st;
    if ((st = ctx->ensure_device(L.total)) != PLM_OK) return st;
    std::memcpy(ctx->h_buf + o_l, ln_l, size_t(n1) * 16);
    if (n2 > 0) std::memcpy(ctx->h_buf + o_r, ln_r, size_t(n2) * 16);
    std::memcpy(ctx->h_buf + o_m, m12, size_t(n1) * 4);
    CU_TRY(cudaMemcpyAsync(ctx->d_buf, ctx->h_buf, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    double *d_disp = reinterpret_cast<double *>(ctx->d_buf + o_out);
    uint8_t *d_keep = reinterpret_cast<uint8_t *>(ctx->d_buf + o_out + size_t(n1) * 16);
    const size_t cnt_off = align_up(size_t(n1) * 16 + size_t(n1), 4);
    int32_t *d_cnt = reinterpret_cast<int32_t *>(ctx->d_buf + o_out + cnt_off);
    CU_TRY(cudaMemsetAsync(d_cnt, 0, 4, ctx->stream));
    plm::stereo_filter_lines_kernel<<<(n1 + 127) / 128, 128, 0, ctx->stream>>>(
        reinterpret_cast<const float4 *>(ctx->d_buf + o_l), reinterpret_cast<const float4 *>(ctx->d_buf + o_r), n2,
        reinterpret_cast<const int32_t *>(ctx->d_buf + o_m), n1, min_disp, line_horiz_th, stereo_overlap_th,
        ls_min_disp_ratio, d_keep, d_disp, d_cnt);
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(ctx->h_buf + o_out, ctx->d_buf + o_out, cnt_off + 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    std::memcpy(disp_se, ctx->h_buf + o_out, size_t(n1) * 16);
    std::memcpy(keep, ctx->h_buf + o_out + size_t(n1) * 16, size_t(n1));
    int32_t cnt;
    std::memcpy(&cnt, ctx->h_buf + o_out + cnt_off, 4);
    *n_kept = cnt;
    return PLM_OK;
}

// ---------------------------------------------------------------------------------------------
// Database shard
PLM_API int plm_db_create(plm_ctx *ctx, int64_t capacity_rows, plm_db **out) {
    if (!out) return fail(PLM_E_INVALID, "null out");
    *out = nullptr;
    if (capacity_rows < 0) return fail(PLM_E_INVALID, "negative capacity");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    plm_db *db = new (std::nothrow) plm_db();
    if (!db) return fail(PLM_E_NOMEM, "host allocation failed");
    db->ctx = ctx;
    db->capacity = capacity_rows;
    if (capacity_rows > 0) {
        cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&db->rows), size_t(capacity_rows) * 32);
        if (e != cudaSuccess) {
            delete db;
            return fail(e == cudaErrorMemoryAllocation ? PLM_E_NOMEM : PLM_E_CUDA, cudaGetErrorString(e));
        }
    }
    *out = db;
    return PLM_OK;
}

PLM_API int plm_db_destroy(plm_db *db) {
    if (!db) return PLM_OK;
    if (db->ctx) cudaSetDevice(db->ctx->device);
    if (db->rows) cudaFree(db->rows);
    delete db;
    return PLM_OK;
}

PLM_API int plm_db_upload(plm_db *db, const uint8_t *rows, int64_t n, size_t step, int64_t at_row) {
    if (!db) return fail(PLM_E_INVALID, "null db");
    if (n < 0 || at_row < 0 || at_row + n > db->capacity) return fail(PLM_E_INVALID, "rows outside the database capacity");
    if (n == 0) return PLM_OK;
    if (!rows || step < 32) return fail(PLM_E_INVALID, "null rows / step < 32");
    plm_ctx *ctx = db->ctx;
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    // staged through pinned memory in 32 MB pieces
    const int64_t piece = (32 << 20) / 32;
    if ((st = ctx->ensure_pinned(size_t(std::min(n, piece)) * 32)) != PLM_OK) return st;
    for (int64_t r = 0; r < n; r += piece) {
        const int64_t m = std::min(piece, n - r);
        pack_rows(ctx->h_buf, rows + size_t(r) * step, m, step);
        CU_TRY(cudaMemcpyAsync(db->rows + 2 * (at_row + r), ctx->h_buf, size_t(m) * 32, cudaMemcpyHostToDevice, ctx->stream));
        CU_TRY(cudaStreamSynchronize(ctx->stream));
    }
    db->size = std::max(db->size, at_row + n);
    return PLM_OK;
}

PLM_API int64_t plm_db_size(const plm_db *db) { return db ? db->size : 0; }
PLM_API void *plm_db_device_ptr(const plm_db *db) { return db ? static_cast<void *>(db->rows) : nullptr; }

PLM_API int plm_db_knn2(plm_db *db, const uint8_t *q, int nq, size_t step, uint64_t idx_base, uint64_t *top2) {
    if (!db) return fail(PLM_E_INVALID, "null db");
    int st = check_desc(q, nq, step);
    if (st != PLM_OK) return st;
    if (nq > 0 && !top2) return fail(PLM_E_INVALID, "null top2");
    if (idx_base + static_cast<uint64_t>(db->size) > (1ull << 32)) return fail(PLM_E_UNSUPPORTED, "train index does not fit 32 bits");
    if (nq == 0) return PLM_OK;
    plm_ctx *ctx = db->ctx;
    if ((st = resolve_ctx(ctx)) != PLM_OK) return st;
    Layout L;
    const size_t o_q = L.add(size_t(nq) * 32);
    const size_t o_top2 = L.add(size_t(nq) * 16);
    const size_t staged = L.total;
    plm::KnnTaskPair tp;
    std::memset(&tp, 0, sizeof(tp));
    KnnPlan plan;
    size_t part_off = 0;
    build_knn_task(ctx, L, tp.t[0], plan, nullptr, nq, db->rows, db->size, idx_base, part_off, true);
    if ((st = ctx->ensure_pinned(staged)) != PLM_OK) return st;
    if ((st = ctx->ensure_device(L.total)) != PLM_OK) return st;
    pack_rows(ctx->h_buf + o_q, q, nq, step);
    CU_TRY(cudaMemcpyAsync(ctx->d_buf + o_q, ctx->h_buf + o_q, size_t(nq) * 32, cudaMemcpyHostToDevice, ctx->stream));
    tp.t[0].q = reinterpret_cast<const uint4 *>(ctx->d_buf + o_q);
    tp.t[0].part = reinterpret_cast<ulonglong2 *>(ctx->d_buf + part_off);
    tp.t[0].top2 = reinterpret_cast<ulonglong2 *>(ctx->d_buf + o_top2);
    if ((st = launch_knn_slices(ctx, tp, 1, plan.threads)) != PLM_OK) return st;
    if ((st = launch_knn_merge(ctx, tp, 1, 0.f, 0)) != PLM_OK) return st;
    CU_TRY(cudaMemcpyAsync(ctx->h_buf + o_top2, ctx->d_buf + o_top2, size_t(nq) * 16, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    std::memcpy(top2, ctx->h_buf + o_top2, size_t(nq) * 16);
    return PLM_OK;
}

// ---------------------------------------------------------------------------------------------
PLM_API int plm_measure_int_peaks(plm_ctx *ctx, double *popc_gops, double *lop3_gops) {
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    if ((st = ctx->ensure_device(1 << 20)) != PLM_OK) return st;
    cudaEvent_t e0, e1;
    CU_TRY(cudaEventCreate(&e0));
    CU_TRY(cudaEventCreate(&e1));
    const int blocks = ctx->sm_count * 8, threads = 256, iters = 4096;
    double out[2] = {0, 0};
    for (int which = 0; which < 2; ++which) {
        float best_ms = 1e30f;
        for (int rep = 0; rep < 4; ++rep) {
            CU_TRY(cudaEventRecord(e0, ctx->stream));
            if (which == 0) plm::popc_rate_kernel<<<blocks, threads, 0, ctx->stream>>>(reinterpret_cast<uint32_t *>(ctx->d_buf), iters);
            else plm::lop3_rate_kernel<<<blocks, threads, 0, ctx->stream>>>(reinterpret_cast<uint32_t *>(ctx->d_buf), iters);
            ctx->launches++;
            CU_TRY(cudaGetLastError());
            CU_TRY(cudaEventRecord(e1, ctx->stream));
            CU_TRY(cudaEventSynchronize(e1));
            float ms = 0.f;
            CU_TRY(cudaEventElapsedTime(&ms, e0, e1));
            if (rep > 0) best_ms = std::min(best_ms, ms);
        }
        const double ops = double(blocks) * threads * double(iters) * plm::MICRO_OPS_PER_ITER;
        out[which] = ops / (best_ms * 1e-3) * 1e-9;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (popc_gops) *popc_gops = out[0];
    if (lop3_gops) *lop3_gops = out[1];
    return PLM_OK;
}

PLM_API int plm_measure_mma_i8_rate(plm_ctx *ctx, int n, int with_stores, double *tops) {
    if (n != 128 && n != 256) return fail(PLM_E_INVALID, "plm_measure_mma_i8_rate: n must be 128 or 256");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    if ((st = umma_error_word(ctx)) != PLM_OK) return st;
    void (*kern)(int, int32_t *, long long) = n == 256 ? (with_stores ? plm::mma_i8_rate_kernel<256, true> : plm::mma_i8_rate_kernel<256, false>)
                                                       : (with_stores ? plm::mma_i8_rate_kernel<128, true> : plm::mma_i8_rate_kernel<128, false>);
    CU_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, plm::KNN_UMMA_RATE_SMEM));
    cudaEvent_t e0, e1;
    CU_TRY(cudaEventCreate(&e0));
    CU_TRY(cudaEventCreate(&e1));
    const int iters = 16384 * (256 / n); // 8 MMAs of 128 x n x 32 each: ~10 ms at the data-sheet rate
    float best_ms = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {
        CU_TRY(cudaEventRecord(e0, ctx->stream));
        kern<<<ctx->sm_count, 128, plm::KNN_UMMA_RATE_SMEM, ctx->stream>>>(iters, ctx->umma_err_dev, g_peer_spin_ticks);
        ctx->launches++;
        CU_TRY(cudaGetLastError());
        CU_TRY(cudaEventRecord(e1, ctx->stream));
        CU_TRY(cudaEventSynchronize(e1));
        float ms = 0.f;
        CU_TRY(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0) best_ms = std::min(best_ms, ms);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if ((st = umma_error_word(ctx)) != PLM_OK) return st;
    const double ops = 2.0 * ctx->sm_count * double(iters) * 8.0 * 128.0 * double(n) * 32.0;
    if (tops) *tops = ops / (best_ms * 1e-3) * 1e-12;
    return PLM_OK;
}

PLM_API int plm_measure_mma_i8_peak(plm_ctx *ctx, double *tops) { return plm_measure_mma_i8_rate(ctx, 256, 0, tops); }

#ifdef PLM_UMMA_STAMPS
// debug builds: the role stamps of the last knn2_umma_kernel launch, [KNN_UMMA_STAMP_CTAS][4 roles][3] (see the kernel)
extern "C" __attribute__((visibility("default"))) int plm_debug_umma_stamps(long long *out) {
    cudaDeviceSynchronize();
    return cudaMemcpyFromSymbol(out, plm::g_umma_stamps, sizeof(plm::g_umma_stamps)) == cudaSuccess ? 0 : -1;
}
#endif

// ---------------------------------------------------------------------------------------------
// Batched replay
struct plm_batch {
    plm_ctx *ctx = nullptr;
    int kind = 0; // 0 unset, 1 match, 2 grid
    char *d_buf = nullptr;
    size_t d_cap = 0;
    int n_jobs = 0;
    int64_t n_m = 0;
    size_t o_work = 0, o_init = 0, work_bytes = 0; // [m12 | counts] working copy and pristine copy
    // match
    size_t o_tasks = 0, o_cta_map = 0, o_merge_map = 0, o_xjobs = 0, o_xmap = 0, o_m21 = 0, m21_bytes = 0;
    int n_slice_ctas = 0, n_merge_ctas = 0, n_x_ctas = 0;
    float nnr = 0.f;
    int best_lr = 0;
    // grid
    size_t o_gjobs = 0;
    plm::GridParams gp;
    int n1_max = 0, n2_max = 0, items_max = 1;
    bool any_lines = false;
    int64_t h2d = 0, d2h = 0;

    int ensure(size_t bytes) {
        if (bytes <= d_cap) return PLM_OK;
        CU_TRY(cudaStreamSynchronize(ctx->stream));
        if (d_buf) CU_TRY(cudaFree(d_buf));
        d_buf = nullptr;
        d_cap = 0;
        CU_TRY(cudaMalloc(reinterpret_cast<void **>(&d_buf), align_up(bytes, 1 << 20)));
        d_cap = align_up(bytes, 1 << 20);
        return PLM_OK;
    }
};

PLM_API int plm_batch_create(plm_ctx *ctx, plm_batch **out) {
    if (!out) return fail(PLM_E_INVALID, "null out");
    *out = nullptr;
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    plm_batch *b = new (std::nothrow) plm_batch();
    if (!b) return fail(PLM_E_NOMEM, "host allocation failed");
    b->ctx = ctx;
    *out = b;
    return PLM_OK;
}

PLM_API int plm_batch_destroy(plm_batch *b) {
    if (!b) return PLM_OK;
    if (b->ctx) {
        cudaSetDevice(b->ctx->device);
        cudaStreamSynchronize(b->ctx->stream);
    }
    if (b->d_buf) cudaFree(b->d_buf);
    delete b;
    return PLM_OK;
}

PLM_API int64_t plm_batch_h2d_bytes(const plm_batch *b) { return b ? b->h2d : 0; }
PLM_API int64_t plm_batch_d2h_bytes(const plm_batch *b) { return b ? b->d2h : 0; }

namespace {
constexpr int BATCH_THREADS = 64;
}

namespace {
int batch_set_match_impl(plm_batch *b, const uint8_t *arena, const void *arena_dev, int64_t n_rows, const plm_pair_job *jobs,
                         int n_jobs, float nnr, int best_lr, const int32_t *m12_arena, int64_t n_m);
} // namespace

PLM_API int plm_batch_set_match(plm_batch *b, const uint8_t *arena, int64_t n_rows, const plm_pair_job *jobs, int n_jobs,
                                float nnr, int best_lr, const int32_t *m12_arena, int64_t n_m) {
    if (n_rows > 0 && !arena) return fail(PLM_E_INVALID, "null pointer");
    if (n_m > 0 && !m12_arena) return fail(PLM_E_INVALID, "null pointer");
    return batch_set_match_impl(b, arena, nullptr, n_rows, jobs, n_jobs, nnr, best_lr, m12_arena, n_m);
}

PLM_API int plm_batch_set_match_dev(plm_batch *b, const void *arena_dev, int64_t n_rows, const plm_pair_job *jobs, int n_jobs,
                                    float nnr, int best_lr, const int32_t *m12_arena, int64_t n_m) {
    if (n_rows > 0 && !arena_dev) return fail(PLM_E_INVALID, "null pointer");
    if (reinterpret_cast<uintptr_t>(arena_dev) & 15) return fail(PLM_E_INVALID, "device descriptor pointers must be 16-byte aligned");
    return batch_set_match_impl(b, nullptr, arena_dev ? arena_dev : reinterpret_cast<const void *>(16), n_rows, jobs, n_jobs, nnr,
                                best_lr, m12_arena, n_m);
}

namespace {
int batch_set_match_impl(plm_batch *b, const uint8_t *arena, const void *arena_dev, int64_t n_rows, const plm_pair_job *jobs,
                         int n_jobs, float nnr, int best_lr, const int32_t *m12_arena, int64_t n_m) {
    if (!b) return fail(PLM_E_INVALID, "null batch");
    if (n_rows < 0 || n_jobs < 0 || n_m < 0) return fail(PLM_E_INVALID, "negative size");
    if (n_jobs > 0 && !jobs) return fail(PLM_E_INVALID, "null pointer");
    plm_ctx *ctx = b->ctx;
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    best_lr = best_lr ? 1 : 0;

    // host-side tables
    std::vector<plm::KnnTask> tasks;
    std::vector<int4> cta_map;
    std::vector<int2> merge_map, xmap;
    std::vector<plm::XJob> xjobs;
    std::vector<int32_t> counts_init(static_cast<size_t>(n_jobs), 0);
    std::vector<size_t> part_off; // per task, relative to the part arena
    std::vector<int64_t> m21_off(static_cast<size_t>(n_jobs), 0);
    int64_t m21_rows = 0;
    size_t part_bytes = 0;
    long long total_qblocks = 0;
    for (int j = 0; j < n_jobs; ++j) {
        const plm_pair_job &jb = jobs[j];
        if (jb.n1 < 0 || jb.n2 < 0 || jb.off1 < 0 || jb.off2 < 0 || jb.off_m < 0 || jb.off1 + jb.n1 > n_rows ||
            jb.off2 + jb.n2 > n_rows || jb.off_m + jb.n1 > n_m)
            return fail(PLM_E_INVALID, "batch job outside its arena");
        if (jb.n2 < 2 || (best_lr && jb.n1 < 2)) continue;
        total_qblocks += (jb.n1 + BATCH_THREADS - 1) / BATCH_THREADS;
        if (best_lr) total_qblocks += (jb.n2 + BATCH_THREADS - 1) / BATCH_THREADS;
    }
    // slices per direction: enough CTAs for a few waves when the batch is small, 1 when it is large
    const long long target = static_cast<long long>(ctx->sm_count) * 16;
    const int want_slices = static_cast<int>(std::max<long long>(1, target / std::max<long long>(1, total_qblocks)));
    for (int j = 0; j < n_jobs; ++j) {
        const plm_pair_job &jb = jobs[j];
        if (jb.n2 < 2 || (best_lr && jb.n1 < 2)) {
            counts_init[j] = INT32_MIN;
            continue;
        }
        m21_off[j] = m21_rows;
        if (best_lr) m21_rows += jb.n2;
        for (int dir = 0; dir <= best_lr; ++dir) {
            plm::KnnTask t;
            std::memset(&t, 0, sizeof(t));
            const int nq = dir ? jb.n2 : jb.n1, nt = dir ? jb.n1 : jb.n2;
            int slices = std::min(want_slices, std::max(1, (nt + 63) / 64)); // workers of this task
            const int rows = std::min(plm::KNN_STAGE_ROWS, ((nt + slices - 1) / slices + 63) / 64 * 64);
            const int units = std::max(1, (nt + rows - 1) / rows);
            slices = std::min(slices, units);
            t.n1 = nq;
            t.n2 = nt;
            t.unit_rows = rows;
            t.n_units = units;
            t.n_workers = slices;
            t.idx_base = 0;
            // pointers are patched once the device block exists; stash offsets in the fields
            t.q = reinterpret_cast<const uint4 *>(static_cast<uintptr_t>(dir ? jb.off2 : jb.off1));
            t.db = reinterpret_cast<const uint4 *>(static_cast<uintptr_t>(dir ? jb.off1 : jb.off2));
            t.m = reinterpret_cast<int32_t *>(static_cast<uintptr_t>(dir ? m21_off[j] : jb.off_m));
            t.count = dir ? nullptr : reinterpret_cast<int32_t *>(static_cast<uintptr_t>(j) + 1); // +1: non-null marker
            t.threads = dir; // direction marker until the pointers are patched
            part_off.push_back(part_bytes);
            part_bytes += align_up(size_t(slices) * nq * sizeof(ulonglong2));
            const int task_id = static_cast<int>(tasks.size());
            for (int qb = 0; qb * BATCH_THREADS < nq; ++qb) {
                for (int s = 0; s < slices; ++s) cta_map.push_back(make_int4(task_id, qb, s, 0));
                merge_map.push_back(make_int2(task_id, qb * BATCH_THREADS));
            }
            tasks.push_back(t);
        }
        if (best_lr) {
            plm::XJob x;
            x.m12 = reinterpret_cast<int32_t *>(static_cast<uintptr_t>(jb.off_m));
            x.m21 = reinterpret_cast<const int32_t *>(static_cast<uintptr_t>(m21_off[j]));
            x.count = reinterpret_cast<int32_t *>(static_cast<uintptr_t>(j));
            x.n1 = jb.n1;
            x.n2 = jb.n2;
            const int xid = static_cast<int>(xjobs.size());
            xjobs.push_back(x);
            for (int r = 0; r < jb.n1; r += 128) xmap.push_back(make_int2(xid, r));
        }
    }

    Layout L;
    const size_t o_arena = L.add(arena_dev ? 0 : size_t(n_rows) * 32); // a resident arena is used in place
    b->work_bytes = align_up(size_t(n_m) * 4, 16) + size_t(n_jobs) * 4;
    b->o_work = L.add(b->work_bytes);
    b->o_init = L.add(b->work_bytes);
    b->o_tasks = L.add(tasks.size() * sizeof(plm::KnnTask));
    b->o_cta_map = L.add(cta_map.size() * sizeof(int4));
    b->o_merge_map = L.add(merge_map.size() * sizeof(int2));
    b->o_xjobs = L.add(xjobs.size() * sizeof(plm::XJob));
    b->o_xmap = L.add(xmap.size() * sizeof(int2));
    b->m21_bytes = size_t(m21_rows) * 4;
    b->o_m21 = L.add(b->m21_bytes);
    const size_t o_part = L.add(part_bytes);
    if ((st = b->ensure(L.total)) != PLM_OK) return st;

    char *D = b->d_buf;
    int32_t *d_m12 = reinterpret_cast<int32_t *>(D + b->o_work);
    int32_t *d_counts = reinterpret_cast<int32_t *>(D + b->o_work + align_up(size_t(n_m) * 4, 16));
    int32_t *d_m21 = reinterpret_cast<int32_t *>(D + b->o_m21);
    const uint4 *d_arena = arena_dev ? static_cast<const uint4 *>(arena_dev) : reinterpret_cast<const uint4 *>(D + o_arena);
    for (size_t i = 0; i < tasks.size(); ++i) {
        plm::KnnTask &t = tasks[i];
        const bool dir = t.threads != 0;
        t.q = d_arena + 2 * reinterpret_cast<uintptr_t>(t.q);
        t.db = d_arena + 2 * reinterpret_cast<uintptr_t>(t.db);
        t.m = (dir ? d_m21 : d_m12) + reinterpret_cast<uintptr_t>(t.m);
        t.count = t.count ? d_counts + (reinterpret_cast<uintptr_t>(t.count) - 1) : nullptr;
        t.part = reinterpret_cast<ulonglong2 *>(D + o_part + part_off[i]);
        t.top2 = nullptr;
        t.threads = 0;
    }
    for (plm::XJob &x : xjobs) {
        x.m12 = d_m12 + reinterpret_cast<uintptr_t>(x.m12);
        x.m21 = d_m21 + reinterpret_cast<uintptr_t>(x.m21);
        x.count = d_counts + reinterpret_cast<uintptr_t>(x.count);
    }

    // uploads: arenas straight from the caller's memory, tables through the pinned staging block
    const size_t tbl_bytes = L.total - b->o_tasks; // generous upper bound of the table region
    (void)tbl_bytes;
    // without an IN vector every match vector starts at -1: filled on the device, only the counts are staged
    const size_t counts_off = align_up(size_t(n_m) * 4, 16);
    Layout S;
    const size_t s_init = S.add(m12_arena ? b->work_bytes : size_t(n_jobs) * 4);
    const size_t s_tasks = S.add(tasks.size() * sizeof(plm::KnnTask));
    const size_t s_cta = S.add(cta_map.size() * sizeof(int4));
    const size_t s_merge = S.add(merge_map.size() * sizeof(int2));
    const size_t s_xjobs = S.add(xjobs.size() * sizeof(plm::XJob));
    const size_t s_xmap = S.add(xmap.size() * sizeof(int2));
    if ((st = ctx->ensure_pinned(S.total)) != PLM_OK) return st;
    char *H = ctx->h_buf;
    if (m12_arena) {
        if (n_m > 0) std::memcpy(H + s_init, m12_arena, size_t(n_m) * 4);
        if (n_jobs > 0) std::memcpy(H + s_init + counts_off, counts_init.data(), size_t(n_jobs) * 4);
    } else if (n_jobs > 0) {
        std::memcpy(H + s_init, counts_init.data(), size_t(n_jobs) * 4);
    }
    if (!tasks.empty()) std::memcpy(H + s_tasks, tasks.data(), tasks.size() * sizeof(plm::KnnTask));
    if (!cta_map.empty()) std::memcpy(H + s_cta, cta_map.data(), cta_map.size() * sizeof(int4));
    if (!merge_map.empty()) std::memcpy(H + s_merge, merge_map.data(), merge_map.size() * sizeof(int2));
    if (!xjobs.empty()) std::memcpy(H + s_xjobs, xjobs.data(), xjobs.size() * sizeof(plm::XJob));
    if (!xmap.empty()) std::memcpy(H + s_xmap, xmap.data(), xmap.size() * sizeof(int2));
    cudaStream_t s = ctx->stream;
    if (n_rows > 0 && !arena_dev) CU_TRY(cudaMemcpyAsync(D + o_arena, arena, size_t(n_rows) * 32, cudaMemcpyHostToDevice, s));
    if (m12_arena) {
        if (b->work_bytes) CU_TRY(cudaMemcpyAsync(D + b->o_init, H + s_init, b->work_bytes, cudaMemcpyHostToDevice, s));
    } else {
        if (n_m > 0) CU_TRY(cudaMemsetAsync(D + b->o_init, 0xFF, size_t(n_m) * 4, s));
        if (n_jobs > 0) CU_TRY(cudaMemcpyAsync(D + b->o_init + counts_off, H + s_init, size_t(n_jobs) * 4, cudaMemcpyHostToDevice, s));
    }
    if (!tasks.empty()) CU_TRY(cudaMemcpyAsync(D + b->o_tasks, H + s_tasks, tasks.size() * sizeof(plm::KnnTask), cudaMemcpyHostToDevice, s));
    if (!cta_map.empty()) CU_TRY(cudaMemcpyAsync(D + b->o_cta_map, H + s_cta, cta_map.size() * sizeof(int4), cudaMemcpyHostToDevice, s));
    if (!merge_map.empty()) CU_TRY(cudaMemcpyAsync(D + b->o_merge_map, H + s_merge, merge_map.size() * sizeof(int2), cudaMemcpyHostToDevice, s));
    if (!xjobs.empty()) CU_TRY(cudaMemcpyAsync(D + b->o_xjobs, H + s_xjobs, xjobs.size() * sizeof(plm::XJob), cudaMemcpyHostToDevice, s));
    if (!xmap.empty()) CU_TRY(cudaMemcpyAsync(D + b->o_xmap, H + s_xmap, xmap.size() * sizeof(int2), cudaMemcpyHostToDevice, s));
    CU_TRY(cudaStreamSynchronize(s)); // the pinned block is reused by the next call

    b->kind = 1;
    b->n_jobs = n_jobs;
    b->n_m = n_m;
    b->nnr = nnr;
    b->best_lr = best_lr;
    b->n_slice_ctas = static_cast<int>(cta_map.size());
    b->n_merge_ctas = static_cast<int>(merge_map.size());
    b->n_x_ctas = static_cast<int>(xmap.size());
    b->h2d = static_cast<int64_t>((arena_dev ? 0 : size_t(n_rows) * 32) + S.total);
    b->d2h = static_cast<int64_t>(size_t(n_m) * 4 + size_t(n_jobs) * 4);
    return PLM_OK;
}
} // namespace

PLM_API int plm_batch_set_match_grid(plm_batch *b, const uint8_t *arena, int64_t n_rows, const int32_t *coords,
                                     int64_t n_coords, const int32_t *cell_start, int64_t n_cell_start,
                                     const int32_t *cell_items, int64_t n_cell_items, const double *dirs2, int64_t n_dirs2,
                                     int grid_rows, int grid_cols, const plm_grid_job *jobs, int n_jobs, double ratio,
                                     double line_sim_th, int best_lr, const int32_t *m12_arena, int64_t n_m) {
    if (!b) return fail(PLM_E_INVALID, "null batch");
    if (n_rows < 0 || n_jobs < 0 || n_m < 0 || n_coords < 0 || n_cell_start < 0 || n_cell_items < 0 || n_dirs2 < 0)
        return fail(PLM_E_INVALID, "negative size");
    if ((n_rows > 0 && !arena) || (n_jobs > 0 && !jobs) || (n_m > 0 && !m12_arena) || (n_coords > 0 && !coords) ||
        (n_cell_start > 0 && !cell_start) || (n_cell_items > 0 && !cell_items) || (n_dirs2 > 0 && !dirs2))
        return fail(PLM_E_INVALID, "null pointer");
    if (grid_rows <= 0 || grid_cols <= 0) return fail(PLM_E_GRID, "[GridStructure] invalid dimension");
    if (ratio > 1.0) return fail(PLM_E_RATIO, plm_status_string(PLM_E_RATIO));
    plm_ctx *ctx = b->ctx;
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    const int64_t n_cells = static_cast<int64_t>(grid_rows) * grid_cols;

    Layout L;
    const size_t o_arena = L.add(size_t(n_rows) * 32);
    const size_t o_coords = L.add(size_t(n_coords) * 4);
    const size_t o_cs = L.add(size_t(n_cell_start) * 4);
    const size_t o_ci = L.add(size_t(n_cell_items) * 4);
    const size_t o_dirs = L.add(size_t(n_dirs2) * 8);
    b->work_bytes = align_up(size_t(n_m) * 4, 16) + size_t(n_jobs) * 4;
    b->o_work = L.add(b->work_bytes);
    b->o_init = L.add(b->work_bytes);
    b->o_gjobs = L.add(size_t(std::max(n_jobs, 1)) * sizeof(plm::GridJob));
    if ((st = b->ensure(L.total)) != PLM_OK) return st;
    char *D = b->d_buf;
    int32_t *d_m12 = reinterpret_cast<int32_t *>(D + b->o_work);
    int32_t *d_counts = reinterpret_cast<int32_t *>(D + b->o_work + align_up(size_t(n_m) * 4, 16));

    std::vector<plm::GridJob> gj(static_cast<size_t>(n_jobs));
    int n1_max = 1, n2_max = 1, items_max = 1;
    bool any_lines = false;
    for (int j = 0; j < n_jobs; ++j) {
        const plm_grid_job &jb = jobs[j];
        const int cpq = jb.is_lines ? 4 : 2;
        if (jb.n1 < 0 || jb.n2 < 0 || jb.off1 < 0 || jb.off2 < 0 || jb.off_m < 0 || jb.off_coords < 0 ||
            jb.off_cell_start < 0 || jb.off_cell_items < 0 || jb.off_dirs2 < 0 || jb.off1 + jb.n1 > n_rows ||
            jb.off2 + jb.n2 > n_rows || jb.off_m + jb.n1 > n_m || jb.off_coords + int64_t(jb.n1) * cpq > n_coords ||
            jb.off_cell_start + n_cells + 1 > n_cell_start || (jb.is_lines && jb.off_dirs2 + int64_t(jb.n2) * 2 > n_dirs2))
            return fail(PLM_E_INVALID, "grid job outside its arena");
        const int32_t *cs = cell_start + jb.off_cell_start;
        if (cs[0] != 0) return fail(PLM_E_GRID, "cell_start[0] must be 0");
        for (int64_t c = 0; c < n_cells; ++c)
            if (cs[c + 1] < cs[c]) return fail(PLM_E_GRID, "cell_start must be non-decreasing");
        if (jb.off_cell_items + cs[n_cells] > n_cell_items) return fail(PLM_E_INVALID, "grid job outside its item arena");
        if (jb.n1 > GRID_FUSED_MAX_ROWS || jb.n2 > GRID_N2_MAX)
            return fail(PLM_E_UNSUPPORTED, "batched matchGrid jobs must be frame-sized");
        plm::GridJob &g = gj[j];
        std::memset(&g, 0, sizeof(g));
        g.coords = reinterpret_cast<const int32_t *>(D + o_coords) + jb.off_coords;
        g.d1 = reinterpret_cast<const uint4 *>(D + o_arena) + 2 * jb.off1;
        g.d2 = reinterpret_cast<const uint4 *>(D + o_arena) + 2 * jb.off2;
        g.cell_start = reinterpret_cast<const int32_t *>(D + o_cs) + jb.off_cell_start;
        g.cell_items = reinterpret_cast<const int32_t *>(D + o_ci) + jb.off_cell_items;
        g.dirs2 = reinterpret_cast<const double *>(D + o_dirs) + jb.off_dirs2;
        g.m12 = d_m12 + jb.off_m;
        g.count = d_counts + j;
        g.n1 = jb.n1;
        g.n2 = jb.n2;
        g.is_lines = jb.is_lines ? 1 : 0;
        for (int i = 0; i < 4; ++i) g.win[i] = jb.win[i];
        n1_max = std::max(n1_max, jb.n1);
        n2_max = std::max(n2_max, jb.n2);
        items_max = std::max(items_max, cs[n_cells]);
        any_lines = any_lines || jb.is_lines != 0;
    }
    b->items_max = items_max;
    b->any_lines = any_lines;

    Layout S;
    const size_t s_init = S.add(b->work_bytes);
    const size_t s_jobs = S.add(gj.size() * sizeof(plm::GridJob));
    if ((st = ctx->ensure_pinned(S.total)) != PLM_OK) return st;
    char *H = ctx->h_buf;
    if (n_m > 0) std::memcpy(H + s_init, m12_arena, size_t(n_m) * 4);
    std::memset(H + s_init + align_up(size_t(n_m) * 4, 16), 0, size_t(n_jobs) * 4);
    if (!gj.empty()) std::memcpy(H + s_jobs, gj.data(), gj.size() * sizeof(plm::GridJob));
    cudaStream_t s = ctx->stream;
    if (n_rows > 0) CU_TRY(cudaMemcpyAsync(D + o_arena, arena, size_t(n_rows) * 32, cudaMemcpyHostToDevice, s));
    if (n_coords > 0) CU_TRY(cudaMemcpyAsync(D + o_coords, coords, size_t(n_coords) * 4, cudaMemcpyHostToDevice, s));
    if (n_cell_start > 0) CU_TRY(cudaMemcpyAsync(D + o_cs, cell_start, size_t(n_cell_start) * 4, cudaMemcpyHostToDevice, s));
    if (n_cell_items > 0) CU_TRY(cudaMemcpyAsync(D + o_ci, cell_items, size_t(n_cell_items) * 4, cudaMemcpyHostToDevice, s));
    if (n_dirs2 > 0) CU_TRY(cudaMemcpyAsync(D + o_dirs, dirs2, size_t(n_dirs2) * 8, cudaMemcpyHostToDevice, s));
    if (b->work_bytes) CU_TRY(cudaMemcpyAsync(D + b->o_init, H + s_init, b->work_bytes, cudaMemcpyHostToDevice, s));
    if (!gj.empty()) CU_TRY(cudaMemcpyAsync(D + b->o_gjobs, H + s_jobs, gj.size() * sizeof(plm::GridJob), cudaMemcpyHostToDevice, s));
    CU_TRY(cudaStreamSynchronize(s));

    b->kind = 2;
    b->n_jobs = n_jobs;
    b->n_m = n_m;
    b->best_lr = best_lr ? 1 : 0;
    std::memset(&b->gp, 0, sizeof(b->gp));
    b->gp.grid_rows = grid_rows;
    b->gp.grid_cols = grid_cols;
    b->gp.best_lr = b->best_lr;
    b->gp.ratio = ratio;
    b->gp.line_sim_th = line_sim_th;
    b->n1_max = n1_max;
    b->n2_max = n2_max;
    b->h2d = static_cast<int64_t>(size_t(n_rows) * 32 + size_t(n_coords) * 4 + size_t(n_cell_start) * 4 +
                                  size_t(n_cell_items) * 4 + size_t(n_dirs2) * 8 + S.total);
    b->d2h = static_cast<int64_t>(size_t(n_m) * 4 + size_t(n_jobs) * 4);
    return PLM_OK;
}

PLM_API int plm_batch_run(plm_batch *b) {
    if (!b || b->kind == 0) return fail(PLM_E_INVALID, "batch not prepared");
    plm_ctx *ctx = b->ctx;
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    cudaStream_t s = ctx->stream;
    char *D = b->d_buf;
    if (b->work_bytes) CU_TRY(cudaMemcpyAsync(D + b->o_work, D + b->o_init, b->work_bytes, cudaMemcpyDeviceToDevice, s));
    if (b->n_jobs == 0) return PLM_OK;
    if (b->kind == 1) {
        if (b->n_slice_ctas == 0) return PLM_OK;
        const plm::KnnTask *tasks = reinterpret_cast<const plm::KnnTask *>(D + b->o_tasks);
        if (b->best_lr && b->m21_bytes) CU_TRY(cudaMemsetAsync(D + b->o_m21, 0xFF, b->m21_bytes, s));
        // batches of short train sets (per-keyframe-pair loop closure, replay stages) are throughput work: the 13-LOP3
        // distance with the per-pair update (variant 5) unless a variant is forced; single calls keep variant 1, whose
        // stages need no in-place transform (lower latency)
        (void)knn_variant_for(0); // reads PLM_KNN_VARIANT on first use
        const int forced = g_knn_variant;
        if (forced == 0)
            plm::knn2_slice_list_kernel<BATCH_THREADS, 0><<<b->n_slice_ctas, BATCH_THREADS, 0, s>>>(tasks, reinterpret_cast<const int4 *>(D + b->o_cta_map));
        else if (forced == 1)
            plm::knn2_slice_list_kernel<BATCH_THREADS, 1><<<b->n_slice_ctas, BATCH_THREADS, 0, s>>>(tasks, reinterpret_cast<const int4 *>(D + b->o_cta_map));
        else
            plm::knn2_slice_list_kernel<BATCH_THREADS, 5><<<b->n_slice_ctas, BATCH_THREADS, 0, s>>>(tasks, reinterpret_cast<const int4 *>(D + b->o_cta_map));
        ctx->launches++;
        CU_TRY(cudaGetLastError());
        plm::knn2_merge_list_kernel<<<b->n_merge_ctas, BATCH_THREADS, 0, s>>>(tasks, reinterpret_cast<const int2 *>(D + b->o_merge_map), b->nnr, 1);
        ctx->launches++;
        CU_TRY(cudaGetLastError());
        if (b->best_lr && b->n_x_ctas) {
            plm::cross_check_list_kernel<<<b->n_x_ctas, 128, 0, s>>>(reinterpret_cast<const plm::XJob *>(D + b->o_xjobs), reinterpret_cast<const int2 *>(D + b->o_xmap));
            ctx->launches++;
            CU_TRY(cudaGetLastError());
        }
        return PLM_OK;
    }
    return launch_grid_fused(ctx, reinterpret_cast<const plm::GridJob *>(D + b->o_gjobs), b->n_jobs, b->gp, b->n1_max, b->n2_max,
                             b->items_max, b->any_lines);
}

PLM_API int plm_batch_fetch(plm_batch *b, int32_t *m12_arena, int32_t *counts) {
    if (!b || b->kind == 0) return fail(PLM_E_INVALID, "batch not prepared");
    plm_ctx *ctx = b->ctx;
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    cudaStream_t s = ctx->stream;
    char *D = b->d_buf;
    if (m12_arena && b->n_m > 0) CU_TRY(cudaMemcpyAsync(m12_arena, D + b->o_work, size_t(b->n_m) * 4, cudaMemcpyDeviceToHost, s));
    if (counts && b->n_jobs > 0)
        CU_TRY(cudaMemcpyAsync(counts, D + b->o_work + align_up(size_t(b->n_m) * 4, 16), size_t(b->n_jobs) * 4, cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaStreamSynchronize(s));
    return PLM_OK;
}

// ---------------------------------------------------------------------------------------------

// ---------------------------------------------------------------------------------------------
// Frame session: the host-buffer calls of one frame (stereo matchGrid for points and lines, temporal match for
// points and lines, ...) executed as ONE round trip.
namespace {

int frame_run(plm_ctx *ctx, const plm_ctx::FrameCall &c, Exec *ex) {
    if (c.kind == 0) return match_impl(ctx, c.d1, c.n1, c.step1, c.d2, c.n2, c.step2, c.nnr, c.best_lr, c.m12, c.n_matches, ex);
    return match_grid_impl(ctx, c.is_lines, c.coords, c.d1, c.n1, c.step1, c.cell_start, c.cell_items, c.grid_rows, c.grid_cols, c.d2, c.n2,
                           c.step2, c.dirs2, c.line_sim_th, c.win, c.ratio, c.best_lr, c.m12, c.n_matches, ex);
}

// The whole session as ONE launch (csrc/plm_frame_fused.cuh): job table + in/out vectors + inputs of every call in one
// pinned block -> one copy in, frame_fused_kernel (clusters of 8 CTAs per call), which stores the final in/out vectors and
// counts straight into the pinned block (zero-copy), one synchronisation.
// *done stays false when a call does not fit the fused kernel (the caller then runs one lane per call).
int frame_end_fused(plm_ctx *ctx, const plm_ctx::FrameCall *calls, int n, bool *done) {
    *done = false;
    if (!g_frame_fused || g_grid_cluster < 2 || n > plm::FRAME_MAX_JOBS) return PLM_OK;
    struct Plan {
        size_t o_io = 0, o_d1 = 0, o_d2 = 0, o_xy = 0, o_cs = 0, o_ci = 0, o_dir = 0, o_scr = 0;
        int n_items = 0, n_cta = plm::FRAME_CLUSTER, c12 = 0;
        plm::GridParams gp;
    };
    std::vector<Plan> plan(n);
    Layout L;
    for (int k = 0; k < n; ++k) plan[k].o_io = L.add(size_t(calls[k].n1) * 4 + 8); // m12, the counter, the arrival counter of a match job
    size_t smem = 0;
    for (int k = 0; k < n; ++k) {
        const plm_ctx::FrameCall &c = calls[k];
        Plan &p = plan[k];
        std::memset(&p.gp, 0, sizeof(p.gp));
        p.o_d1 = L.add(size_t(c.n1) * 32);
        p.o_d2 = L.add(size_t(std::max(c.n2, 1)) * 32);
        if (c.kind == 0) {
            if (c.n1 > plm::FRAME_MATCH_MAX_ROWS || c.n2 > plm::FRAME_MATCH_MAX_ROWS) return PLM_OK;
            smem = std::max(smem, plm::match_cta_smem(c.n1, c.n2, c.best_lr));
            // ~24 query rows per CTA (both directions count), whole clusters, at most 64 CTAs per job
            const int q_rows = c.n1 + (c.best_lr ? c.n2 : 0);
            p.n_cta = std::min(64, (q_rows + 24 * plm::FRAME_CLUSTER - 1) / (24 * plm::FRAME_CLUSTER) * plm::FRAME_CLUSTER);
            p.c12 = p.n_cta;
            if (c.best_lr) p.c12 = std::max(1, std::min(p.n_cta - 1, static_cast<int>((static_cast<long long>(p.n_cta) * c.n1 + q_rows / 2) / std::max(q_rows, 1))));
            continue;
        }
        if (c.n1 > plm::FRAME_CLUSTER * plm::GRID_ROW_THREADS || c.n1 >= (1 << plm::GRID_KEY_BITS)) return PLM_OK;
        const int n_cells = c.grid_rows * c.grid_cols;
        p.n_items = c.cell_start[n_cells];
        size_t job_smem = 0;
        if (!plan_grid_rows_smem(ctx, std::max(c.n2, 1), n_cells, c.is_lines != 0, p.gp, job_smem)) return PLM_OK;
        smem = std::max(smem, job_smem);
        // the rows are spread over the 8 CTAs of the cluster in multiples of a warp
        int rpc = ((c.n1 + plm::FRAME_CLUSTER - 1) / plm::FRAME_CLUSTER + 31) / 32 * 32;
        p.gp.rows_per_cta = std::min(rpc, plm::GRID_ROW_THREADS);
        p.gp.grid_rows = c.grid_rows;
        p.gp.grid_cols = c.grid_cols;
        p.gp.best_lr = c.best_lr ? 1 : 0;
        p.gp.ratio = c.ratio;
        p.gp.line_sim_th = c.line_sim_th;
        p.o_xy = L.add(size_t(c.n1) * (c.is_lines ? 4 : 2) * 4);
        p.o_cs = L.add(size_t(n_cells + 1) * 4);
        p.o_ci = L.add(size_t(std::max(p.n_items, 1)) * 4);
        p.o_dir = L.add(c.is_lines ? size_t(std::max(c.n2, 1)) * 16 : 0);
    }
    const size_t in_end = L.total;
    for (int k = 0; k < n; ++k) // device-only scratch: matches_21 (match) / per-column keys (matchGrid)
        plan[k].o_scr = L.add(size_t(std::max(calls[k].n2, 1)) * (calls[k].kind == 0 ? 4 : 8));
    if (smem > ctx->smem_optin - 2048) return PLM_OK;
    int st;
    if ((st = ctx->ensure_pinned(in_end)) != PLM_OK) return st;
    if (!ctx->h_buf_dev) return PLM_OK; // no device mapping of the pinned block: one lane per call
    if ((st = ctx->ensure_device(L.total)) != PLM_OK) return st;
    if (!ctx->frame_fused_attr_set) {
        CU_TRY(cudaFuncSetAttribute(plm::frame_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(ctx->smem_optin - 2048)));
        ctx->frame_fused_attr_set = true;
    }
    static const bool trace = std::getenv("PLM_FRAME_TRACE") != nullptr;
    static thread_local double t_acc[5] = {0, 0, 0, 0, 0};
    static thread_local int t_n = 0;
    const auto t0 = std::chrono::steady_clock::now();
    char *HB = ctx->h_buf, *DB = ctx->d_buf;
    plm::FrameTable table; // travels as the kernel parameter
    std::memset(&table, 0, sizeof(table));
    plm::FrameJobRec *tab = table.job;
    int n_cta_total = 0;
    for (int k = 0; k < n; ++k) {
        const plm_ctx::FrameCall &c = calls[k];
        const Plan &p = plan[k];
        plm::FrameJobRec &r = tab[k];
        std::memset(&r, 0, sizeof(r));
        r.kind = c.kind;
        pack_rows(HB + p.o_d1, c.d1, c.n1, c.step1);
        pack_rows(HB + p.o_d2, c.d2, c.n2, c.step2);
        std::memcpy(HB + p.o_io, c.m12, size_t(c.n1) * 4);
        std::memset(HB + p.o_io + size_t(c.n1) * 4, 0, 8);
        int32_t *dm12 = reinterpret_cast<int32_t *>(DB + p.o_io);
        r.cta_begin = n_cta_total;
        r.h_io = reinterpret_cast<int32_t *>(ctx->h_buf_dev + p.o_io); // the pinned block as the device addresses it
        n_cta_total += p.n_cta;
        if (c.kind == 0) {
            r.mj.done = dm12 + c.n1 + 1;
            r.mj.n_cta = p.n_cta;
            r.mj.c12 = p.c12;
            r.mj.d1 = reinterpret_cast<const uint4 *>(DB + p.o_d1);
            r.mj.d2 = reinterpret_cast<const uint4 *>(DB + p.o_d2);
            r.mj.m12 = dm12;
            r.mj.count = dm12 + c.n1;
            r.mj.m21 = reinterpret_cast<int32_t *>(DB + p.o_scr);
            r.mj.n1 = c.n1;
            r.mj.n2 = c.n2;
            r.mj.best_lr = c.best_lr ? 1 : 0;
            r.mj.nnr = c.nnr;
            continue;
        }
        const int n_cells = c.grid_rows * c.grid_cols;
        std::memcpy(HB + p.o_xy, c.coords, size_t(c.n1) * (c.is_lines ? 4 : 2) * 4);
        std::memcpy(HB + p.o_cs, c.cell_start, size_t(n_cells + 1) * 4);
        if (p.n_items > 0) std::memcpy(HB + p.o_ci, c.cell_items, size_t(p.n_items) * 4);
        if (c.is_lines && c.n2 > 0) std::memcpy(HB + p.o_dir, c.dirs2, size_t(c.n2) * 16);
        r.gj.coords = reinterpret_cast<const int32_t *>(DB + p.o_xy);
        r.gj.d1 = reinterpret_cast<const uint4 *>(DB + p.o_d1);
        r.gj.cell_start = reinterpret_cast<const int32_t *>(DB + p.o_cs);
        r.gj.cell_items = reinterpret_cast<const int32_t *>(DB + p.o_ci);
        r.gj.d2 = reinterpret_cast<const uint4 *>(DB + p.o_d2);
        r.gj.dirs2 = reinterpret_cast<const double *>(DB + p.o_dir);
        r.gj.m12 = dm12;
        r.gj.count = dm12 + c.n1;
        r.gj.n1 = c.n1;
        r.gj.n2 = c.n2;
        r.gj.is_lines = c.is_lines;
        for (int i = 0; i < 4; ++i) r.gj.win[i] = c.win[i];
        r.gp = p.gp;
        r.gp.n_items_p1 = p.n_items + 1;
        r.gp.m21key = reinterpret_cast<unsigned long long *>(DB + p.o_scr);
    }
    table.n_jobs = n;
    table.n_cta = n_cta_total;
    const auto t1 = std::chrono::steady_clock::now();
    CU_TRY(cudaMemcpyAsync(DB, HB, in_end, cudaMemcpyHostToDevice, ctx->stream));
    const auto t2 = std::chrono::steady_clock::now();
    cudaLaunchConfig_t cfg;
    std::memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(n_cta_total, 1, 1);
    cfg.blockDim = dim3(plm::GRID_ROW_THREADS, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = plm::FRAME_CLUSTER;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    CU_TRY(cudaLaunchKernelEx(&cfg, plm::frame_fused_kernel, table));
    ctx->launches++;
    const auto t3 = std::chrono::steady_clock::now();
    const auto t4 = t3; // no copy out: the kernel stores the results into the pinned block itself
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    if (trace) {
        const auto t5 = std::chrono::steady_clock::now();
        auto us = [](auto a, auto b) { return std::chrono::duration<double, std::micro>(b - a).count(); };
        t_acc[0] += us(t0, t1); t_acc[1] += us(t1, t2); t_acc[2] += us(t2, t3); t_acc[3] += us(t3, t4); t_acc[4] += us(t4, t5);
        if (++t_n % 200 == 0) {
            std::fprintf(stderr, "[frame_fused] pack %.1f  h2d-issue %.1f  launch %.1f  d2h-issue %.1f  sync %.1f us  (in %zu B, smem %zu)\n",
                         t_acc[0] / 200, t_acc[1] / 200, t_acc[2] / 200, t_acc[3] / 200, t_acc[4] / 200, in_end, smem);
            for (double &v : t_acc) v = 0;
        }
    }
    for (int k = 0; k < n; ++k) {
        const plm_ctx::FrameCall &c = calls[k];
        std::memcpy(c.m12, HB + plan[k].o_io, size_t(c.n1) * 4);
        int32_t cnt;
        std::memcpy(&cnt, HB + plan[k].o_io + size_t(c.n1) * 4, 4);
        *c.n_matches = cnt;
    }
    *done = true;
    return PLM_OK;
}

} // namespace

#ifdef PLM_TIMELINE
// debug builds: the phase stamps of the last frame_fused_kernel launch, [128 CTAs][24] SM clock values
extern "C" __attribute__((visibility("default"))) int plm_debug_timeline(long long *out) {
    cudaDeviceSynchronize();
    return cudaMemcpyFromSymbol(out, plm::g_timeline, sizeof(long long) * 128 * 24) == cudaSuccess ? 0 : -1;
}
#endif

PLM_API int plm_frame_begin(plm_ctx *ctx) {
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    if (ctx->in_frame) return fail(PLM_E_INVALID, "plm_frame_begin: a frame session is already open on this context");
    ctx->in_frame = true;
    ctx->frame_calls.clear();
    return PLM_OK;
}

PLM_API int plm_frame_active(plm_ctx *ctx) {
    if (!ctx) ctx = g_tls.ctx;
    return ctx && ctx->in_frame ? 1 : 0;
}

PLM_API int plm_frame_end(plm_ctx *ctx) {
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    if (!ctx->in_frame) return fail(PLM_E_INVALID, "plm_frame_end without plm_frame_begin");
    ctx->in_frame = false;
    std::vector<plm_ctx::FrameCall> calls;
    calls.swap(ctx->frame_calls);
    const int n = static_cast<int>(calls.size());
    if (n == 0) return PLM_OK;
    bool fused_done = false;
    if ((st = frame_end_fused(ctx, calls.data(), n, &fused_done)) != PLM_OK) return st;
    if (fused_done) return PLM_OK;
    std::vector<Exec> ex(n);
    size_t h_total = 0, d_total = 0;
    std::vector<size_t> h_off(n), d_off(n);
    for (int k = 0; k < n; ++k) {
        ex[k].phase = EXEC_SIZE;
        if ((st = frame_run(ctx, calls[k], &ex[k])) != PLM_OK) return st;
        h_off[k] = h_total;
        d_off[k] = d_total;
        h_total += align_up(ex[k].h_bytes);
        d_total += align_up(ex[k].d_bytes);
    }
    if ((st = ctx->ensure_pinned(h_total)) != PLM_OK) return st;
    if ((st = ctx->ensure_device(d_total)) != PLM_OK) return st;
    if (!ctx->frame_streams[0]) {
        for (int i = 0; i < 3; ++i) CU_TRY(cudaStreamCreateWithFlags(&ctx->frame_streams[i], cudaStreamNonBlocking));
        for (int i = 0; i < 4; ++i) CU_TRY(cudaEventCreateWithFlags(&ctx->frame_events[i], cudaEventDisableTiming));
    }
    // the calls are independent: each is packed and immediately launched (copy in, kernels, copy out) on its own lane,
    // round-robin over four streams, so the packing of call k + 1 overlaps the device work of call k and the kernels
    // of different calls run side by side
    cudaStream_t main_stream = ctx->stream;
    cudaStream_t lanes[4] = {main_stream, ctx->frame_streams[0], ctx->frame_streams[1], ctx->frame_streams[2]};
    const int n_lanes = std::min(n, 4);
    if (n_lanes > 1) {
        CU_TRY(cudaEventRecord(ctx->frame_events[0], main_stream)); // earlier work of this context comes first
        for (int i = 1; i < n_lanes; ++i) CU_TRY(cudaStreamWaitEvent(lanes[i], ctx->frame_events[0], 0));
    }
    int rc = PLM_OK;
    for (int k = 0; k < n && rc == PLM_OK; ++k) {
        ex[k].h_base = ctx->h_buf + h_off[k];
        ex[k].d_base = ctx->d_buf + d_off[k];
        ex[k].phase = EXEC_PACK;
        if ((rc = frame_run(ctx, calls[k], &ex[k])) != PLM_OK) break;
        ctx->stream = lanes[k % n_lanes];
        ex[k].phase = EXEC_LAUNCH;
        rc = frame_run(ctx, calls[k], &ex[k]);
    }
    ctx->stream = main_stream;
    for (int i = 1; i < n_lanes; ++i) {
        cudaEventRecord(ctx->frame_events[i], lanes[i]);
        cudaStreamWaitEvent(main_stream, ctx->frame_events[i], 0);
    }
    CU_TRY(cudaStreamSynchronize(main_stream));
    if (rc != PLM_OK) return rc;
    for (int k = 0; k < n; ++k) {
        ex[k].phase = EXEC_UNPACK;
        if ((st = frame_run(ctx, calls[k], &ex[k])) != PLM_OK) return st;
    }
    return PLM_OK;
}

// ---------------------------------------------------------------------------------------------
// Local-map selection and reprojection gates of matchMap2KF* (csrc/plm_reproj.cuh)
namespace {

plm::MapView to_view(const plm_map_view *v) {
    plm::MapView m;
    for (int i = 0; i < 12; ++i) m.T[i] = v->T[i];
    m.fx = v->fx; m.fy = v->fy; m.cx = v->cx; m.cy = v->cy;
    m.inv_width = v->inv_width; m.inv_height = v->inv_height;
    m.width = v->width; m.height = v->height;
    return m;
}

} // namespace

PLM_API int plm_dev_map_select(plm_ctx *ctx, int is_lines, const double *X_dev, const uint8_t *active_dev, int n, const plm_map_view *v,
                               int32_t *sel_dev, int32_t *coords_dev, double *pf_dev, int32_t *n_sel_dev) {
    if (n < 0 || !v || !n_sel_dev) return fail(PLM_E_INVALID, "negative size / null view / null n_sel");
    if (n > 0 && (!X_dev || !sel_dev || !coords_dev || !pf_dev)) return fail(PLM_E_INVALID, "null pointer");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    if (n == 0) {
        CU_TRY(cudaMemsetAsync(n_sel_dev, 0, 4, ctx->stream));
        return PLM_OK;
    }
    const int n_cta = (n + 255) / 256;
    if ((st = ctx->ensure_aux(size_t(n_cta) * 4)) != PLM_OK) return st;
    int32_t *cnt = reinterpret_cast<int32_t *>(ctx->d_aux);
    const plm::MapView mv = to_view(v);
    for (int pass = 0; pass < 2; ++pass) {
        if (is_lines) plm::map_select_kernel<2><<<n_cta, 256, 0, ctx->stream>>>(X_dev, active_dev, n, mv, pass, cnt, sel_dev, coords_dev, pf_dev, n_sel_dev);
        else plm::map_select_kernel<1><<<n_cta, 256, 0, ctx->stream>>>(X_dev, active_dev, n, mv, pass, cnt, sel_dev, coords_dev, pf_dev, n_sel_dev);
        ctx->launches++;
        CU_TRY(cudaGetLastError());
        if (pass == 0) {
            plm::map_count_scan_kernel<<<1, 1024, 0, ctx->stream>>>(cnt, n_cta);
            ctx->launches++;
            CU_TRY(cudaGetLastError());
        }
    }
    return PLM_OK;
}

PLM_API int plm_dev_gather_rows(plm_ctx *ctx, const void *rows_dev, const int32_t *sel_dev, const int32_t *n_sel_dev, int n_max, void *out_dev) {
    if (n_max < 0) return fail(PLM_E_INVALID, "negative size");
    if (n_max == 0) return PLM_OK;
    if (!rows_dev || !sel_dev || !n_sel_dev || !out_dev) return fail(PLM_E_INVALID, "null pointer");
    if ((reinterpret_cast<uintptr_t>(rows_dev) | reinterpret_cast<uintptr_t>(out_dev)) & 15) return fail(PLM_E_INVALID, "device descriptor pointers must be 16-byte aligned");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    plm::gather_rows_kernel<<<(n_max + 255) / 256, 256, 0, ctx->stream>>>(static_cast<const uint4 *>(rows_dev), sel_dev, n_sel_dev, static_cast<uint4 *>(out_dev));
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    return PLM_OK;
}

PLM_API int plm_dev_map_gate(plm_ctx *ctx, int is_lines, const double *pf_dev, const int32_t *m12_dev, const int32_t *n_sel_dev, int n_max,
                             const double *feat_dev, int n2, double max_epip, uint8_t *ok_dev, int32_t *count_inout_dev) {
    if (n_max < 0 || n2 < 0) return fail(PLM_E_INVALID, "negative size");
    if (n_max == 0) return PLM_OK;
    if (!pf_dev || !m12_dev || !n_sel_dev || !ok_dev || !count_inout_dev || (n2 > 0 && !feat_dev)) return fail(PLM_E_INVALID, "null pointer");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    if (is_lines) plm::map_gate_kernel<1><<<(n_max + 255) / 256, 256, 0, ctx->stream>>>(pf_dev, m12_dev, n_sel_dev, feat_dev, n2, max_epip, ok_dev, count_inout_dev);
    else plm::map_gate_kernel<0><<<(n_max + 255) / 256, 256, 0, ctx->stream>>>(pf_dev, m12_dev, n_sel_dev, feat_dev, n2, max_epip, ok_dev, count_inout_dev);
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    return PLM_OK;
}

// Host-buffer forms (tests, hosts that keep the landmarks in host memory).
PLM_API int plm_map_select(plm_ctx *ctx, int is_lines, const double *X, const uint8_t *active, int n, const plm_map_view *v, int32_t *sel,
                           int32_t *coords, double *pf, int *n_sel) {
    if (n < 0 || !v || !n_sel) return fail(PLM_E_INVALID, "negative size / null view / null n_sel");
    *n_sel = 0;
    if (n == 0) return PLM_OK;
    if (!X || !sel || !coords || !pf) return fail(PLM_E_INVALID, "null pointer");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    const int per = is_lines ? 2 : 1;
    Layout L;
    const size_t o_x = L.add(size_t(n) * 24 * per), o_act = L.add(active ? size_t(n) : 0), o_sel = L.add(size_t(n) * 4 + 16),
                 o_co = L.add(size_t(n) * 8 * per), o_pf = L.add(size_t(n) * 16 * per);
    if ((st = ctx->ensure_device(L.total)) != PLM_OK) return st;
    char *D = ctx->d_buf;
    CU_TRY(cudaMemcpyAsync(D + o_x, X, size_t(n) * 24 * per, cudaMemcpyHostToDevice, ctx->stream));
    if (active) CU_TRY(cudaMemcpyAsync(D + o_act, active, size_t(n), cudaMemcpyHostToDevice, ctx->stream));
    int32_t *d_sel = reinterpret_cast<int32_t *>(D + o_sel), *d_n = d_sel + n;
    if ((st = plm_dev_map_select(ctx, is_lines, reinterpret_cast<const double *>(D + o_x), active ? reinterpret_cast<const uint8_t *>(D + o_act) : nullptr, n,
                                 v, d_sel, reinterpret_cast<int32_t *>(D + o_co), reinterpret_cast<double *>(D + o_pf), d_n)) != PLM_OK)
        return st;
    int32_t cnt = 0;
    CU_TRY(cudaMemcpyAsync(&cnt, d_n, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    if (cnt > 0) {
        CU_TRY(cudaMemcpyAsync(sel, d_sel, size_t(cnt) * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU_TRY(cudaMemcpyAsync(coords, D + o_co, size_t(cnt) * 8 * per, cudaMemcpyDeviceToHost, ctx->stream));
        CU_TRY(cudaMemcpyAsync(pf, D + o_pf, size_t(cnt) * 16 * per, cudaMemcpyDeviceToHost, ctx->stream));
        CU_TRY(cudaStreamSynchronize(ctx->stream));
    }
    *n_sel = cnt;
    return PLM_OK;
}

PLM_API int plm_map_gate(plm_ctx *ctx, int is_lines, const double *pf, const int32_t *m12, int n_sel, const double *feat, int n2, double max_epip,
                         uint8_t *ok, int *count_inout) {
    if (n_sel < 0 || n2 < 0 || !count_inout) return fail(PLM_E_INVALID, "negative size / null count");
    if (n_sel == 0) return PLM_OK;
    if (!pf || !m12 || !ok || (n2 > 0 && !feat)) return fail(PLM_E_INVALID, "null pointer");
    int st = resolve_ctx(ctx);
    if (st != PLM_OK) return st;
    const int per = is_lines ? 2 : 1, fw = is_lines ? 3 : 2;
    Layout L;
    const size_t o_pf = L.add(size_t(n_sel) * 16 * per), o_m = L.add(size_t(n_sel) * 4), o_f = L.add(size_t(std::max(n2, 1)) * 8 * fw),
                 o_ok = L.add(size_t(n_sel)), o_c = L.add(16);
    if ((st = ctx->ensure_device(L.total)) != PLM_OK) return st;
    char *D = ctx->d_buf;
    int32_t head[2] = {n_sel, *count_inout};
    CU_TRY(cudaMemcpyAsync(D + o_pf, pf, size_t(n_sel) * 16 * per, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(cudaMemcpyAsync(D + o_m, m12, size_t(n_sel) * 4, cudaMemcpyHostToDevice, ctx->stream));
    if (n2 > 0) CU_TRY(cudaMemcpyAsync(D + o_f, feat, size_t(n2) * 8 * fw, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(cudaMemcpyAsync(D + o_c, head, 8, cudaMemcpyHostToDevice, ctx->stream));
    int32_t *d_head = reinterpret_cast<int32_t *>(D + o_c);
    if ((st = plm_dev_map_gate(ctx, is_lines, reinterpret_cast<const double *>(D + o_pf), reinterpret_cast<const int32_t *>(D + o_m), d_head, n_sel,
                               reinterpret_cast<const double *>(D + o_f), n2, max_epip, reinterpret_cast<uint8_t *>(D + o_ok), d_head + 1)) != PLM_OK)
        return st;
    CU_TRY(cudaMemcpyAsync(ok, D + o_ok, size_t(n_sel), cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaMemcpyAsync(head, d_head, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    *count_inout = head[1];
    return PLM_OK;
}

#include "plm_frames_api.inl"
#include "plm_shard_api.inl"
#include "plm_loopdb_api.inl"
