// Both directions of every keyframe pair of a batch on the tensor cores (K1c, knn2_umma_pairs_kernel): the pipeline of
// plm_knn2_umma.cuh with a unit table as its unit source and a two-direction readout.
//
// A loop-closure batch (KeyframeDB.match_all, plm_loopdb_match) runs StVO::match of ONE query keyframe Q (n1 rows)
// against many keyframes K_j.  Both directions of a pair are the same distance matrix D_j = d(Q, K_j): the top-2 of a
// row of D_j inside K_j's columns is direction 12, the top-2 of a column of D_j over the rows of Q is direction 21.  So
// one exact int8 product per (query group, 128-row unit) serves both directions of every pair.
//
// Units: the host cuts every live job's train rows into units of <= 128 consecutive rows (units never cross jobs;
// units[u] = (job, first row of the unit in the job), job-major); unit u is read from the arena at the job's train
// offset.  A run of units of one (group, job) inside a CTA's share is a PIECE; its index among the CTAs that scan that
// (group, job) is the partial slot of direction 12.
// Readout:
//   * direction 12 (thread = query row): the pipeline's blocked top-2 over the unit's columns -- exact, columns ascend
//     within a job.  Keys carry the row index local to the job (as the integer list kernels), and the threshold is the
//     thread's own second best (no shared bound).  At the end of a piece the thread writes (best, second) to the job's
//     part12[slot][q] and starts over; the last piece of a (group, job) writes absent into the slots nobody used.
//   * direction 21 (column = train row, BOTH only): per accumulator value one IMAD makes the 32-bit key
//     (|q| + v) << 8 | q (q < 256 the row in the group; padding rows past n1 give 0xFFFFFFFF); per column a warp takes
//     two __reduce_min_sync (min, then min without it).  The 8 warps leave (m1, m2) per column in shared memory
//     (8 KB per accumulator buffer, double-buffered); after a named barrier of the readout warps thread c < rows merges
//     column c's 16 keys and writes (d << 32 | g * 256 + q) pairs to the job's part21[g][row].  Every (group, row) is
//     written exactly once, so columns keep no state across units.
// knn2_merge_list_kernel and cross_check_list_kernel then run unchanged on these partials (plm_batch_run).
#pragma once
#include "plm_knn2_umma.cuh"

namespace plm {

// One live job of the batch (device table).
struct PairsJob {
    long long train_off;  // first train row of the job in the arena
    ulonglong2 *part12;   // [n_slots12][n1] direction-12 partials (the job's 12 task)
    ulonglong2 *part21;   // [groups][n2] direction-21 partials (the job's 21 task; null without best_lr)
    int n2, unit0, n_units, n_slots12;
};
struct PairsTask {
    const uint4 *q;       // the n1 query rows every job shares
    const uint4 *arena;   // train rows
    const PairsJob *jobs;
    const int2 *units;    // [n_units] (job, first row of the unit within the job), job-major
    int n1, n_units;
};

// the pipeline's shared memory + the per-warp column minima of direction 21: [2 accumulator buffers][8 warps][128 columns] uint2
constexpr int KNN_UMMA_PAIRS_COLBUF = 2 * 8 * KNN_UMMA_ROWS * 8;
constexpr int KNN_UMMA_PAIRS_SMEM = KNN_UMMA_SMEM + KNN_UMMA_PAIRS_COLBUF;

template <bool BOTH>
struct PairsScan {
    static constexpr bool PACKED = false; // direction 21 reduces the exact 32-bit values of each half (loaded)
    PairsTask t;
    // per segment
    uint32_t base21; // direction-21 key of this row: (|q| + v) << 8 | row in the group = v * 256 + base21
    int2 un;         // the unit the readout is at
    int un_rows;     // and its row count, read before the unit's accumulator wait

    __device__ __forceinline__ const uint4 *unit_src(long long u, int &rows) const {
        const int2 un = __ldg(t.units + u);
        const PairsJob &jb = t.jobs[un.x];
        rows = min(KNN_UMMA_ROWS, jb.n2 - un.y);
        return t.arena + 2 * (jb.train_off + un.y);
    }
    __device__ __forceinline__ void read_unit(long long u) {
        un = __ldg(t.units + u);
        un_rows = min(KNN_UMMA_ROWS, t.jobs[un.x].n2 - un.y);
    }
    __device__ __forceinline__ uint2 *colbuf() const { return reinterpret_cast<uint2 *>(umma_smem() + KNN_UMMA_PIPE_BYTES); }
    __device__ __forceinline__ void begin_segment(const UmmaSeg &s) {
        base21 = s.valid ? (static_cast<uint32_t>(s.qn) << 8) | static_cast<uint32_t>(threadIdx.x) : 0xFFFFFFFFu; // v = 0 on padding rows
        read_unit(s.u0);
    }
    __device__ __forceinline__ UmmaCols begin_unit(const UmmaSeg &, int, int &) const { return {un_rows, static_cast<uint32_t>(un.y)}; }
    __device__ __forceinline__ int threshold(unsigned long long B1) const { return (B1 == KEY64_ABSENT) ? 1023 : static_cast<int>(B1 >> 32); }
    __device__ __forceinline__ void loaded(int (&v)[2][32], int half, uint32_t k) const {
        if (!BOTH) return;
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            uint32_t r1 = 0xFFFFFFFFu, r2 = 0xFFFFFFFFu; // lane jj keeps column jj's two smallest keys of the warp
#pragma unroll
            for (int jj = 0; jj < 32; ++jj) {
                const uint32_t key = static_cast<uint32_t>(v[q][jj]) * 256u + base21;
                const uint32_t m1 = __reduce_min_sync(0xFFFFFFFFu, key);
                const uint32_t m2 = __reduce_min_sync(0xFFFFFFFFu, key == m1 ? 0xFFFFFFFFu : key);
                if (lane == jj) {
                    r1 = m1;
                    r2 = m2;
                }
            }
            colbuf()[(k * 8 + warp) * KNN_UMMA_ROWS + 64 * half + 32 * q + lane] = make_uint2(r1, r2);
        }
    }
    __device__ __forceinline__ void end_unit(const UmmaSeg &s, int i, uint32_t k, int rows, unsigned long long &B0, unsigned long long &B1, int &thr) {
        const PairsJob &jb = t.jobs[un.x];
        const int tid = threadIdx.x;
        if (BOTH) { // column tid of the unit: the two smallest of the 8 warps' pairs -> part21[g][row]
            asm volatile("bar.sync 1, %0;" ::"n"(KNN_UMMA_THREADS) : "memory"); // the readout warps only
            if (tid < rows) {
                uint32_t b0 = 0xFFFFFFFFu, b1 = 0xFFFFFFFFu;
#pragma unroll
                for (int w = 0; w < 8; ++w) {
                    const uint2 p = colbuf()[(k * 8 + w) * KNN_UMMA_ROWS + tid];
                    top2_insert(b0, b1, p.x);
                    top2_insert(b0, b1, p.y);
                }
                const uint32_t qb = static_cast<uint32_t>(s.g) * KNN_UMMA_THREADS;
                const unsigned long long k0 = b0 == 0xFFFFFFFFu ? KEY64_ABSENT : make_key64(b0 >> 8, qb + (b0 & 255u));
                const unsigned long long k1 = b1 == 0xFFFFFFFFu ? KEY64_ABSENT : make_key64(b1 >> 8, qb + (b1 & 255u));
                jb.part21[static_cast<size_t>(s.g) * jb.n2 + un.y + tid] = make_ulonglong2(k0, k1);
            }
        }
        // end of a piece (the next unit is another job's, or the segment ends): direction-12 partials
        const int job = un.x;
        if (i + 1 < s.n) read_unit(s.u0 + i + 1);
        if (i + 1 == s.n || un.x != job) {
            if (s.valid) {
                const int slot = umma_slot(static_cast<long long>(s.g) * t.n_units + jb.unit0, t.n1, t.n_units);
                jb.part12[static_cast<size_t>(slot) * t.n1 + s.qi] = make_ulonglong2(B0, B1);
                if (s.u0 + i + 1 == jb.unit0 + jb.n_units) // the last piece of (group, job)
                    for (int p = slot + 1; p < jb.n_slots12; ++p) jb.part12[static_cast<size_t>(p) * t.n1 + s.qi] = make_ulonglong2(KEY64_ABSENT, KEY64_ABSENT);
            }
            B0 = B1 = KEY64_ABSENT;
            thr = s.valid ? 1023 : 0;
        }
    }
    __device__ __forceinline__ void end_segment(const UmmaSeg &, unsigned long long, unsigned long long) {}
};

template <bool BOTH>
__global__ void __launch_bounds__(KNN_UMMA_CTA_THREADS, 1) knn2_umma_pairs_kernel(const PairsTask t, int32_t *err, long long spin_limit) {
    PairsScan<BOTH> sc{t};
    umma_pipeline(sc, t.q, t.n1, t.n_units, err, spin_limit);
}

} // namespace plm
