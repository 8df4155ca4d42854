// Both directions of every keyframe pair of a batch on the tensor cores (K1c, knn2_umma_pairs_kernel).
//
// A loop-closure batch (KeyframeDB.match_all, plm_loopdb_match) runs StVO::match of ONE query keyframe Q (n1 rows)
// against many keyframes K_j.  Both directions of a pair are the same distance matrix D_j = d(Q, K_j): the top-2 of a
// row of D_j inside K_j's columns is direction 12, the top-2 of a column of D_j over the rows of Q is direction 21.  So
// one exact int8 product per (query group, 128-row unit) -- the same d = |q| + dot(+-1 query, 0/1 row) as K1b
// (plm_knn2_umma.cuh) -- serves both directions of every pair.
//
// Work list: the host cuts every live job's train rows into units of <= 128 consecutive rows (units never cross jobs;
// units[u] = (job, first row of the unit in the job), job-major) and the list is (query group of 256, unit),
// group-major.  Every CTA owns an equal contiguous share, as in K1b; A is rewritten only where the share crosses a
// group.  A run of units of one (group, job) inside a share is a PIECE; its index among the CTAs that scan that
// (group, job) (umma_cta_of, as K1b per group) is the partial slot of direction 12.
// Roles, barriers, rings, descriptors and the TMEM budget (512 columns, two accumulator buffers) are those of K1b; only
// the producer's addresses (per unit, from the unit table) and the readout differ:
//   * direction 12 (thread = query row): K1b's blocked top-2 over the unit's columns -- exact, columns ascend within a
//     job and the test is strict.  Keys carry the row index local to the job (as the integer list kernels).  At the end
//     of a piece the thread writes (best, second) to the job's part12[slot][q]; the last piece of a (group, job) writes
//     absent into the slots nobody used.
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

// K1b's shared memory + the per-warp column minima of direction 21: [2 accumulator buffers][8 warps][128 columns] uint2
constexpr int KNN_UMMA_PAIRS_COLBUF = 2 * 8 * KNN_UMMA_ROWS * 8;
constexpr int KNN_UMMA_PAIRS_SMEM = KNN_UMMA_SMEM + KNN_UMMA_PAIRS_COLBUF;

__device__ __forceinline__ void readout_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(KNN_UMMA_THREADS) : "memory"); }

template <bool BOTH>
__global__ void __launch_bounds__(KNN_UMMA_CTA_THREADS, 1) knn2_umma_pairs_kernel(const PairsTask t, int32_t *err, long long spin_limit) {
    extern __shared__ uint8_t smem_raw[];
    // packed full / empty [STAGES], B full / empty [BSTAGES], accumulator full / empty [2], A ready
    __shared__ __align__(8) unsigned long long mbar[2 * KNN_UMMA_STAGES + 2 * KNN_UMMA_BSTAGES + 5];
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint8_t *smem = smem_raw + ((1024 - (static_cast<uint32_t>(__cvta_generic_to_shared(smem_raw)) & 1023)) & 1023); // 1024-aligned
    uint8_t *tileA = smem;                                  // 2 M-tiles
    uint8_t *tileB = smem + 2 * KNN_UMMA_TILE_BYTES;        // BSTAGES unit tiles
    const uint4 *ring = reinterpret_cast<const uint4 *>(smem + (2 + KNN_UMMA_BSTAGES) * KNN_UMMA_TILE_BYTES);
    uint2 *colbuf = reinterpret_cast<uint2 *>(smem + (2 + KNN_UMMA_BSTAGES) * KNN_UMMA_TILE_BYTES + KNN_UMMA_STAGES * KNN_UMMA_ROWS * 32);
    const uint32_t sA = static_cast<uint32_t>(__cvta_generic_to_shared(tileA));
    const uint32_t sB = static_cast<uint32_t>(__cvta_generic_to_shared(tileB));
    const uint32_t sRing = static_cast<uint32_t>(__cvta_generic_to_shared(ring));
    const uint32_t PFULL = static_cast<uint32_t>(__cvta_generic_to_shared(mbar)), PEMPTY = PFULL + 8 * KNN_UMMA_STAGES;
    const uint32_t BFULL = PEMPTY + 8 * KNN_UMMA_STAGES, BEMPTY = BFULL + 8 * KNN_UMMA_BSTAGES;
    const uint32_t AFULL = BEMPTY + 8 * KNN_UMMA_BSTAGES, AEMPTY = AFULL + 16, AREADY = AEMPTY + 16;

    if (warp == 0) {
        const uint32_t slot = static_cast<uint32_t>(__cvta_generic_to_shared(&tmem_slot));
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(slot) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 0) {
        for (int s = 0; s < KNN_UMMA_STAGES; ++s) {
            mbar_init(PFULL + 8 * s, 1);     // the producer's arrive + the copy's bytes
            mbar_init(PEMPTY + 8 * s, 128);  // every expander thread
        }
        for (int j = 0; j < KNN_UMMA_BSTAGES; ++j) {
            mbar_init(BFULL + 8 * j, 128);   // every expander thread
            mbar_init(BEMPTY + 8 * j, 1);    // MMA commit
        }
        for (int k = 0; k < 2; ++k) {
            mbar_init(AFULL + 8 * k, 1);     // MMA commit
            mbar_init(AEMPTY + 8 * k, KNN_UMMA_THREADS); // every readout thread
        }
        mbar_init(AREADY, KNN_UMMA_THREADS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;

    const int n1 = t.n1;
    const long long n_units = t.n_units, groups = (n1 + KNN_UMMA_THREADS - 1) / KNN_UMMA_THREADS;
    const long long total = groups * n_units, ctas = gridDim.x;
    const long long x0 = static_cast<long long>(blockIdx.x) * total / ctas, x1 = (static_cast<long long>(blockIdx.x) + 1) * total / ctas;
    const int g0 = static_cast<int>(x0 / n_units);
    const int u0 = static_cast<int>(x0 - static_cast<long long>(g0) * n_units); // unit of the share's first item
    bool ok = true; // false after a wait timed out: this thread waits no more
#ifdef PLM_UMMA_STAMPS
    const long long t_start = clock64();
    long long waited = 0, units_done = 0;
#endif
    auto wait = [&](uint32_t bar, uint32_t parity) {
#ifdef PLM_UMMA_STAMPS
        const long long w0 = clock64();
#endif
        if (ok && !mbar_wait(bar, parity, spin_limit)) {
            ok = false;
            atomicExch(err, 1);
        }
#ifdef PLM_UMMA_STAMPS
        waited += clock64() - w0;
#endif
    };

    if (warp == 12) { // producer: packed units -> ring
        if (lane == 0) {
            int s = 0, u = u0;
            uint32_t ph = 0;
            for (long long x = x0; x < x1; ++x) {
                const int2 un = __ldg(t.units + u);
                const PairsJob &jb = t.jobs[un.x];
                const uint32_t bytes = static_cast<uint32_t>(min(KNN_UMMA_ROWS, jb.n2 - un.y)) * 32;
                wait(PEMPTY + 8 * s, ph ^ 1);
                mbar_arrive_tx(PFULL + 8 * s, bytes);
                bulk_copy_g2s(sRing + s * (KNN_UMMA_ROWS * 32), t.arena + 2 * (jb.train_off + un.y), bytes, PFULL + 8 * s);
                if (++s == KNN_UMMA_STAGES) { s = 0; ph ^= 1; }
                if (++u == n_units) u = 0;
#ifdef PLM_UMMA_STAMPS
                ++units_done;
#endif
            }
        }
    } else if (warp >= 8 && warp < 12) { // expanders: packed stage -> 0/1 bytes in a B tile (rows past the unit: stale, masked later)
        const int r = tid - KNN_UMMA_THREADS;
        int s = 0, j = 0;
        uint32_t ph = 0, bph = 0;
        for (long long x = x0; x < x1; ++x) {
            wait(PFULL + 8 * s, ph);
            const uint4 lo = ring[s * (2 * KNN_UMMA_ROWS) + 2 * r], hi = ring[s * (2 * KNN_UMMA_ROWS) + 2 * r + 1];
            mbar_arrive(PEMPTY + 8 * s);
            if (++s == KNN_UMMA_STAGES) { s = 0; ph ^= 1; }
            wait(BEMPTY + 8 * j, bph ^ 1);
            expand_half<false>(tileB + j * KNN_UMMA_TILE_BYTES, r, 0, lo);
            expand_half<false>(tileB + j * KNN_UMMA_TILE_BYTES, r, 1, hi);
            fence_proxy_async_smem(); // generic-proxy stores -> visible to the MMA (async proxy)
            mbar_arrive(BFULL + 8 * j);
            if (++j == KNN_UMMA_BSTAGES) { j = 0; bph ^= 1; }
#ifdef PLM_UMMA_STAMPS
            ++units_done;
#endif
        }
    } else if (warp == 13) { // MMA issuer: 2 M-tiles x 8 K-steps of 32 per unit into accumulator buffer unit & 1
        if (lane == 0) {
            int j = 0, u = u0;
            uint32_t bph = 0, c = 0, seg = 0;
            for (long long x = x0; x < x1; ++x, ++c) {
                if (x == x0 || u == 0) wait(AREADY, seg++ & 1u); // a new query group: its A is written
                const uint32_t k = c & 1u;
                wait(BFULL + 8 * j, bph);
                wait(AEMPTY + 8 * k, ((c >> 1) & 1u) ^ 1u);
                tc_fence_after();
#pragma unroll
                for (int m = 0; m < 2; ++m)
#pragma unroll
                    for (int st = 0; st < 8; ++st) {
                        const uint32_t koff = static_cast<uint32_t>((st >> 2) * (KNN_UMMA_TILE_BYTES / 2) + (st & 3) * 32);
                        umma_i8(tmem + k * 256 + static_cast<uint32_t>(m * 128), umma_desc_sw128(sA + m * KNN_UMMA_TILE_BYTES + koff),
                                umma_desc_sw128(sB + j * KNN_UMMA_TILE_BYTES + koff), KNN_UMMA_IDESC, st > 0 ? 1u : 0u);
                    }
                umma_commit(BEMPTY + 8 * j);
                umma_commit(AFULL + 8 * k);
                if (++j == KNN_UMMA_BSTAGES) { j = 0; bph ^= 1; }
                if (++u == n_units) u = 0;
#ifdef PLM_UMMA_STAMPS
                ++units_done;
#endif
            }
        }
    } else { // readout: thread = query of the group
        // this thread's accumulator lane: M-tile warp >> 2 at columns (warp >> 2) * 128, lanes 32 (warp & 3) ..
        const uint32_t tlane = tmem + (static_cast<uint32_t>(32 * (warp & 3)) << 16) + static_cast<uint32_t>((warp >> 2) * 128);
        uint32_t c = 0;
        int g = g0, u = u0;
        for (long long x = x0; x < x1; ++g, u = 0) {
            const int n = static_cast<int>(min(n_units - u, x1 - x)); // units of group g in this share
            x += n;
            // queries of the group -> A (+-1 bytes), |q| per thread.  The previous group's last accumulator wait
            // covered every MMA that read the old A.
            const int qi = g * KNN_UMMA_THREADS + tid;
            const bool valid = qi < n1;
            uint4 qlo = make_uint4(0, 0, 0, 0), qhi = qlo;
            if (valid) {
                qlo = __ldg(t.q + 2 * static_cast<long long>(qi));
                qhi = __ldg(t.q + 2 * static_cast<long long>(qi) + 1);
            }
            const int qn = __popc(qlo.x) + __popc(qlo.y) + __popc(qlo.z) + __popc(qlo.w) + __popc(qhi.x) + __popc(qhi.y) +
                           __popc(qhi.z) + __popc(qhi.w);
            uint8_t *a_tile = tileA + (tid >> 7) * KNN_UMMA_TILE_BYTES;
            if (valid) {
                expand_half<true>(a_tile, tid & 127, 0, qlo);
                expand_half<true>(a_tile, tid & 127, 1, qhi);
            } else { // zero rows: dot = 0; the lane never inserts (thr = 0 below), its column key is all ones
#pragma unroll
                for (int q = 0; q < 16; ++q)
                    *reinterpret_cast<uint4 *>(a_tile + (q >> 3) * (KNN_UMMA_TILE_BYTES / 2) + (tid & 127) * 128 + ((q & 7) << 4)) = make_uint4(0, 0, 0, 0);
            }
            fence_proxy_async_smem();
            mbar_arrive(AREADY);
            // direction-21 key of this row: (|q| + v) << 8 | row in the group = v * 256 + base21 (v = 0 on padding rows)
            const uint32_t base21 = valid ? (static_cast<uint32_t>(qn) << 8) | static_cast<uint32_t>(tid) : 0xFFFFFFFFu;

            unsigned long long B0 = KEY64_ABSENT, B1 = KEY64_ABSENT;
            int thr = valid ? 1023 : 0; // a distance must be < thr to enter the top-2 (> 256: none yet)
            int2 un = __ldg(t.units + u);
            for (int i = 0; i < n; ++i, ++c) {
                const uint32_t k = c & 1u;
                const PairsJob &jb = t.jobs[un.x];
                const int rows = min(KNN_UMMA_ROWS, jb.n2 - un.y);
                wait(AFULL + 8 * k, (c >> 1) & 1u);
                tc_fence_after();
                // two halves of 64 columns; the buffer is released for unit c + 2 as soon as the second half is in registers
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    int v[2][32];
                    tmem_ld32(tlane + k * 256 + static_cast<uint32_t>(64 * half), v[0]);
                    tmem_ld32(tlane + k * 256 + static_cast<uint32_t>(64 * half + 32), v[1]);
                    tmem_wait_ld(v[0]);
                    tmem_wait_ld(v[1]);
                    if (half == 1) {
                        tc_fence_before();
                        mbar_arrive(AEMPTY + 8 * k);
                    }
                    if (BOTH) {
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
                            colbuf[(k * 8 + warp) * KNN_UMMA_ROWS + 64 * half + 32 * q + lane] = make_uint2(r1, r2);
                        }
                    }
                    if (rows < KNN_UMMA_ROWS) {
#pragma unroll
                        for (int q = 0; q < 2; ++q)
#pragma unroll
                            for (int jj = 0; jj < 32; ++jj)
                                if (64 * half + 32 * q + jj >= rows) v[q][jj] = 0x3FFFFFFF; // rows past the unit: never below any bound
                    }
#pragma unroll
                    for (int q = 0; q < 2; ++q)
#pragma unroll
                        for (int h = 0; h < 32; h += KNN_UMMA_BLOCK) {
                            int m = v[q][h];
#pragma unroll
                            for (int jj = 1; jj + 1 < KNN_UMMA_BLOCK; jj += 2) m = __vimin3_s32(m, v[q][h + jj], v[q][h + jj + 1]);
                            m = min(m, v[q][h + KNN_UMMA_BLOCK - 1]);
                            if (qn + m < thr) {
#pragma unroll
                                for (int jj = 0; jj < KNN_UMMA_BLOCK; ++jj) {
                                    const int col = 64 * half + 32 * q + h + jj;
                                    if (col < rows) top2_insert(B0, B1, make_key64(static_cast<uint32_t>(qn + v[q][h + jj]), static_cast<uint32_t>(un.y + col)));
                                }
                                thr = (B1 == KEY64_ABSENT) ? 1023 : static_cast<int>(B1 >> 32);
                            }
                        }
                }
                if (BOTH) { // column tid of the unit: the two smallest of the 8 warps' pairs -> part21[g][row]
                    readout_bar_sync();
                    if (tid < rows) {
                        uint32_t b0 = 0xFFFFFFFFu, b1 = 0xFFFFFFFFu;
#pragma unroll
                        for (int w = 0; w < 8; ++w) {
                            const uint2 p = colbuf[(k * 8 + w) * KNN_UMMA_ROWS + tid];
                            top2_insert(b0, b1, p.x);
                            top2_insert(b0, b1, p.y);
                        }
                        const uint32_t qb = static_cast<uint32_t>(g) * KNN_UMMA_THREADS;
                        const unsigned long long k0 = b0 == 0xFFFFFFFFu ? KEY64_ABSENT : make_key64(b0 >> 8, qb + (b0 & 255u));
                        const unsigned long long k1 = b1 == 0xFFFFFFFFu ? KEY64_ABSENT : make_key64(b1 >> 8, qb + (b1 & 255u));
                        jb.part21[static_cast<size_t>(g) * jb.n2 + un.y + tid] = make_ulonglong2(k0, k1);
                    }
                }
                // end of a piece (the next unit is another job's, or the share leaves the group): direction-12 partials
                const int job = un.x;
                const bool last_unit = u + i + 1 == n_units;
                if (!last_unit) un = __ldg(t.units + u + i + 1);
                if (i + 1 == n || last_unit || un.x != job) {
                    if (valid) {
                        const int slot = static_cast<int>(blockIdx.x - umma_cta_of(static_cast<long long>(g) * n_units + jb.unit0, total, ctas));
                        jb.part12[static_cast<size_t>(slot) * n1 + qi] = make_ulonglong2(B0, B1);
                        if (u + i + 1 == jb.unit0 + jb.n_units) // the last piece of (group, job)
                            for (int p = slot + 1; p < jb.n_slots12; ++p) jb.part12[static_cast<size_t>(p) * n1 + qi] = make_ulonglong2(KEY64_ABSENT, KEY64_ABSENT);
                    }
                    B0 = B1 = KEY64_ABSENT;
                    thr = valid ? 1023 : 0;
                }
#ifdef PLM_UMMA_STAMPS
                ++units_done;
#endif
            }
        }
    }
#ifdef PLM_UMMA_STAMPS
    if ((tid == 0 || tid == KNN_UMMA_THREADS || tid == 384 || tid == 416) && blockIdx.x < KNN_UMMA_STAMP_CTAS) {
        const int role = tid == 0 ? 0 : tid == KNN_UMMA_THREADS ? 1 : tid == 384 ? 2 : 3;
        g_umma_stamps[blockIdx.x][role][0] = clock64() - t_start;
        g_umma_stamps[blockIdx.x][role][1] = waited;
        g_umma_stamps[blockIdx.x][role][2] = units_done;
    }
#endif
    tc_fence_before();
    __syncthreads(); // every MMA was waited for by the readout (or a wait timed out and the results are discarded)
    tc_fence_after();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

} // namespace plm
