// Brute-force Hamming top-2 on the tensor cores (knn2 variant 7, long scans only).
//
// Over K = 256 bits the Hamming distance is an exact integer dot product.  With the query as +-1 bytes and the train
// row as 0/1 bytes:
//     q'_i = 1 - 2 q_i,  r_i in {0, 1}   =>   dot(q', r) = |r| - 2 |q & r|   =>   d(q, r) = |q| + dot(q', r)
// so one `tcgen05.mma.cta_group::1.kind::i8` with s32 accumulation per 128 x 128 x 32 block gives every distance
// exactly, and keys and tie-breaks are those of knn2_slice_kernel bit for bit.
//
// One CTA per SM, the whole 512-column tensor memory.  A CTA owns a contiguous range of the (query group, 128-row
// unit) work list, so every SM gets the same number of units whatever the number of query groups; the range is cut
// into segments, one per query group it touches, each scanned in increasing row order.  The CTA is warp-specialised,
// its roles meet only on mbarriers (full/empty pairs, every wait bounded), so loading, expansion, MMA and readout of
// different units overlap:
//   * producer (warp 12, one thread): packed train units (4 KB, rows * 32 B for a short last unit) -> a
//     KNN_UMMA_STAGES-deep ring with cp.async.bulk, completion counted in bytes on the stage's full barrier;
//   * expanders (warps 8-11, thread = train row): packed stage -> 0/1 bytes in one of KNN_UMMA_BSTAGES B tiles,
//     fence.proxy.async, arrive on the B tile's full barrier;
//   * MMA issuer (warp 13, one thread): per unit 2 M-tiles x 8 K-steps of tcgen05.mma into accumulator buffer
//     unit & 1, committed to the B tile's empty barrier and to the accumulator's full barrier;
//   * readout (warps 0-7, thread t = query t of the group = TMEM lane t & 127 of M-tile t >> 7): per segment the
//     256 queries are expanded once to +-1 bytes (A = 2 M-tiles x 128 rows x 256 B, resident) and released to the
//     MMA issuer on the A barrier; per unit all 128 accumulator columns are loaded, the buffer is released, and the
//     blocked top-2 test of variants 2/3 runs on the registers (16 columns at a time, exact because columns are rows
//     in increasing order).
// A segment switch drains the pipeline once: the readout finishes the segment's last unit (so no MMA reads A any
// more), writes its partials, rewrites A and arrives on the A barrier.
// Operands are K-major with the 128-byte swizzle: a 256-byte row is two swizzle atoms along K, each operand tile is
// [K half][rows][128 B] with 16-byte chunk c of row r stored at chunk c ^ (r & 7).
// part[p][query] holds the (best, second) keys of segment p of the query's group; slots no CTA scanned are written
// absent, so knn2_merge_kernel reads n_workers slots per query as for the integer kernels.
#pragma once
#include "plm_common.cuh"
#include "plm_knn2.cuh"

namespace plm {

constexpr int KNN_UMMA_THREADS = 256;                      // queries per group (two M = 128 tiles) = readout threads
constexpr int KNN_UMMA_CTA_THREADS = KNN_UMMA_THREADS + 128 + 64; // + 4 expander warps + producer warp + MMA warp
constexpr int KNN_UMMA_ROWS = 128;                         // train rows per unit (MMA N)
constexpr int KNN_UMMA_STAGES = 8;                         // packed-unit ring depth
constexpr int KNN_UMMA_BSTAGES = 3;                        // expanded B tiles
constexpr int KNN_UMMA_TILE_BYTES = 128 * 256;             // one 128-row operand tile of 256 int8 columns
constexpr int KNN_UMMA_SMEM = 2 * KNN_UMMA_TILE_BYTES      // A (queries)
                              + KNN_UMMA_BSTAGES * KNN_UMMA_TILE_BYTES // B ring
                              + KNN_UMMA_STAGES * KNN_UMMA_ROWS * 32   // packed ring
                              + 1024;                      // alignment of the swizzled tiles
// rate kernel: A, B of up to 256 rows, and a 32 KB store target for the concurrent-store case
constexpr int KNN_UMMA_RATE_SMEM = 4 * KNN_UMMA_TILE_BYTES + 1024;
constexpr int KNN_UMMA_BLOCK = 16;                         // columns per blocked threshold test

// Instruction descriptor of kind::i8: D s32 (bits 4-5 = 2), A and B signed 8-bit (bits 7-9, 10-12 = 1), both K-major,
// N >> 3 at bit 17, M >> 4 at bit 24.
constexpr uint32_t KNN_UMMA_IDESC = (2u << 4) | (1u << 7) | (1u << 10) | (uint32_t(KNN_UMMA_ROWS >> 3) << 17) | (uint32_t(128 >> 4) << 24);

// Shared-memory matrix descriptor: K-major, 128-byte swizzle (layout 2 at bit 61), stride between 8-row groups
// 1024 B, descriptor version 1 (bit 46).  The leading offset is unused for swizzled K-major operands.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    return static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (static_cast<uint64_t>(1024 >> 4) << 32) |
           (1ull << 46) | (2ull << 61);
}

__device__ __forceinline__ void umma_i8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate));
}
__device__ __forceinline__ void umma_commit(uint32_t mbar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mbar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
}
// Bounded wait for the phase with the given parity; false after `limit` clock64 ticks.
__device__ __forceinline__ bool mbar_wait(uint32_t mbar, uint32_t parity, long long limit) {
    const long long t0 = clock64();
    for (;;) {
        uint32_t done;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(mbar), "r"(parity) : "memory");
        if (done) return true;
        if (clock64() - t0 > limit) return false;
    }
}

__device__ __forceinline__ void mbar_arrive(uint32_t mbar) {
    asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(mbar) : "memory");
}
// arrive and expect `bytes` more of asynchronous copies on this phase
__device__ __forceinline__ void mbar_arrive_tx(uint32_t mbar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.release.cta.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
// contiguous global -> shared copy on the async proxy, completion counted in bytes on mbar
__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(mbar) : "memory");
}

// 32 consecutive accumulator columns of this warp's 32 lanes (one column per register); the registers hold the values
// only after tmem_wait_ld, which takes them as operands so that no use is scheduled before it.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, int (&v)[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld(int (&v)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                   "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]),
                   "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]),
                   "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
                 :: "memory");
}

// Bits 4k .. 4k + 3 of w as four 0/1 bytes (byte j = bit 4k + j).
__device__ __forceinline__ uint32_t nibble_bytes(uint32_t w, int k) { return (((w >> (4 * k)) & 0xFu) * 0x00204081u) & 0x01010101u; }

// One 128-bit half of a descriptor -> one 128-byte swizzled row of an operand tile: bit b becomes byte b, as 0/1
// (train rows) or as +1 / -1 (queries: 0x01 | 0xFE * bit).
template <bool PLUS_MINUS>
__device__ __forceinline__ void expand_half(uint8_t *tile, int row, int half, const uint4 &h) {
    const uint32_t w[4] = {h.x, h.y, h.z, h.w};
    uint8_t *dst = tile + half * (KNN_UMMA_TILE_BYTES / 2) + row * 128;
#pragma unroll
    for (int c = 0; c < 8; ++c) { // 16-byte chunk c = bits 16c .. 16c + 15
        const uint32_t src = w[c >> 1] >> ((c & 1) * 16);
        uint32_t o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            o[k] = nibble_bytes(src, k);
            if (PLUS_MINUS) o[k] = (o[k] * 0xFEu) | 0x01010101u;
        }
        *reinterpret_cast<uint4 *>(dst + ((c ^ (row & 7)) << 4)) = make_uint4(o[0], o[1], o[2], o[3]);
    }
}

// CTA that scans item x of the (group, unit) list of `total` items over `ctas` CTAs (CTA c owns
// [c * total / ctas, (c + 1) * total / ctas)).
__host__ __device__ __forceinline__ long long umma_cta_of(long long x, long long total, long long ctas) {
    return ((x + 1) * ctas - 1) / total;
}

#ifdef PLM_UMMA_STAMPS
// Debug builds only (PLM_BUILD_DEFINES=-DPLM_UMMA_STAMPS): per CTA and role (0 readout, 1 expander, 2 producer, 3 MMA
// issuer), one thread of the role stamps its SM cycles from kernel start to the end of its loop, the cycles it spent in
// mbarrier waits, and the units it handled; plm_debug_umma_stamps copies them out.
constexpr int KNN_UMMA_STAMP_CTAS = 160;
__device__ long long g_umma_stamps[KNN_UMMA_STAMP_CTAS][4][3];
#endif

__global__ void __launch_bounds__(KNN_UMMA_CTA_THREADS, 1) knn2_umma_kernel(const KnnTask t, int32_t *err, long long spin_limit) {
    extern __shared__ uint8_t smem_raw[];
    // packed full / empty [STAGES], B full / empty [BSTAGES], accumulator full / empty [2], A ready
    __shared__ __align__(8) unsigned long long mbar[2 * KNN_UMMA_STAGES + 2 * KNN_UMMA_BSTAGES + 5];
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint8_t *smem = smem_raw + ((1024 - (static_cast<uint32_t>(__cvta_generic_to_shared(smem_raw)) & 1023)) & 1023); // 1024-aligned
    uint8_t *tileA = smem;                                  // 2 M-tiles
    uint8_t *tileB = smem + 2 * KNN_UMMA_TILE_BYTES;        // BSTAGES unit tiles
    const uint4 *ring = reinterpret_cast<const uint4 *>(smem + (2 + KNN_UMMA_BSTAGES) * KNN_UMMA_TILE_BYTES);
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

    const int n1 = t.n1, nw = t.n_workers;
    const long long n_units = t.n_units, groups = (n1 + KNN_UMMA_THREADS - 1) / KNN_UMMA_THREADS;
    const long long total = groups * n_units, ctas = gridDim.x;
    const long long x0 = static_cast<long long>(blockIdx.x) * total / ctas, x1 = (static_cast<long long>(blockIdx.x) + 1) * total / ctas;
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
    // every role walks the same segments: query group g, first unit u0, n units
    auto segment = [&](long long x, int &g, long long &u0, int &n) {
        g = static_cast<int>(x / n_units);
        u0 = x - static_cast<long long>(g) * n_units;
        n = static_cast<int>(min(x1, static_cast<long long>(g + 1) * n_units) - x);
    };
    auto rows_of = [&](long long u) { return static_cast<int>(min(static_cast<long long>(KNN_UMMA_ROWS), t.n2 - u * KNN_UMMA_ROWS)); };

    if (warp == 12) { // producer: packed units -> ring
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            for (long long x = x0; x < x1;) {
                int g, n;
                long long u0;
                segment(x, g, u0, n);
                x += n;
                for (int i = 0; i < n; ++i) {
                    wait(PEMPTY + 8 * s, ph ^ 1);
                    const uint32_t bytes = static_cast<uint32_t>(rows_of(u0 + i)) * 32;
                    mbar_arrive_tx(PFULL + 8 * s, bytes);
                    bulk_copy_g2s(sRing + s * (KNN_UMMA_ROWS * 32), t.db + 2 * ((u0 + i) * KNN_UMMA_ROWS), bytes, PFULL + 8 * s);
                    if (++s == KNN_UMMA_STAGES) { s = 0; ph ^= 1; }
#ifdef PLM_UMMA_STAMPS
                    ++units_done;
#endif
                }
            }
        }
    } else if (warp >= 8 && warp < 12) { // expanders: packed stage -> 0/1 bytes in a B tile (rows past n2: stale bits, masked later)
        const int r = tid - KNN_UMMA_THREADS;
        int s = 0, j = 0;
        uint32_t ph = 0, bph = 0;
        for (long long x = x0; x < x1;) {
            int g, n;
            long long u0;
            segment(x, g, u0, n);
            x += n;
            for (int i = 0; i < n; ++i) {
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
        }
    } else if (warp == 13) { // MMA issuer: 2 M-tiles x 8 K-steps of 32 per unit into accumulator buffer unit & 1
        if (lane == 0) {
            int j = 0;
            uint32_t bph = 0, c = 0, seg = 0;
            for (long long x = x0; x < x1;) {
                int g, n;
                long long u0;
                segment(x, g, u0, n);
                x += n;
                wait(AREADY, seg++ & 1u);
                for (int i = 0; i < n; ++i, ++c) {
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
#ifdef PLM_UMMA_STAMPS
                    ++units_done;
#endif
                }
            }
        }
    } else { // readout: thread = query of the group
        // this thread's accumulator lane: M-tile warp >> 2 at columns (warp >> 2) * 128, lanes 32 (warp & 3) ..
        const uint32_t tlane = tmem + (static_cast<uint32_t>(32 * (warp & 3)) << 16) + static_cast<uint32_t>((warp >> 2) * 128);
        const uint32_t idx_base = static_cast<uint32_t>(t.idx_base); // idx_base + n2 <= 2^32 (checked by the host)
        uint32_t c = 0;
        for (long long x = x0; x < x1;) {
            int g, n;
            long long u0;
            segment(x, g, u0, n);
            const int slot = static_cast<int>(blockIdx.x - umma_cta_of(static_cast<long long>(g) * n_units, total, ctas));
            const bool last_of_group = x + n == static_cast<long long>(g + 1) * n_units;
            x += n;

            // queries of the group -> A (+-1 bytes), |q| per thread.  The previous segment's last accumulator wait
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
            } else { // zero rows: dot = 0; the lane never inserts (thr = 0 below)
#pragma unroll
                for (int q = 0; q < 16; ++q)
                    *reinterpret_cast<uint4 *>(a_tile + (q >> 3) * (KNN_UMMA_TILE_BYTES / 2) + (tid & 127) * 128 + ((q & 7) << 4)) = make_uint4(0, 0, 0, 0);
            }
            fence_proxy_async_smem();
            mbar_arrive(AREADY);

            unsigned long long B0 = KEY64_ABSENT, B1 = KEY64_ABSENT;
            int thr = valid ? 1023 : 0, gcap = 1023; // a distance must be < thr to enter the top-2 (> 256: none yet)
            uint32_t *gthr = (t.gthr && valid) ? t.gthr + qi : nullptr;
            auto lower_thr = [&]() {
                const int own = (B1 == KEY64_ABSENT) ? 1023 : static_cast<int>(B1 >> 32);
                if (gthr && own < 1023) atomicMin(gthr, static_cast<uint32_t>(own));
                thr = min(own, gcap);
            };
            for (int i = 0; i < n; ++i, ++c) {
                const uint32_t k = c & 1u;
                wait(AFULL + 8 * k, (c >> 1) & 1u);
                tc_fence_after();
                if (gthr) { // once per unit: the bound the other CTAs have reached (rows AT the bound stay in)
                    const uint32_t gv = *reinterpret_cast<volatile uint32_t *>(gthr);
                    gcap = static_cast<int>(min(gv, 1022u)) + 1;
                    thr = min(thr, gcap);
                }
                const int rows = rows_of(u0 + i);
                const uint32_t gbase = idx_base + static_cast<uint32_t>((u0 + i) * KNN_UMMA_ROWS);
                // two halves of 64 columns (128 live values would spill); the buffer is released for unit c + 2 as soon
                // as the second half is in registers
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
                    if (rows < KNN_UMMA_ROWS) {
#pragma unroll
                        for (int q = 0; q < 2; ++q)
#pragma unroll
                            for (int jj = 0; jj < 32; ++jj)
                                if (64 * half + 32 * q + jj >= rows) v[q][jj] = 0x3FFFFFFF; // rows past n2: never below any bound
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
                                    if (col < rows) top2_insert(B0, B1, make_key64(static_cast<uint32_t>(qn + v[q][h + jj]), gbase + col));
                                }
                                lower_thr();
                            }
                        }
                }
#ifdef PLM_UMMA_STAMPS
                ++units_done;
#endif
            }
            if (valid) {
                t.part[static_cast<size_t>(slot) * n1 + qi] = make_ulonglong2(B0, B1);
                if (last_of_group)
                    for (int p = slot + 1; p < nw; ++p) t.part[static_cast<size_t>(p) * n1 + qi] = make_ulonglong2(KEY64_ABSENT, KEY64_ABSENT);
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

// Back-to-back 128 x N x 32 int8 MMAs on zeroed operands (one CTA per SM): the INT8 tensor-core rate of this card at
// N = 256 (the peak) and at N = 128 (the shape knn2_umma_kernel issues).  With STS, warps 1-3 keep storing 16-byte
// chunks to a separate 32 KB tile while the MMAs run, as the expansion of train units does.  Shared memory:
// KNN_UMMA_RATE_SMEM.
template <int N, bool STS>
__global__ void __launch_bounds__(128, 1) mma_i8_rate_kernel(int iters, int32_t *err, long long spin_limit) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) unsigned long long bar;
    __shared__ uint32_t tmem_slot;
    uint8_t *smem = smem_raw + ((1024 - (static_cast<uint32_t>(__cvta_generic_to_shared(smem_raw)) & 1023)) & 1023); // 1024-aligned
    for (int i = threadIdx.x; i < 3 * KNN_UMMA_TILE_BYTES / 16; i += blockDim.x) reinterpret_cast<uint4 *>(smem)[i] = make_uint4(0, 0, 0, 0);
    const uint32_t sA = static_cast<uint32_t>(__cvta_generic_to_shared(smem)), sB = sA + KNN_UMMA_TILE_BYTES;
    const uint32_t sbar = static_cast<uint32_t>(__cvta_generic_to_shared(&bar));
    if (threadIdx.x < 32) {
        const uint32_t slot = static_cast<uint32_t>(__cvta_generic_to_shared(&tmem_slot));
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(slot) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (threadIdx.x == 0) {
        mbar_init(sbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    // B is read as N rows from the zeroed tiles behind A
    constexpr uint32_t idesc = (KNN_UMMA_IDESC & ~(0x3Fu << 17)) | (uint32_t(N >> 3) << 17);
    if (threadIdx.x == 0) {
        for (int it = 0; it < iters; ++it)
#pragma unroll
            for (int s = 0; s < 8; ++s) {
                const uint32_t koff = static_cast<uint32_t>((s >> 2) * (KNN_UMMA_TILE_BYTES / 2) + (s & 3) * 32);
                umma_i8(tmem, umma_desc_sw128(sA + koff), umma_desc_sw128(sB + koff), idesc, (it | s) ? 1u : 0u);
            }
        umma_commit(sbar);
    }
    __syncwarp();
    if (threadIdx.x < 32) {
        if (!mbar_wait(sbar, 0, spin_limit) && threadIdx.x == 0) atomicExch(err, 1);
    } else if (STS) {
        uint4 *dst = reinterpret_cast<uint4 *>(smem + 3 * KNN_UMMA_TILE_BYTES);
        const uint4 val = make_uint4(threadIdx.x, 0, 0, 0);
        const long long t0 = clock64();
        for (uint32_t done = 0; !done;) {
#pragma unroll 4
            for (int i = threadIdx.x - 32; i < KNN_UMMA_TILE_BYTES / 16; i += 96) dst[i] = val;
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                         : "=r"(done) : "r"(sbar) : "memory");
            if (clock64() - t0 > spin_limit) break;
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (threadIdx.x < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem) : "memory");
}

} // namespace plm
