// Brute-force Hamming top-2 on the tensor cores: the warp-specialised tcgen05 pipeline (umma_pipeline) and the
// long-scan kernel built on it (knn2 variant 7, knn2_umma_kernel).  knn2_umma_pairs_kernel (plm_knn2_umma_pairs.cuh)
// is the other kernel on the same pipeline.
//
// Over K = 256 bits the Hamming distance is an exact integer dot product.  With the query as +-1 bytes and the train
// row as 0/1 bytes:
//     q'_i = 1 - 2 q_i,  r_i in {0, 1}   =>   dot(q', r) = |r| - 2 |q & r|   =>   d(q, r) = |q| + dot(q', r)
// so one `tcgen05.mma.cta_group::1.kind::i8` with s32 accumulation per 128 x 128 x 32 block gives every distance
// exactly, and keys and tie-breaks are those of knn2_slice_kernel bit for bit.
//
// One CTA per SM, the whole 512-column tensor memory.  A CTA owns a contiguous range of the (query group, 128-row
// unit) work list, so every SM gets the same number of units whatever the number of query groups; the range is cut
// into segments, one per query group it touches, each scanned in increasing unit order.  The CTA is warp-specialised,
// its roles meet only on mbarriers (full/empty pairs, every wait bounded), so loading, expansion, MMA and readout of
// different units overlap:
//   * producer (warp 12, one thread): packed train units (4 KB, rows * 32 B for a short unit) -> a
//     KNN_UMMA_STAGES-deep ring with cp.async.bulk, completion counted in bytes on the stage's full barrier;
//   * expanders (warps 8-11, thread = train row): packed stage -> 0/1 bytes in one of KNN_UMMA_BSTAGES B tiles,
//     fence.proxy.async, arrive on the B tile's full barrier and on the packed stage's empty barrier;
//   * MMA issuer (warp 13, one thread): per unit 2 M-tiles x 8 K-steps of tcgen05.mma into accumulator buffer
//     unit & 1, committed to the B tile's empty barrier and to the accumulator's full barrier;
//   * readout (warps 0-7, thread t = query t of the group = TMEM lane t & 127 of M-tile t >> 7): per segment the
//     256 queries are expanded once to +-1 bytes (A = 2 M-tiles x 128 rows x 256 B, resident) and released to the
//     MMA issuer on the A barrier; per unit all 128 accumulator columns are loaded, the buffer is released, and the
//     blocked top-2 test of variants 2/3 runs on the registers (16 columns at a time, exact because the columns of a
//     unit are rows in increasing order and the test is strict).  K1b loads the columns packed two per register and
//     runs the blocked test only on a unit whose minimum passes the bound (Scan::PACKED).
// A segment switch drains the pipeline once: the readout finishes the segment's last unit (so no MMA reads A any
// more), writes its partials, rewrites A and arrives on the A barrier.
// A stage is released only after its reads have completed: a packed stage after the expander has stored its values
// into the B tile and fenced the proxies (its next writer is the async proxy), a B tile by the MMA commit, an
// accumulator buffer after tcgen05.wait::ld, A at the segment's last accumulator wait.
// Operands are K-major with the 128-byte swizzle: a 256-byte row is two swizzle atoms along K, each operand tile is
// [K half][rows][128 B] with 16-byte chunk c of row r stored at chunk c ^ (r & 7).
//
// knn2_umma_kernel: unit u is train rows [128 u, 128 u + 128) of one task, keys carry idx_base + row, and the
// per-query second-best bound gthr is shared with the other CTAs.  part[p][query] holds the (best, second) keys of
// segment p of the query's group; slots no CTA scanned are written absent, so knn2_merge_kernel reads n_workers slots
// per query as for the integer kernels.
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
constexpr int KNN_UMMA_PIPE_BYTES = 2 * KNN_UMMA_TILE_BYTES // A (queries)
                                    + KNN_UMMA_BSTAGES * KNN_UMMA_TILE_BYTES // B ring
                                    + KNN_UMMA_STAGES * KNN_UMMA_ROWS * 32;  // packed ring
constexpr int KNN_UMMA_SMEM = KNN_UMMA_PIPE_BYTES + 1024;  // + alignment of the swizzled tiles
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
// __syncthreads ordered against the tensor-core operations (TMEM alloc, MMA, loads) on both sides of it
__device__ __forceinline__ void tc_syncthreads() { tc_fence_before(); __syncthreads(); tc_fence_after(); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Warp-wide: COLS columns of tensor memory (a power of two >= 32), their address to *slot; the CTA then gives up its
// allocation permit (it allocates once).
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t *slot) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(slot))), "n"(COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t tmem) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(COLS) : "memory");
}

__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
}
// after the last mbar_init: the initialised barriers are visible to the other threads and the async proxy
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
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
// 128 consecutive accumulator columns of this warp's 32 lanes, two per register (.pack::16b keeps the low 16 bits of
// each column: column 2i in bits 0-15 of v[i], column 2i + 1 in bits 16-31; .x64 counts the registers).  One
// instruction, so that no use of the first columns can be scheduled between two loads and serialise their round
// trips; the registers hold the values only after tmem_wait_ld.
__device__ __forceinline__ void tmem_ld128p(uint32_t taddr, uint32_t (&v)[64]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x64.pack::16b.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, "
                 "%13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32, %33, "
                 "%34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, %48, %49, %50, %51, %52, %53, %54, "
                 "%55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31]),
                   "=r"(v[32]), "=r"(v[33]), "=r"(v[34]), "=r"(v[35]), "=r"(v[36]), "=r"(v[37]), "=r"(v[38]), "=r"(v[39]),
                   "=r"(v[40]), "=r"(v[41]), "=r"(v[42]), "=r"(v[43]), "=r"(v[44]), "=r"(v[45]), "=r"(v[46]), "=r"(v[47]),
                   "=r"(v[48]), "=r"(v[49]), "=r"(v[50]), "=r"(v[51]), "=r"(v[52]), "=r"(v[53]), "=r"(v[54]), "=r"(v[55]),
                   "=r"(v[56]), "=r"(v[57]), "=r"(v[58]), "=r"(v[59]), "=r"(v[60]), "=r"(v[61]), "=r"(v[62]), "=r"(v[63])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld(uint32_t (&v)[64]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                   "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]),
                   "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]),
                   "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31]),
                   "+r"(v[32]), "+r"(v[33]), "+r"(v[34]), "+r"(v[35]), "+r"(v[36]), "+r"(v[37]), "+r"(v[38]), "+r"(v[39]),
                   "+r"(v[40]), "+r"(v[41]), "+r"(v[42]), "+r"(v[43]), "+r"(v[44]), "+r"(v[45]), "+r"(v[46]), "+r"(v[47]),
                   "+r"(v[48]), "+r"(v[49]), "+r"(v[50]), "+r"(v[51]), "+r"(v[52]), "+r"(v[53]), "+r"(v[54]), "+r"(v[55]),
                   "+r"(v[56]), "+r"(v[57]), "+r"(v[58]), "+r"(v[59]), "+r"(v[60]), "+r"(v[61]), "+r"(v[62]), "+r"(v[63])
                 :: "memory");
}
// the two signed 16-bit halves of a packed register
__device__ __forceinline__ int s16_lo(uint32_t x) { return static_cast<int16_t>(x & 0xFFFFu); }
__device__ __forceinline__ int s16_hi(uint32_t x) { return static_cast<int>(x) >> 16; }
// Signed 16x2 min of v[0 .. N - 1] as a tree of three-input mins: depth log3 N, so each level's mins issue back to back.
template <int N>
__device__ __forceinline__ uint32_t vmin_s16x2(const uint32_t *v) {
    if constexpr (N == 1) {
        return v[0];
    } else if constexpr (N == 2) {
        return __vmins2(v[0], v[1]);
    } else {
        constexpr int A = (N + 2) / 3, B = (N - A + 1) / 2;
        return __vimin3_s16x2(vmin_s16x2<A>(v), vmin_s16x2<B>(v + A), vmin_s16x2<N - A - B>(v + A + B));
    }
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
// Number of CTAs the items [first, first + n) of that list are spread over (n >= 1): the partial slots they need.
__host__ __device__ __forceinline__ long long umma_ctas_spanned(long long first, long long n, long long total, long long ctas) {
    return umma_cta_of(first + n - 1, total, ctas) - umma_cta_of(first, total, ctas) + 1;
}
// This CTA's partial slot in a run of items that starts at item `first` of the list of n1 queries x n_units units: its
// index among the CTAs the run is spread over.
__device__ __forceinline__ int umma_slot(long long first, int n1, long long n_units) {
    const long long total = static_cast<long long>((n1 + KNN_UMMA_THREADS - 1) / KNN_UMMA_THREADS) * n_units;
    return static_cast<int>(blockIdx.x - umma_cta_of(first, total, gridDim.x));
}

// The kernel's dynamic shared memory, aligned to 1024 bytes for the swizzled tiles.
__device__ __forceinline__ uint8_t *umma_smem() {
    extern __shared__ uint8_t smem_raw[];
    return smem_raw + ((1024 - (static_cast<uint32_t>(__cvta_generic_to_shared(smem_raw)) & 1023)) & 1023);
}

#ifdef PLM_UMMA_STAMPS
// Debug builds only (PLM_BUILD_DEFINES=-DPLM_UMMA_STAMPS): per CTA and role (0 readout, 1 expander, 2 producer, 3 MMA
// issuer), one thread of the role stamps its SM cycles from kernel start to the end of its loop, the cycles it spent in
// mbarrier waits, and the units it handled; plm_debug_umma_stamps copies them out.
constexpr int KNN_UMMA_STAMP_CTAS = 160;
__device__ long long g_umma_stamps[KNN_UMMA_STAMP_CTAS][4][3];
#endif

// A segment as the readout sees it: units [u0, u0 + n) of query group g; this thread is query qi (valid: qi < n1), |q| = qn.
struct UmmaSeg {
    long long u0;
    int g, n, qi, qn;
    bool valid;
};
// Columns of one unit as the readout sees them: `rows` live columns, column j has key index key0 + j.
struct UmmaCols {
    int rows;
    uint32_t key0;
};

// The pipeline over this CTA's share of the (query group of 256 of the n1 `queries`, unit) list of n_units units per
// group; launched with KNN_UMMA_CTA_THREADS threads, one CTA per SM, shared memory from KNN_UMMA_PIPE_BYTES on is the
// Scan's.  The Scan supplies the unit source and the readout's rules (each call is inlined):
//   const uint4 *unit_src(long long u, int &rows)     producer: unit u's packed rows in global memory and their count
//   void begin_segment(const UmmaSeg &s)              readout, after A is written
//   UmmaCols begin_unit(const UmmaSeg &s, int i, int &thr)  unit s.u0 + i, its accumulators ready; may lower thr
//   int threshold(unsigned long long B1)              the insert bound after an insert into (B0, B1)
//   static constexpr bool PACKED                      the readout's form: true, all 128 columns as 16-bit halves in one
//                                                     load and one whole-unit test; false, two halves of 64 exact
//                                                     32-bit columns, each passed to `loaded` before the blocked test
//   void loaded(int (&v)[2][32], int half, uint32_t k)  (PACKED false) accumulator columns 64 half .. + 63 of buffer k, unmasked
//   void end_unit(const UmmaSeg &s, int i, uint32_t k, int rows, unsigned long long &B0, unsigned long long &B1, int &thr)
//   void end_segment(const UmmaSeg &s, unsigned long long B0, unsigned long long B1)
template <class Scan>
__device__ __forceinline__ void umma_pipeline(Scan &sc, const uint4 *queries, int n1, int n_units, int32_t *err, long long spin_limit) {
    // packed full / empty [STAGES], B full / empty [BSTAGES], accumulator full / empty [2], A ready
    __shared__ __align__(8) unsigned long long mbar[2 * KNN_UMMA_STAGES + 2 * KNN_UMMA_BSTAGES + 5];
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint8_t *smem = umma_smem();
    uint8_t *tileA = smem;                                  // 2 M-tiles
    uint8_t *tileB = smem + 2 * KNN_UMMA_TILE_BYTES;        // BSTAGES unit tiles
    const uint4 *ring = reinterpret_cast<const uint4 *>(smem + (2 + KNN_UMMA_BSTAGES) * KNN_UMMA_TILE_BYTES);
    const uint32_t sA = static_cast<uint32_t>(__cvta_generic_to_shared(tileA));
    const uint32_t sB = static_cast<uint32_t>(__cvta_generic_to_shared(tileB));
    const uint32_t sRing = static_cast<uint32_t>(__cvta_generic_to_shared(ring));
    const uint32_t PFULL = static_cast<uint32_t>(__cvta_generic_to_shared(mbar)), PEMPTY = PFULL + 8 * KNN_UMMA_STAGES;
    const uint32_t BFULL = PEMPTY + 8 * KNN_UMMA_STAGES, BEMPTY = BFULL + 8 * KNN_UMMA_BSTAGES;
    const uint32_t AFULL = BEMPTY + 8 * KNN_UMMA_BSTAGES, AEMPTY = AFULL + 16, AREADY = AEMPTY + 16;

    if (warp == 0) tmem_alloc<512>(&tmem_slot);
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
        mbar_init_fence();
    }
    tc_syncthreads();
    const uint32_t tmem = tmem_slot;

    const long long groups = (n1 + KNN_UMMA_THREADS - 1) / KNN_UMMA_THREADS;
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
                    int rows;
                    const uint4 *src = sc.unit_src(u0 + i, rows);
                    const uint32_t bytes = static_cast<uint32_t>(rows) * 32;
                    mbar_arrive_tx(PFULL + 8 * s, bytes);
                    bulk_copy_g2s(sRing + s * (KNN_UMMA_ROWS * 32), src, bytes, PFULL + 8 * s);
                    if (++s == KNN_UMMA_STAGES) { s = 0; ph ^= 1; }
#ifdef PLM_UMMA_STAMPS
                    ++units_done;
#endif
                }
            }
        }
    } else if (warp >= 8 && warp < 12) { // expanders: packed stage -> 0/1 bytes in a B tile (rows past the unit: stale bits, masked later)
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
                wait(BEMPTY + 8 * j, bph ^ 1);
                expand_half<false>(tileB + j * KNN_UMMA_TILE_BYTES, r, 0, lo);
                expand_half<false>(tileB + j * KNN_UMMA_TILE_BYTES, r, 1, hi);
                // One proxy fence orders this thread's generic-proxy accesses against the async proxy in both
                // directions: the B-tile stores before the MMA reads them, and the packed-stage loads (complete: their
                // values were just stored) before the producer's next cp.async.bulk writes that stage.  The mbarrier's
                // release/acquire alone orders generic accesses only, and an arrive issued right after the loads does
                // not wait for them: the stage could be refilled with unit c + KNN_UMMA_STAGES before they read it.
                fence_proxy_async_smem();
                mbar_arrive(BFULL + 8 * j);
                mbar_arrive(PEMPTY + 8 * s);
                if (++s == KNN_UMMA_STAGES) { s = 0; ph ^= 1; }
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
        uint32_t c = 0;
        for (long long x = x0; x < x1;) {
            int g, n;
            long long u0;
            segment(x, g, u0, n);
            x += n;

            // queries of the group -> A (+-1 bytes), |q| per thread.  The previous segment's last accumulator wait
            // covered every MMA that read the old A.
            const int qi = g * KNN_UMMA_THREADS + tid;
            const bool valid = qi < n1;
            uint4 qlo = make_uint4(0, 0, 0, 0), qhi = qlo;
            if (valid) {
                qlo = __ldg(queries + 2 * static_cast<long long>(qi));
                qhi = __ldg(queries + 2 * static_cast<long long>(qi) + 1);
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
            const UmmaSeg sg{u0, g, n, qi, qn, valid};
            sc.begin_segment(sg);

            unsigned long long B0 = KEY64_ABSENT, B1 = KEY64_ABSENT;
            int thr = valid ? 1023 : 0; // a distance must be < thr to enter the top-2 (> 256: none yet)
            for (int i = 0; i < n; ++i, ++c) {
                const uint32_t k = c & 1u;
                wait(AFULL + 8 * k, (c >> 1) & 1u);
                tc_fence_after();
                const UmmaCols u = sc.begin_unit(sg, i, thr);
                if constexpr (Scan::PACKED) {
                    // All 128 columns in one load of 64 registers, 16 bits per column (every value is a dot in
                    // [-256, 256]); the buffer is released for unit c + 2 before any test.  Every min is signed 16x2.
                    uint32_t p[KNN_UMMA_ROWS / 2];
                    tmem_ld128p(tlane + k * 256, p);
                    tmem_wait_ld(p);
                    tc_fence_before();
                    mbar_arrive(AEMPTY + 8 * k);
                    // One test for the whole unit; only a unit that can insert takes the blocked test, exact as in
                    // the unpacked form.  In a short unit the blocks that reach past u.rows take their minimum with
                    // those columns as 0x7FFF per 16-bit half (never below any bound), and inserts skip them by column.
                    const uint32_t um = vmin_s16x2<KNN_UMMA_ROWS / 2>(p);
                    if (qn + min(s16_lo(um), s16_hi(um)) < thr) {
#pragma unroll
                        for (int h = 0; h < KNN_UMMA_ROWS / 2; h += KNN_UMMA_BLOCK / 2) {
                            const uint32_t *b = p + h;
                            uint32_t bm = vmin_s16x2<KNN_UMMA_BLOCK / 2>(b);
                            if (2 * h + KNN_UMMA_BLOCK > u.rows) {
                                bm = 0x7FFF7FFFu;
#pragma unroll
                                for (int jj = 0; jj < KNN_UMMA_BLOCK / 2; ++jj) {
                                    const int col = 2 * (h + jj);
                                    bm = __vmins2(bm, col >= u.rows ? 0x7FFF7FFFu : col + 1 >= u.rows ? (b[jj] & 0xFFFFu) | 0x7FFF0000u : b[jj]);
                                }
                            }
                            if (qn + min(s16_lo(bm), s16_hi(bm)) < thr) {
#pragma unroll
                                for (int jj = 0; jj < KNN_UMMA_BLOCK; ++jj) {
                                    const int col = 2 * h + jj;
                                    const int v = (jj & 1) ? s16_hi(b[jj >> 1]) : s16_lo(b[jj >> 1]);
                                    if (col < u.rows) top2_insert(B0, B1, make_key64(static_cast<uint32_t>(qn + v), u.key0 + col));
                                }
                                thr = sc.threshold(B1);
                            }
                        }
                    }
                } else {
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
                        sc.loaded(v, half, k);
                        if (u.rows < KNN_UMMA_ROWS) {
#pragma unroll
                            for (int q = 0; q < 2; ++q)
#pragma unroll
                                for (int jj = 0; jj < 32; ++jj)
                                    if (64 * half + 32 * q + jj >= u.rows) v[q][jj] = 0x3FFFFFFF; // rows past the unit: never below any bound
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
                                        if (col < u.rows) top2_insert(B0, B1, make_key64(static_cast<uint32_t>(qn + v[q][h + jj]), u.key0 + col));
                                    }
                                    thr = sc.threshold(B1);
                                }
                            }
                    }
                }
                sc.end_unit(sg, i, k, u.rows, B0, B1, thr);
#ifdef PLM_UMMA_STAMPS
                ++units_done;
#endif
            }
            sc.end_segment(sg, B0, B1);
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
    tc_syncthreads(); // every MMA was waited for by the readout (or a wait timed out and the results are discarded)
    if (warp == 0) tmem_dealloc<512>(tmem);
}

// knn2_umma_kernel's units and readout: rows of one task, keys idx_base + row, the shared bound gthr, one partial slot
// per segment.
struct KnnScan {
    static constexpr bool PACKED = true;
    KnnTask t;
    // per segment
    int slot, gcap;
    uint32_t *gthr;
    uint32_t gnext; // *gthr as read one unit ahead of its use

    __device__ __forceinline__ int rows_of(long long u) const { return static_cast<int>(min(static_cast<long long>(KNN_UMMA_ROWS), t.n2 - u * KNN_UMMA_ROWS)); }
    __device__ __forceinline__ const uint4 *unit_src(long long u, int &rows) const {
        rows = rows_of(u);
        return t.db + 2 * (u * KNN_UMMA_ROWS);
    }
    __device__ __forceinline__ void begin_segment(const UmmaSeg &s) {
        slot = umma_slot(static_cast<long long>(s.g) * t.n_units, t.n1, t.n_units);
        gthr = (t.gthr && s.valid) ? t.gthr + s.qi : nullptr;
        gcap = 1023;
        if (gthr) gnext = *reinterpret_cast<volatile uint32_t *>(gthr);
    }
    __device__ __forceinline__ UmmaCols begin_unit(const UmmaSeg &s, int i, int &thr) {
        // Once per unit: the bound the other CTAs have reached (rows AT the bound stay in), read one unit ahead so that
        // no unit waits an L2 round trip for it.  This is exact: gthr only decreases (atomicMin), so the value read a
        // unit earlier is >= the current one, and a larger bound only lets more rows into the insert path, whose test
        // and top2_insert are exact.  Unit 0 of a segment uses the value read at segment start.
        if (gthr) {
            gcap = static_cast<int>(min(gnext, 1022u)) + 1;
            thr = min(thr, gcap);
            gnext = *reinterpret_cast<volatile uint32_t *>(gthr); // for unit i + 1
        }
        // idx_base + n2 <= 2^32 (checked by the host)
        const long long u = s.u0 + i;
        return {rows_of(u), static_cast<uint32_t>(t.idx_base) + static_cast<uint32_t>(u * KNN_UMMA_ROWS)};
    }
    __device__ __forceinline__ int threshold(unsigned long long B1) const {
        const int own = (B1 == KEY64_ABSENT) ? 1023 : static_cast<int>(B1 >> 32);
        if (gthr && own < 1023) atomicMin(gthr, static_cast<uint32_t>(own));
        return min(own, gcap);
    }
    __device__ __forceinline__ void end_unit(const UmmaSeg &, int, uint32_t, int, unsigned long long &, unsigned long long &, int &) {}
    __device__ __forceinline__ void end_segment(const UmmaSeg &s, unsigned long long B0, unsigned long long B1) {
        if (!s.valid) return;
        t.part[static_cast<size_t>(slot) * t.n1 + s.qi] = make_ulonglong2(B0, B1);
        if (s.u0 + s.n == t.n_units) // the last segment of the group
            for (int p = slot + 1; p < t.n_workers; ++p) t.part[static_cast<size_t>(p) * t.n1 + s.qi] = make_ulonglong2(KEY64_ABSENT, KEY64_ABSENT);
    }
};

__global__ void __launch_bounds__(KNN_UMMA_CTA_THREADS, 1) knn2_umma_kernel(const KnnTask t, int32_t *err, long long spin_limit) {
    KnnScan sc{t};
    umma_pipeline(sc, t.q, t.n1, t.n_units, err, spin_limit);
}

// Back-to-back 128 x N x 32 int8 MMAs on zeroed operands (one CTA per SM): the INT8 tensor-core rate of this card at
// N = 256 (the peak) and at N = 128 (the shape knn2_umma_kernel issues).  With STS, warps 1-3 keep storing 16-byte
// chunks to a separate 32 KB tile while the MMAs run, as the expansion of train units does.  Shared memory:
// KNN_UMMA_RATE_SMEM.
template <int N, bool STS>
__global__ void __launch_bounds__(128, 1) mma_i8_rate_kernel(int iters, int32_t *err, long long spin_limit) {
    __shared__ __align__(8) unsigned long long bar;
    __shared__ uint32_t tmem_slot;
    uint8_t *smem = umma_smem();
    for (int i = threadIdx.x; i < 3 * KNN_UMMA_TILE_BYTES / 16; i += blockDim.x) reinterpret_cast<uint4 *>(smem)[i] = make_uint4(0, 0, 0, 0);
    const uint32_t sA = static_cast<uint32_t>(__cvta_generic_to_shared(smem)), sB = sA + KNN_UMMA_TILE_BYTES;
    const uint32_t sbar = static_cast<uint32_t>(__cvta_generic_to_shared(&bar));
    if (threadIdx.x < 32) tmem_alloc<256>(&tmem_slot);
    if (threadIdx.x == 0) {
        mbar_init(sbar, 1);
        mbar_init_fence();
    }
    fence_proxy_async_smem();
    tc_syncthreads();
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
    tc_syncthreads();
    if (threadIdx.x < 32) tmem_dealloc<256>(tmem);
}

} // namespace plm
