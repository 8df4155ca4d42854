// Map landmarks: representative ("median") descriptor and mean observation direction, batched.
//
// PLSLAM::MapPoint::updateAverageDescDir (src/mapFeatures.cpp:51-93) and MapLine::updateAverageDescDir
// (:121-163) -- the producer of the med_desc rows that map-to-keyframe matching reads
// (mapHandler.cpp:596-609, :698-714).  For a landmark with n observations the reference builds the n x n
// Hamming matrix, takes per row the element at sorted position int(1 + 0.5*(n-1)) (self distance
// included) and keeps the FIRST row whose value is strictly smallest; the direction is the plain mean of
// the observation directions, summed in list order.
//
// Layout: observations of landmark l are rows obs_start[l] .. obs_start[l+1]-1 of one descriptor arena
// (n_obs x 32 B) and one direction arena (n_obs x 3 doubles).  The work is HBM / latency bound
// (n*n/2 pairs on n*56 bytes), so the kernels are organised around one coalesced pass over the arenas:
//
//  * med_desc_warp_kernel: lists of up to 32 observations (every list the SLAM system produces in practice: a
//    landmark is seen from a few dozen keyframes at most).  A warp takes 4 consecutive landmarks and packs them
//    by their longest list -- 4 landmarks x 8 lanes, 2 x 16 or 1 x 32 -- so short lists do not idle most of the
//    warp.  Sub-lane i of a group owns observation i in registers; row j is re-read from L1; the distances of a
//    lane's row stay in registers, padded to the group width, and go through a bitonic sorting network (all
//    indices compile-time); the winner is a butterfly min over the group on (value << 5 | sub-lane) -- lowest row on ties
//    like the reference's strict `<`.
//  * med_desc_cta_kernel: landmarks with more than 32 observations are appended to a device work list by
//    the first kernel and handled by persistent CTAs (one thread per row, distances recomputed in each
//    search step from L1-resident rows).  No host round trip between the two launches.
#pragma once
#include "plm_common.cuh"

namespace plm {

constexpr int MED_WARPS = 4;   // landmarks in flight per CTA of the warp kernel
constexpr int MED_CTA_THREADS = 256;

// A work item finds its list in one of two ways:
//  * CSR (lm_ids == null): item l is landmark l, its rows are obs_start[l] .. obs_start[l+1]-1;
//  * start / length table (lm_ids != null): item w is landmark l = lm_ids[w], its rows are obs_start[l] ..
//    obs_start[l] + obs_len[l] - 1 (the reserved runs of the resident local map, plm_localmap_api.inl); med_desc and
//    med_dir are then written at landmark l, med_idx at item w.
struct MedArgs {
    const uint4 *desc;        // n_obs x 32 B
    const double *dirs;       // n_obs x 3, or null
    const int32_t *obs_start; // n_lm + 1 (CSR) or one entry per landmark (table)
    long long n_obs;
    int n_lm;                 // work items
    int32_t *med_idx;        // n_lm: winning position inside the list, -1 for an empty / malformed list
    uint4 *med_desc;         // n_lm x 32 B, or null
    const int32_t *dst_rows; // optional: landmark l writes row dst_rows[l] of med_desc (< 0: skip) -- scatter into a map DB
    double *med_dir;         // n_lm x 3, or null
    int32_t *work;           // [0] = number of long lists, [1 ..] = their item ids
    const int32_t *lm_ids;   // optional: landmark of each item (table form)
    const int32_t *obs_len;  // table form: list length per landmark
};

// Rows of item w: [*lo, *lo + returned length) (the raw length; the caller rejects malformed ranges).
template <bool TABLE>
__device__ __forceinline__ long long med_list(const MedArgs &a, long long w, long long &lo) {
    if (TABLE) {
        const int l = __ldg(a.lm_ids + w);
        lo = __ldg(a.obs_start + l);
        return __ldg(a.obs_len + l);
    }
    lo = __ldg(a.obs_start + w);
    return static_cast<long long>(__ldg(a.obs_start + w + 1)) - lo;
}

// Row of med_desc / med_dir that item w writes.
template <bool TABLE>
__device__ __forceinline__ long long med_out(const MedArgs &a, long long w) { return TABLE ? __ldg(a.lm_ids + w) : w; }

// int(1 + 0.5 * (n - 1)) of mapFeatures.cpp:79 for n >= 2
__device__ __forceinline__ int med_rank(int n) { return 1 + (n - 1) / 2; }

__device__ __forceinline__ Desc shfl_desc(const Desc &q, int src) {
    Desc t;
    t.lo.x = __shfl_sync(0xFFFFFFFFu, q.lo.x, src);
    t.lo.y = __shfl_sync(0xFFFFFFFFu, q.lo.y, src);
    t.lo.z = __shfl_sync(0xFFFFFFFFu, q.lo.z, src);
    t.lo.w = __shfl_sync(0xFFFFFFFFu, q.lo.w, src);
    t.hi.x = __shfl_sync(0xFFFFFFFFu, q.hi.x, src);
    t.hi.y = __shfl_sync(0xFFFFFFFFu, q.hi.y, src);
    t.hi.z = __shfl_sync(0xFFFFFFFFu, q.hi.z, src);
    t.hi.w = __shfl_sync(0xFFFFFFFFu, q.hi.w, src);
    return t;
}

// Mean direction of one landmark, component c (mapFeatures.cpp:88-91): sequential fp64 sum in list
// order from zero, one IEEE division by n.  A single observation keeps its direction (constructor, :38).
__device__ __forceinline__ double med_dir_component(const double *__restrict__ dirs, long long lo, int n, int c) {
    if (n <= 0) return 0.0;
    if (n == 1) return __ldg(dirs + 3 * lo + c);
    double s = 0.0;
    for (int i = 0; i < n; ++i) s = __dadd_rn(s, __ldg(dirs + 3 * (lo + i) + c));
    return __ddiv_rn(s, static_cast<double>(n));
}

// Batcher's odd-even merge sort as a comparator network over a register array (19 / 63 / 191 comparators for 8 / 16 /
// 32 inputs; explicit lists generated and 0-1-verified by tools/gen_sort_networks.py).  Only d[G / 2] is read afterwards,
// so the compiler drops the comparators (and the min or max halves) that output does not depend on.
#include "plm_sort_networks.inc"
#define PLM_CE(A, B)                  \
    {                                 \
        const int x = d[A], y = d[B]; \
        d[A] = min(x, y);             \
        d[B] = max(x, y);             \
    }
__device__ __forceinline__ void med_sort_network(int (&d)[8]) { PLM_SORT_NET_8(PLM_CE) }
__device__ __forceinline__ void med_sort_network(int (&d)[16]) { PLM_SORT_NET_16(PLM_CE) }
__device__ __forceinline__ void med_sort_network(int (&d)[32]) { PLM_SORT_NET_32(PLM_CE) }
#undef PLM_CE

// One pass of a warp over 32 / G landmarks, G lanes each (G = 8, 16 or 32): sub-lane i of a group owns observation i
// and keeps the distances of its row in REGISTERS (every loop below is unrolled over compile-time indices).
// `n` / `lo` are this lane's group values (n = 0 for a group without a landmark in this pass; lists longer than G
// never get here); `nmax` is the warp-uniform maximum of n over the groups of the pass.
//
// Every pair once: lane i computes d(i, i + k mod n) for k = 1 .. n / 2 and receives d(i - k mod n, i) from lane
// i - k by shuffle (k = 1 .. (n - 1) / 2), so a row of n entries costs n / 2 Hamming distances instead of n.  The row
// (self distance 0 included, mapFeatures.cpp:66-76) is a multiset -- its order does not matter to the sort.
//
// Selection instead of a full sort: the wanted element sits at sorted position r = int(1 + 0.5 * (n - 1)) of the n
// real entries (mapFeatures.cpp:79); the G - n unused slots hold 0x7FFF and sink to the end.  The classes are cut so
// that r is one of G / 4 positions (lists of a 16- or 32-lane pass have n > G / 2), and only those outputs of the
// network are read -- the compiler prunes the comparators that none of them depends on.
template <int G, bool TABLE>
__device__ __forceinline__ void med_desc_pass(const MedArgs &a, double *sdir, long long lm, long long lo, int n, int nmax,
                                              bool valid) {
    const int lane = threadIdx.x & 31, sl = lane & (G - 1);
    Desc q{make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0)};
    const bool want_dir = a.med_dir && a.dirs;
    if (sl < n) {
        q = load_desc(a.desc, lo + sl);
        if (want_dir) { // the owner lane fetches its observation's direction now, next to the descriptor (one HBM round trip)
            const double *dp = a.dirs + 3 * (lo + sl);
            sdir[3 * lane] = __ldg(dp);
            sdir[3 * lane + 1] = __ldg(dp + 1);
            sdir[3 * lane + 2] = __ldg(dp + 2);
        }
    }
    int best = n > 0 ? 0 : -1;
    if (nmax >= 2) {
        int d[G];
        d[0] = (sl < n) ? 0 : 0x7FFF; // self distance
        const int gbase = lane - sl;
        const uint4 *rows = a.desc + 2 * (n > 0 ? lo : 0); // a group without a landmark reads row 0 (nmax >= 2: it exists)
#pragma unroll
        for (int k = 1; k <= G / 2; ++k) {
            int own = 0x7FFF, recv = 0x7FFF;
            if (2 * k <= nmax) { // warp-uniform
                const bool act = sl < n && 2 * k <= n;
                int j = sl + k;
                j -= (j >= n) ? n : 0;
                const int jc = act ? j : 0; // idle lanes re-read the list's first row (one broadcast request)
                const uint4 tlo = __ldg(rows + 2 * jc), thi = __ldg(rows + 2 * jc + 1); // L1-resident: the owner lane fetched it above
                const int dist = hamming256_csa4(q, tlo, thi);
                own = act ? dist : 0x7FFF;
                int src = sl - k;
                src += (src < 0) ? n : 0;
                recv = __shfl_sync(0xFFFFFFFFu, own, gbase + (src & (G - 1)));
                recv = (2 * k < n) ? recv : 0x7FFF;
            }
            d[2 * k - 1] = own;
            if (2 * k < G) d[2 * k] = recv;
        }
        // unused slots hold 0x7FFF and sink to the end: the wanted element is at sorted position med_rank(n), one of
        // G / 4 + 1 .. G / 2 for the lists of this class (n > G / 2) -- and of 1 .. 4 in the 8-lane class
        med_sort_network(d);
        const int rank = med_rank(n);
        int med = d[G / 2];
#pragma unroll
        for (int pos = (G == 8) ? 1 : G / 4 + 1; pos < G / 2; ++pos) med = (rank == pos) ? d[pos] : med;
        uint32_t key = (sl < n && n >= 2) ? (static_cast<uint32_t>(med) << 5) | sl : KEY32_ABSENT;
#pragma unroll
        for (int off = G / 2; off > 0; off >>= 1) key = min(key, __shfl_xor_sync(0xFFFFFFFFu, key, off));
        if (n >= 2) best = static_cast<int>(key & 31u);
    }
    if (valid) {
        if (sl == 0) a.med_idx[lm] = best;
        if (a.med_desc) {
            const long long row = a.dst_rows ? __ldg(a.dst_rows + lm) : med_out<TABLE>(a, lm);
            if (row >= 0 && sl == (best < 0 ? 0 : best)) { // the winner writes its own registers (zeros for an empty list)
                a.med_desc[2 * row] = q.lo;
                a.med_desc[2 * row + 1] = q.hi;
            }
        }
    }
    if (want_dir) {
        __syncwarp();
        if (valid && sl < 3) { // mean direction (mapFeatures.cpp:88-91): sequential sum in list order from zero, / n
            const double *g = sdir + 3 * (lane - sl) + sl; // component sl of the group's observation 0
            double r = 0.0;
            if (n == 1) {
                r = g[0]; // a single observation keeps its direction (constructor, :38)
            } else if (n >= 2) {
                double acc = 0.0;
#pragma unroll
                for (int j = 0; j < G; ++j)
                    if (j < n) acc = __dadd_rn(acc, g[3 * j]);
                r = __ddiv_rn(acc, static_cast<double>(n));
            }
            a.med_dir[3 * med_out<TABLE>(a, lm) + sl] = r;
        }
        __syncwarp();
    }
}

// The g-th (0-based) set bit of `m`, or -1.
__device__ __forceinline__ int med_nth_bit(unsigned m, int g) {
#pragma unroll
    for (int t = 0; t < 3; ++t)
        if (t < g) m &= m - 1;
    return m ? __ffs(m) - 1 : -1;
}

// A warp takes a chunk of 32 consecutive landmarks (lane l reads the offsets of landmark 32 * chunk + l -- one coalesced
// request), sorts them into three classes by list length and works each class off at its own packing: 4 landmarks x 8
// lanes for lists of <= 8 observations, 2 x 16 for <= 16, 1 x 32 for <= 32.  (Packing by the longest list of 4
// NEIGHBOURS put 86 % of a Poisson(8) map into the 16-lane form.)  Longer lists go to the work list of
// med_desc_cta_kernel.
template <bool TABLE>
__global__ void __launch_bounds__(32 * MED_WARPS) med_desc_warp_kernel(MedArgs a) {
    __shared__ double sdir_all[MED_WARPS][32 * 3];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double *sdir = sdir_all[warp];
    const long long n_chunks = (static_cast<long long>(a.n_lm) + 31) / 32;
    const long long stride = static_cast<long long>(gridDim.x) * MED_WARPS;
    auto fetch = [&](long long chunk, long long &lo, int &n) {
        const long long my_lm = chunk * 32 + lane;
        lo = 0;
        n = -2; // past the end
        if (chunk < n_chunks && my_lm < a.n_lm) {
            const long long len = med_list<TABLE>(a, my_lm, lo);
            n = (lo < 0 || len < 0 || lo + len > a.n_obs) ? 0 : static_cast<int>(min(len, 1LL << 30)); // malformed: empty
        }
    };
    long long chunk = static_cast<long long>(blockIdx.x) * MED_WARPS + warp;
    long long nx_lo;
    int nx_n;
    fetch(chunk, nx_lo, nx_n);
    for (; chunk < n_chunks; chunk += stride) {
        const long long my_lo = nx_lo;
        const int my_n = nx_n;
        // the chunk's observations are one contiguous range of the arenas: ask L2 for all of it now, the passes below
        // then wait on L2, not on HBM (CSR form only: the runs of the table form are scattered)
        if (!TABLE) {
            const long long first = __shfl_sync(0xFFFFFFFFu, my_lo, 0);
            const unsigned live = __ballot_sync(0xFFFFFFFFu, my_n >= 0);
            const int last_lane = 31 - __clz(live | 1u);
            const long long end = __shfl_sync(0xFFFFFFFFu, my_lo + max(my_n, 0), last_lane);
            const char *p0 = reinterpret_cast<const char *>(a.desc) + first * 32;
            const long long bytes = min((end - first) * 32, 64LL * 1024);
            for (long long o = static_cast<long long>(lane) * 128; o < bytes; o += 32 * 128)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(p0 + o));
            if (a.dirs && a.med_dir) {
                const char *p1 = reinterpret_cast<const char *>(a.dirs) + first * 24;
                const long long b1 = min((end - first) * 24, 64LL * 1024);
                for (long long o = static_cast<long long>(lane) * 128; o < b1; o += 32 * 128)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(p1 + o));
            }
        }
        fetch(chunk + stride, nx_lo, nx_n);
        const unsigned m_long = __ballot_sync(0xFFFFFFFFu, my_n > 32);
        if (m_long) {
            int base = 0;
            if (lane == 0) base = atomicAdd(a.work, __popc(m_long));
            base = __shfl_sync(0xFFFFFFFFu, base, 0);
            if (my_n > 32) a.work[1 + base + __popc(m_long & ((1u << lane) - 1))] = static_cast<int32_t>(chunk * 32 + lane);
        }
        unsigned m8 = __ballot_sync(0xFFFFFFFFu, my_n >= 0 && my_n <= 8);
        unsigned m16 = __ballot_sync(0xFFFFFFFFu, my_n > 8 && my_n <= 16);
        unsigned m32 = __ballot_sync(0xFFFFFFFFu, my_n > 16 && my_n <= 32);
        while (m8) {
            const int src = med_nth_bit(m8, lane >> 3);
            const int n_src = __shfl_sync(0xFFFFFFFFu, my_n, src & 31);
            const int n = src >= 0 ? n_src : 0;
            const long long lo = __shfl_sync(0xFFFFFFFFu, my_lo, src & 31);
            const int nmax = __reduce_max_sync(0xFFFFFFFFu, n);
            med_desc_pass<8, TABLE>(a, sdir, chunk * 32 + src, lo, n, nmax, src >= 0);
#pragma unroll
            for (int t = 0; t < 4; ++t) m8 &= m8 - 1;
        }
        while (m16) {
            const int src = med_nth_bit(m16, lane >> 4);
            const int n_src = __shfl_sync(0xFFFFFFFFu, my_n, src & 31);
            const int n = src >= 0 ? n_src : 0;
            const long long lo = __shfl_sync(0xFFFFFFFFu, my_lo, src & 31);
            const int nmax = __reduce_max_sync(0xFFFFFFFFu, n);
            med_desc_pass<16, TABLE>(a, sdir, chunk * 32 + src, lo, n, nmax, src >= 0);
            m16 &= m16 - 1;
            m16 &= m16 - 1;
        }
        while (m32) {
            const int src = __ffs(m32) - 1;
            const int n = __shfl_sync(0xFFFFFFFFu, my_n, src);
            const long long lo = __shfl_sync(0xFFFFFFFFu, my_lo, src);
            med_desc_pass<32, TABLE>(a, sdir, chunk * 32 + src, lo, n, n, true);
            m32 &= m32 - 1;
        }
    }
}

constexpr int MED_CTA_CACHE_N = 128; // lists up to this length keep their rows and their distance matrix in shared memory

// Lists of more than 32 observations (the work list of the warp kernel), one per CTA at a time.  Up to 128 observations
// the rows are staged in shared memory, every pair is computed once into a uint16 matrix, and a row's rank search
// (smallest v with #{d <= v} >= rank + 1, bisection over 0 .. 256) is shared by 2 or 4 lanes that each count a
// strided part of the row and add up by shuffle; longer lists fall back to one thread per row recomputing distances.
template <bool TABLE>
__global__ void __launch_bounds__(MED_CTA_THREADS) med_desc_cta_kernel(MedArgs a) {
    __shared__ unsigned long long s_best;
    __shared__ uint16_t s_dist[MED_CTA_CACHE_N * MED_CTA_CACHE_N];
    __shared__ uint4 s_rows[MED_CTA_CACHE_N * 2];
    __shared__ double s_dirs[MED_CTA_CACHE_N * 3];
    const int n_work = a.work[0];
    for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
        const long long lm = a.work[1 + w];
        long long lo;
        const int n = static_cast<int>(med_list<TABLE>(a, lm, lo));
        if (threadIdx.x == 0) s_best = KEY64_ABSENT;
        const bool cached = n <= MED_CTA_CACHE_N;
        const int need = med_rank(n) + 1;
        if (cached) {
            for (int i = threadIdx.x; i < 2 * n; i += MED_CTA_THREADS) s_rows[i] = __ldg(a.desc + 2 * lo + i);
            if (a.med_dir && a.dirs)
                for (int i = threadIdx.x; i < 3 * n; i += MED_CTA_THREADS) s_dirs[i] = __ldg(a.dirs + 3 * lo + i);
            __syncthreads();
            // every pair once, mirrored: item (i, k) is the pair (i, i + k mod n), k = 1 .. n / 2; for even n the offset
            // n / 2 reaches each pair from both ends, so only its first half is taken
            const int half = n >> 1;
            for (int idx = threadIdx.x; idx < n * half; idx += MED_CTA_THREADS) {
                const int k = idx / n + 1, i = idx - (k - 1) * n;
                if (2 * k == n && i >= half) continue;
                int j = i + k;
                j -= (j >= n) ? n : 0;
                const Desc qa{s_rows[2 * i], s_rows[2 * i + 1]};
                const uint16_t dist = static_cast<uint16_t>(hamming256(qa, s_rows[2 * j], s_rows[2 * j + 1]));
                s_dist[i * n + j] = dist;
                s_dist[j * n + i] = dist;
            }
            for (int i = threadIdx.x; i < n; i += MED_CTA_THREADS) s_dist[i * n + i] = 0;
            __syncthreads();
            const int T = (n <= MED_CTA_THREADS / 4) ? 4 : 2; // lanes per row
            const int part = threadIdx.x & (T - 1);
            for (int base = 0; base < n; base += MED_CTA_THREADS / T) { // uniform trip count: the shuffles need whole warps
                const int i = base + threadIdx.x / T;
                const uint16_t *row = s_dist + min(i, n - 1) * n;
                int v_lo = 0, v_hi = 256;
#pragma unroll 1
                for (int step = 0; step < 8; ++step) { // 256 -> 1 in exactly 8 halvings; v_lo == v_hi earlier is harmless
                    const int mid = (v_lo + v_hi) >> 1;
                    int c = 0;
                    for (int j = part; j < n; j += T) c += (row[j] <= mid);
                    c += __shfl_xor_sync(0xFFFFFFFFu, c, 1);
                    if (T == 4) c += __shfl_xor_sync(0xFFFFFFFFu, c, 2);
                    if (v_lo < v_hi) {
                        if (c >= need) v_hi = mid;
                        else v_lo = mid + 1;
                    }
                }
                if (i < n && part == 0) atomicMin(&s_best, make_key64(static_cast<uint32_t>(v_lo), static_cast<uint32_t>(i)));
            }
        } else {
            __syncthreads();
            for (int i = threadIdx.x; i < n; i += MED_CTA_THREADS) {
                const Desc q = load_desc(a.desc, lo + i);
                int v_lo = 0, v_hi = 256;
                while (v_lo < v_hi) {
                    const int mid = (v_lo + v_hi) >> 1;
                    int c = 0;
                    for (int j = 0; j < n; ++j) c += (hamming256(q, load_desc(a.desc, lo + j)) <= mid);
                    if (c >= need) v_hi = mid;
                    else v_lo = mid + 1;
                }
                atomicMin(&s_best, make_key64(static_cast<uint32_t>(v_lo), static_cast<uint32_t>(i)));
            }
        }
        __syncthreads();
        const int best = static_cast<int>(s_best & 0xFFFFFFFFull);
        if (threadIdx.x == 0) a.med_idx[lm] = best;
        if (a.med_desc && threadIdx.x < 2) {
            const long long row = a.dst_rows ? __ldg(a.dst_rows + lm) : med_out<TABLE>(a, lm);
            if (row >= 0) a.med_desc[2 * row + threadIdx.x] = __ldg(a.desc + 2 * (lo + best) + threadIdx.x);
        }
        if (a.med_dir && a.dirs && threadIdx.x >= 32 && threadIdx.x < 35) {
            const int c = threadIdx.x - 32;
            const long long out = med_out<TABLE>(a, lm);
            if (cached) { // same sequential sum as med_dir_component, from the staged copy (60 dependent L2 reads otherwise)
                double acc = 0.0;
                for (int i = 0; i < n; ++i) acc = __dadd_rn(acc, s_dirs[3 * i + c]);
                a.med_dir[3 * out + c] = __ddiv_rn(acc, static_cast<double>(n));
            } else {
                a.med_dir[3 * out + c] = med_dir_component(a.dirs, lo, n, c);
            }
        }
        __syncthreads();
    }
}

} // namespace plm
