// Kernels of the resident local map (plm_localmap_*, csrc/plm_localmap_api.inl): the scatters that keep the per-landmark
// arrays up to date.  Selection, gather, matchGrid, the brute-force fallback, the gate and the medoid are the existing
// kernels (plm_reproj.cuh, plm_grid.cuh, plm_knn2.cuh, plm_map.cuh); nothing here computes a match.
//
// Per landmark l (slot = the reference's index into map_points / map_lines):
//   X[l]          3 doubles (point) or 6 (segment endpoints)
//   active[l]     the selection byte of plm_map_select (0 for a culled slot)
//   med_desc[l]   32 B, med_dir[l] 3 doubles
//   obs_start[l], obs_len[l]: the landmark's observations are rows obs_start .. obs_start + obs_len - 1 of the observation
//                 arenas (obs_desc: 32 B per row, obs_dir: 3 doubles per row), inside a run reserved for it.
//
// kf_grid_kernel builds the keyframe side's grids for plm_localmap_match_kf_pl: one CTA per kind (points, segments).
#pragma once
#include "plm_common.cuh"
#include "plm_grid.cuh"
#include "plm_line_walk.cuh"

namespace plm {

struct LmArrays {
    double *X;
    uint8_t *active;
    uint4 *med_desc;
    double *med_dir;
    int32_t *obs_start, *obs_len;
    uint4 *obs_desc;
    double *obs_dir;
    int xw; // doubles per landmark position: 3 or 6
};

// n new landmarks first .. first + n - 1; landmark first + k gets rows row0 + k * run .. (one observation used): the
// constructors of MapPoint / MapLine (mapFeatures.cpp:29-40, :99-110): med_desc = desc, med_dir = dir.
__global__ void __launch_bounds__(256) localmap_insert_kernel(LmArrays m, int first, int n, int row0, int run, const double *__restrict__ X,
                                                              const uint4 *__restrict__ desc, const double *__restrict__ dir) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const size_t l = size_t(first) + k, row = size_t(row0) + size_t(k) * run;
    for (int c = 0; c < m.xw; ++c) m.X[l * m.xw + c] = X[size_t(k) * m.xw + c];
    m.active[l] = 1;
    const uint4 lo = desc[2 * size_t(k)], hi = desc[2 * size_t(k) + 1];
    m.med_desc[2 * l] = lo;
    m.med_desc[2 * l + 1] = hi;
    m.obs_desc[2 * row] = lo;
    m.obs_desc[2 * row + 1] = hi;
    for (int c = 0; c < 3; ++c) {
        const double d = dir[3 * size_t(k) + c];
        m.med_dir[3 * l + c] = d;
        m.obs_dir[3 * row + c] = d;
    }
    m.obs_start[l] = static_cast<int32_t>(row);
    m.obs_len[l] = 1;
}

// Sparse updates of one call: entry k with idx[k] >= 0 writes X[idx] (X != null) and active[idx] = val[k] (val != null)
// or 0 (cull != 0).  Entries with idx < 0 are skipped (an earlier duplicate of the same slot: the last one wins).
__global__ void __launch_bounds__(256) localmap_scatter_kernel(LmArrays m, int n, const int32_t *__restrict__ idx, const double *__restrict__ X,
                                                               const uint8_t *__restrict__ val, int cull) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int l = idx[k];
    if (l < 0) return;
    if (X)
        for (int c = 0; c < m.xw; ++c) m.X[size_t(l) * m.xw + c] = X[size_t(k) * m.xw + c];
    if (val) m.active[l] = val[k];
    if (cull) m.active[l] = 0;
}

// Observation append of one call.  u touched landmarks (record r: landmark ids[r], list old_start[r] / old_len[r] ->
// new_start[r] / new_len[r]); a record whose start moved copies its old_len rows to the new run (the list outgrew its
// run and was given a doubled one at the tail of the arenas).  n new observations go to rows dst[i].  Moved rows,
// appended rows and the old runs are disjoint, so one launch does all of it: a warp per record, a thread per observation.
__global__ void __launch_bounds__(256) localmap_append_kernel(LmArrays m, int u, const int32_t *__restrict__ ids, const int32_t *__restrict__ old_start,
                                                              const int32_t *__restrict__ new_start, const int32_t *__restrict__ old_len,
                                                              const int32_t *__restrict__ new_len, int n, const int32_t *__restrict__ dst,
                                                              const uint4 *__restrict__ desc, const double *__restrict__ dir) {
    const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long rec_threads = 32LL * u;
    if (t < rec_threads) {
        const int r = static_cast<int>(t >> 5), lane = static_cast<int>(t & 31);
        const size_t s0 = size_t(old_start[r]), s1 = size_t(new_start[r]);
        if (s0 != s1)
            for (int i = lane; i < old_len[r]; i += 32) {
                m.obs_desc[2 * (s1 + i)] = m.obs_desc[2 * (s0 + i)];
                m.obs_desc[2 * (s1 + i) + 1] = m.obs_desc[2 * (s0 + i) + 1];
                for (int c = 0; c < 3; ++c) m.obs_dir[3 * (s1 + i) + c] = m.obs_dir[3 * (s0 + i) + c];
            }
        if (lane == 0) {
            m.obs_start[ids[r]] = new_start[r];
            m.obs_len[ids[r]] = new_len[r];
        }
        return;
    }
    const long long i = t - rec_threads;
    if (i >= n) return;
    const size_t row = size_t(dst[i]);
    m.obs_desc[2 * row] = desc[2 * i];
    m.obs_desc[2 * row + 1] = desc[2 * i + 1];
    for (int c = 0; c < 3; ++c) m.obs_dir[3 * row + c] = dir[3 * i + c];
}

// Read-back gather: entry k of idx -> X, med_desc, med_dir rows k of the outputs (each may be null).
__global__ void __launch_bounds__(256) localmap_read_kernel(LmArrays m, int n, const int32_t *__restrict__ idx, double *__restrict__ X,
                                                            uint4 *__restrict__ med_desc, double *__restrict__ med_dir) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const size_t l = size_t(idx[k]);
    if (X)
        for (int c = 0; c < m.xw; ++c) X[size_t(k) * m.xw + c] = m.X[l * m.xw + c];
    if (med_desc) {
        med_desc[2 * size_t(k)] = m.med_desc[2 * l];
        med_desc[2 * size_t(k) + 1] = m.med_desc[2 * l + 1];
    }
    if (med_dir)
        for (int c = 0; c < 3; ++c) med_dir[3 * size_t(k) + c] = m.med_dir[3 * l + c];
}

// ---- keyframe grids in global memory (StVO::GridStructure as CSR, the layout of grid.py) ----------------------------
// One kind's grid: n features (points: (x, y) float pixels; segments: (sx, sy, ex, ey)), n <= KF_GRID_MAX_FEATS.
// cell_start: n_cells + 1 entries, cell_items: the items, unsorted: the same capacity (the fill before the in-cell sort),
// big: n_cells entries of scratch, dirs: n x 2 unit directions (segments only).
struct KfGridJob {
    const float *geo;
    int32_t *cell_start, *cell_items, *unsorted, *big;
    double *dirs;
    int32_t n, is_lines;
};
struct KfGridArgs {
    KfGridJob job[2];
    double inv_w, inv_h;  // of the map view: GRID_COLS / image width, GRID_ROWS / image height
    int32_t grid_rows, grid_cols;
};
constexpr int KF_GRID_THREADS = 1024;
constexpr int KF_GRID_MAX_FEATS = 32 * KF_GRID_THREADS; // one bit per feature, one bitmap word per thread
constexpr int KF_GRID_MAX_CELLS = 8192;                 // cell counters in shared memory
constexpr int KF_GRID_SMALL_CELL = 32;                  // larger cells are sorted through the bitmap

// Exclusive sum of one value per thread over the CTA.  s_part needs blockDim.x / 32 ints.
__device__ __forceinline__ int block_exclusive_sum(int v, int32_t *s_part) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int s = 1; s < 32; s <<= 1) {
        const int t = __shfl_up_sync(0xFFFFFFFFu, incl, s);
        if (lane >= s) incl += t;
    }
    if (lane == 31) s_part[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = (lane < int(blockDim.x >> 5)) ? s_part[lane] : 0;
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            const int t = __shfl_up_sync(0xFFFFFFFFu, w, s);
            if (lane >= s) w += t;
        }
        if (lane < int(blockDim.x >> 5)) s_part[lane] = w;
    }
    __syncthreads();
    const int r = incl - v + (warp ? s_part[warp - 1] : 0);
    __syncthreads();
    return r;
}

// The grid fill of stereoFrame.cpp:146-150 (points: grid.at(px * inv_width, py * inv_height), a double product truncated
// toward zero, off-grid points go to the sink) and :336-349 (segments: every cell of getLineCoords over the scaled
// endpoints, plus the direction (ex - sx, ey - sy) -- a float subtraction, then the double product -- normalised as
// matching.h:43-48 does).  The CSR is the host's exactly, items in ascending feature index inside a cell (the
// list::push_back order): a counting sort fills each cell in arbitrary order, then every cell is sorted -- small cells
// by one thread, larger ones by the whole CTA through a bitmap of the features.
__global__ void __launch_bounds__(KF_GRID_THREADS) kf_grid_kernel(const KfGridArgs a) {
    extern __shared__ int32_t s_cs[]; // n_cells + 1
    __shared__ uint32_t s_bits[KF_GRID_MAX_FEATS / 32];
    __shared__ int32_t s_part[KF_GRID_THREADS / 32];
    __shared__ int s_nbig;
    const KfGridJob J = blockIdx.x ? a.job[1] : a.job[0];
    if (J.n <= 0) return;
    const int tid = threadIdx.x, rows = a.grid_rows, cols = a.grid_cols, n_cells = rows * cols;
    const double inv_w = a.inv_w, inv_h = a.inv_h;
    for (int i = tid; i <= n_cells; i += KF_GRID_THREADS) s_cs[i] = 0;
    if (tid == 0) s_nbig = 0;
    __syncthreads();
    auto cells = [&](int j, auto &&f) {
        if (!J.is_lines) {
            const float2 k = reinterpret_cast<const float2 *>(J.geo)[j];
            // compared as doubles: NaN and values past the int range are off the grid, as in grid.py
            const double x = trunc(__dmul_rn(static_cast<double>(k.x), inv_w));
            const double y = trunc(__dmul_rn(static_cast<double>(k.y), inv_h));
            if (x >= 0.0 && x < cols && y >= 0.0 && y < rows) f(static_cast<int>(x) * rows + static_cast<int>(y));
        } else {
            // the host bounds the scaled endpoints (|v| <= 2^20), so the whole walk runs, as the reference's does
            const float4 k = reinterpret_cast<const float4 *>(J.geo)[j];
            line_walk(__dmul_rn(static_cast<double>(k.x), inv_w), __dmul_rn(static_cast<double>(k.y), inv_h),
                      __dmul_rn(static_cast<double>(k.z), inv_w), __dmul_rn(static_cast<double>(k.w), inv_h), INT_MAX,
                      [&](int x, int y) {
                          if (x >= 0 && x < cols && y >= 0 && y < rows) f(x * rows + y);
                      });
        }
    };
    for (int j = tid; j < J.n; j += KF_GRID_THREADS) {
        cells(j, [&](int c) { atomicAdd(&s_cs[c], 1); });
        if (J.is_lines) {
            const float4 k = reinterpret_cast<const float4 *>(J.geo)[j];
            const double vx = __dmul_rn(static_cast<double>(__fsub_rn(k.z, k.x)), inv_w);
            const double vy = __dmul_rn(static_cast<double>(__fsub_rn(k.w, k.y)), inv_h);
            const double mag = __dsqrt_rn(__dadd_rn(__dmul_rn(vx, vx), __dmul_rn(vy, vy)));
            J.dirs[2 * j] = __ddiv_rn(vx, mag);
            J.dirs[2 * j + 1] = __ddiv_rn(vy, mag);
        }
    }
    __syncthreads();
    block_inclusive_scan(s_cs, n_cells, s_part); // cell ends
    if (tid == 0) s_cs[n_cells] = s_cs[n_cells - 1];
    __syncthreads();
    for (int j = tid; j < J.n; j += KF_GRID_THREADS)
        cells(j, [&](int c) { J.unsorted[atomicSub(&s_cs[c], 1) - 1] = j; });
    __syncthreads(); // s_cs[c] = start of cell c
    for (int i = tid; i <= n_cells; i += KF_GRID_THREADS) J.cell_start[i] = s_cs[i];
    for (int c = tid; c < n_cells; c += KF_GRID_THREADS) {
        const int s = s_cs[c], m = s_cs[c + 1] - s;
        if (m > KF_GRID_SMALL_CELL) {
            J.big[atomicAdd(&s_nbig, 1)] = c;
            continue;
        }
        for (int k = 0; k < m; ++k) { // insertion sort
            const int32_t v = J.unsorted[s + k];
            int p = k;
            for (; p > 0 && J.cell_items[s + p - 1] > v; --p) J.cell_items[s + p] = J.cell_items[s + p - 1];
            J.cell_items[s + p] = v;
        }
    }
    __syncthreads();
    const int n_big = s_nbig, words = (J.n + 31) / 32;
    for (int b = 0; b < n_big; ++b) {
        const int c = J.big[b], s = s_cs[c], m = s_cs[c + 1] - s;
        if (tid < words) s_bits[tid] = 0;
        __syncthreads();
        for (int k = tid; k < m; k += KF_GRID_THREADS) {
            const int32_t v = J.unsorted[s + k];
            atomicOr(&s_bits[v >> 5], 1u << (v & 31));
        }
        __syncthreads();
        uint32_t w = tid < words ? s_bits[tid] : 0u;
        int p = s + block_exclusive_sum(__popc(w), s_part);
        for (; w; w &= w - 1) J.cell_items[p++] = tid * 32 + (__ffs(w) - 1);
    }
}

} // namespace plm
