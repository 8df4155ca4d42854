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
#pragma once
#include "plm_common.cuh"

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

} // namespace plm
