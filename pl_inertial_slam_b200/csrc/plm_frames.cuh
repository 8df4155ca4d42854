// Device-resident stereo-frame pipeline (SURVEY 8f-1 and 8f-4; config 3).
//
// The reference processes a frame as  StereoFrame::matchStereoPoints / matchStereoLines  (grid fill,
// matchGrid, geometry gates, compaction of pdesc_l / ldesc_l to the kept rows, back-projection;
// stvo-pl/src/stereoFrame.cpp:131-184, :320-409)  followed by  StereoFrameHandler::matchF2FPoints /
// matchF2FLines  (StVO::match on the COMPACTED left descriptors of the previous and the current frame;
// stvo-pl/src/stereoFrameHandler.cpp:158-207).  Here both stages run on the device from the raw
// keypoints / line segments / descriptors, two launches per feature type for a whole replay:
//
//   stereo_frame_kernel   one CTA per (frame, feature type): builds the CSR bucket grid of the right
//                         features in shared memory (counting sort; Bresenham walk of
//                         lineIterator.cpp:34-77 for lines), runs the matchGrid phases of plm_grid.cuh
//                         on it, applies the gates of plm_stereo.cuh, block-scans the keep flags and
//                         writes the compacted descriptors + stereo_pt / stereo_ls fields.
//   f2f_match_kernel      one CTA per (frame pair, feature type): StVO::match in ONE pass over the
//                         distance tile -- a thread owns a query row (row top-2 in registers), the
//                         column top-2 comes from REDUX warp minima merged with shared-memory atomics --
//                         then both fp32 ratio tests and the mutual check.  Sizes are read from the
//                         kept counts the stereo stage left on the device.
#pragma once
#include "plm_grid.cuh"
#include "plm_line_walk.cuh"
#include "plm_stereo.cuh"

namespace plm {

struct FrameCfg {
    double inv_w, inv_h;   // GRID_COLS / img.cols, GRID_ROWS / img.rows (stereoFrame.cpp:47-48)
    double ratio;          // Config::minRatio12P(), the matchGrid ratio for points AND lines
    double line_sim_th, max_dist_epip, min_disp, line_horiz_th, stereo_overlap_th, ls_min_disp_ratio;
    double cam_b, cam_fx, cam_cx, cam_cy;
    int grid_rows, grid_cols, matching_s_ws, best_lr;
};

struct StereoJob {
    const float *geo_l, *geo_r; // (x, y) per keypoint or (sx, sy, ex, ey) per line, float pixels
    const uint4 *d_l, *d_r;
    int32_t *m12;               // n_l, the matchGrid vector of the frame (written in full)
    uint4 *cdesc;               // compacted left descriptors (kept rows in i1 order)
    int32_t *kept_i1;           // kept slot -> i1
    double *o0, *o1, *o2, *o3;  // points: disp, P(3)      lines: disp_se(2), sP(3), eP(3), le(3)
    int32_t *counts;            // [0] matchGrid return value, [1] number of kept rows
    int32_t n_l, n_r, is_lines, pad_;
};

struct StereoCaps {
    int cap_l, cap_r, cap_items, warps;
    int cap_pairs, pad_; // candidate slots the pair-list form can hold (more -> chunk phases)
};

__host__ __device__ inline size_t stereo_frame_smem(const StereoCaps &c, int n_cells, bool lines) {
    // scratch of the matcher: pair-list arrays, or (fallback) wmin + m21key of the chunk phases
    const size_t chunk = grid_align16(static_cast<size_t>(c.warps) * c.cap_r * 2) + grid_align16(static_cast<size_t>(c.cap_r) * 4);
    const size_t pairs = pairlist_smem(c.cap_pairs, c.cap_l, c.cap_r);
    size_t b = chunk > pairs ? chunk : pairs;
    b += grid_align16(static_cast<size_t>(n_cells + 1) * 4);               // cell ends -> cell starts
    b += grid_align16(static_cast<size_t>(c.cap_items) * 4);               // cell items
    b += static_cast<size_t>(c.cap_r) * 32;                                // right descriptors
    b += grid_align16(static_cast<size_t>(c.cap_l) * (lines ? 16 : 8));    // query cell coordinates
    b += grid_align16(static_cast<size_t>(c.cap_l) * 4);                   // m12
    if (lines) b += static_cast<size_t>(c.cap_r) * 16;                     // directions
    return b;
}

// PinholeStereoCamera::backProjection (pinholeStereoCamera.cpp:229-237).
__device__ __forceinline__ void back_projection(const FrameCfg &c, double u, double v, double disp, double *P) {
    const double bd = __ddiv_rn(c.cam_b, disp);
    P[0] = __dmul_rn(bd, __dsub_rn(u, c.cam_cx));
    P[1] = __dmul_rn(bd, __dsub_rn(v, c.cam_cy));
    P[2] = __dmul_rn(bd, c.cam_fx);
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS)
stereo_frame_kernel(const StereoJob *__restrict__ jobs, const size_t job_stride, const FrameCfg cfg, const StereoCaps caps) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int32_t s_part[THREADS / 32 + 1];
    __shared__ int s_count, s_run;
    constexpr int W = THREADS / 32;
    // the jobs of a frame sit in one record (plm_frames_api.inl FrameJobs): job_stride bytes from one frame to the next
    const StereoJob sj = *reinterpret_cast<const StereoJob *>(reinterpret_cast<const char *>(jobs) + blockIdx.x * job_stride);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_l = sj.n_l, n_r = sj.n_r;
    const bool lines = sj.is_lines != 0;
    const int n_cells = cfg.grid_rows * cfg.grid_cols;
    // StereoFrame::matchStereoPoints / Lines return before anything happens when a side is empty
    // (stereoFrame.cpp:137-138, :326-327): no matches, nothing kept.
    if (n_l <= 0 || n_r <= 0) {
        for (int i = tid; i < n_l; i += THREADS) sj.m12[i] = -1;
        if (tid == 0) {
            sj.counts[0] = 0;
            sj.counts[1] = 0;
        }
        return;
    }

    unsigned char *p = smem_raw;
    unsigned char *scratch = p;
    {
        const size_t chunk = grid_align16(static_cast<size_t>(W) * caps.cap_r * 2) + grid_align16(static_cast<size_t>(caps.cap_r) * 4);
        const size_t pairs = pairlist_smem(caps.cap_pairs, caps.cap_l, caps.cap_r);
        p += chunk > pairs ? chunk : pairs;
    }
    uint16_t *wmin = reinterpret_cast<uint16_t *>(scratch);
    uint32_t *m21key = reinterpret_cast<uint32_t *>(scratch + grid_align16(static_cast<size_t>(W) * caps.cap_r * 2));
    int32_t *cs = reinterpret_cast<int32_t *>(p); p += grid_align16(static_cast<size_t>(n_cells + 1) * 4);
    int32_t *ci = reinterpret_cast<int32_t *>(p); p += grid_align16(static_cast<size_t>(caps.cap_items) * 4);
    uint4 *sd_r = reinterpret_cast<uint4 *>(p); p += static_cast<size_t>(caps.cap_r) * 32;
    int32_t *coords = reinterpret_cast<int32_t *>(p); p += grid_align16(static_cast<size_t>(caps.cap_l) * (lines ? 16 : 8));
    int32_t *m12s = reinterpret_cast<int32_t *>(p); p += grid_align16(static_cast<size_t>(caps.cap_l) * 4);
    double *dirs = reinterpret_cast<double *>(p);

    // ---- stage + initialise ----------------------------------------------------------------------------
    stage_bytes(reinterpret_cast<unsigned char *>(sd_r), sj.d_r, static_cast<size_t>(n_r) * 32);
    for (int i = tid; i <= n_cells; i += THREADS) cs[i] = 0;
    for (int i = tid; i < n_l; i += THREADS) m12s[i] = -1; // matches_12 is a fresh vector (:156, :355)
    if (tid == 0) {
        s_count = 0;
        s_run = 0;
    }
    // query cell coordinates: pair<double,double> -> pair<int,int> truncation (:140-143, :329-333)
    if (!lines) {
        const float2 *kl = reinterpret_cast<const float2 *>(sj.geo_l);
        for (int i = tid; i < n_l; i += THREADS) {
            const float2 k = kl[i];
            coords[2 * i] = static_cast<int>(__dmul_rn(static_cast<double>(k.x), cfg.inv_w));
            coords[2 * i + 1] = static_cast<int>(__dmul_rn(static_cast<double>(k.y), cfg.inv_h));
        }
    } else {
        const float4 *ll = reinterpret_cast<const float4 *>(sj.geo_l);
        for (int i = tid; i < n_l; i += THREADS) {
            const float4 k = ll[i];
            coords[4 * i] = static_cast<int>(__dmul_rn(static_cast<double>(k.x), cfg.inv_w));
            coords[4 * i + 1] = static_cast<int>(__dmul_rn(static_cast<double>(k.y), cfg.inv_h));
            coords[4 * i + 2] = static_cast<int>(__dmul_rn(static_cast<double>(k.z), cfg.inv_w));
            coords[4 * i + 3] = static_cast<int>(__dmul_rn(static_cast<double>(k.w), cfg.inv_h));
        }
    }
    __syncthreads();

    // ---- bucket grid of the right features (stereoFrame.cpp:146-150, :336-349) ---------------------------
    // counting sort in shared memory: count -> inclusive scan (cell ends) -> fill by decrementing the ends,
    // which leaves cs[c] = start of cell c and cs[n_cells] = number of items.  The order inside a bucket is
    // arbitrary; matchGrid's result does not depend on it (SURVEY 8a note 1).
    const int walk_cap = cfg.grid_rows + cfg.grid_cols + 4;
    auto on_grid = [&](int x, int y) { return x >= 0 && x < cfg.grid_cols && y >= 0 && y < cfg.grid_rows; };
    auto right_cells = [&](int j, auto &&f) {
        if (!lines) {
            const float2 k = reinterpret_cast<const float2 *>(sj.geo_r)[j];
            // GridStructure::at(int, int) called with doubles: truncation, off-grid -> sink list
            const int x = static_cast<int>(__dmul_rn(static_cast<double>(k.x), cfg.inv_w));
            const int y = static_cast<int>(__dmul_rn(static_cast<double>(k.y), cfg.inv_h));
            if (on_grid(x, y)) f(x * cfg.grid_rows + y);
        } else {
            const float4 k = reinterpret_cast<const float4 *>(sj.geo_r)[j];
            line_walk(__dmul_rn(static_cast<double>(k.x), cfg.inv_w), __dmul_rn(static_cast<double>(k.y), cfg.inv_h),
                      __dmul_rn(static_cast<double>(k.z), cfg.inv_w), __dmul_rn(static_cast<double>(k.w), cfg.inv_h),
                      walk_cap, [&](int x, int y) {
                          if (on_grid(x, y)) f(x * cfg.grid_rows + y);
                      });
        }
    };
    for (int j = tid; j < n_r; j += THREADS) {
        right_cells(j, [&](int c) { atomicAdd(&cs[c], 1); });
        if (lines) {
            // directions (:342-344): float subtraction, * double, then matching.h:43-48 normalize
            const float4 k = reinterpret_cast<const float4 *>(sj.geo_r)[j];
            const double vx = __dmul_rn(static_cast<double>(__fsub_rn(k.z, k.x)), cfg.inv_w);
            const double vy = __dmul_rn(static_cast<double>(__fsub_rn(k.w, k.y)), cfg.inv_h);
            const double mag = __dsqrt_rn(__dadd_rn(__dmul_rn(vx, vx), __dmul_rn(vy, vy)));
            dirs[2 * j] = __ddiv_rn(vx, mag);
            dirs[2 * j + 1] = __ddiv_rn(vy, mag);
        }
    }
    __syncthreads();
    block_inclusive_scan(cs, n_cells, s_part);
    if (tid == 0) cs[n_cells] = cs[n_cells - 1];
    __syncthreads();
    for (int j = tid; j < n_r; j += THREADS)
        right_cells(j, [&](int c) {
            const int slot = atomicSub(&cs[c], 1) - 1;
            if (slot < caps.cap_items) ci[slot] = j;
        });
    __syncthreads();

    // ---- matchGrid on the shared-memory grid (matching.cpp:111-258; phases of plm_grid.cuh) --------------
    GridJob job;
    job.coords = coords;
    job.d1 = sj.d_l;
    job.cell_start = cs;
    job.cell_items = ci;
    job.d2 = sd_r;
    job.dirs2 = dirs;
    job.m12 = m12s;
    job.count = nullptr;
    job.n1 = n_l;
    job.n2 = n_r;
    job.is_lines = lines ? 1 : 0;
    job.win[0] = cfg.matching_s_ws; // w.width = (matchingSWs, 0), w.height = (0, 0)  (:152-154, :351-353)
    job.win[1] = job.win[2] = job.win[3] = 0;
    job.i1_base = 0;
    job.q_row_base = 0;
    GridParams gp;
    gp.grid_rows = cfg.grid_rows;
    gp.grid_cols = cfg.grid_cols;
    gp.best_lr = cfg.best_lr;
    gp.ratio = cfg.ratio;
    gp.line_sim_th = cfg.line_sim_th;

    const PairArrays pa = pairlist_carve(scratch, caps.cap_pairs, caps.cap_l, caps.cap_r);
    if (!pairlist_match(job, gp, pa, s_part, &s_count)) {
        // too many candidate slots for the pair list (features piled up in a few cells): chunk phases
        __syncthreads();
        for (int i = tid; i < W * caps.cap_r; i += THREADS) wmin[i] = D_INF;
        for (int i = tid; i < n_r; i += THREADS) m21key[i] = KEY32_ABSENT;
        __syncthreads();
        const int rpw = (n_l + W - 1) / W;
        const int row0 = min(n_l, warp * rpw), row1 = min(n_l, row0 + rpw);
        uint16_t *mine = wmin + static_cast<size_t>(warp) * caps.cap_r;
        if (gp.best_lr) {
            chunk_minima(job, gp, row0, row1, mine, lane);
            __syncthreads();
            for (int i2 = tid; i2 < n_r; i2 += THREADS) {
                uint16_t run = D_INF;
                for (int w = 0; w < W; ++w) {
                    const uint16_t t = wmin[static_cast<size_t>(w) * caps.cap_r + i2];
                    wmin[static_cast<size_t>(w) * caps.cap_r + i2] = run;
                    run = min(run, t);
                }
            }
            __syncthreads();
        }
        const int acc = chunk_match(job, gp, row0, row1, mine, lane, [&](int i2, int d, int i1) {
            atomicMin(&m21key[i2], (static_cast<uint32_t>(d) << GRID_KEY_BITS) | static_cast<uint32_t>(i1));
        });
        if (lane == 0 && acc) atomicAdd(&s_count, acc);
        __syncthreads();
        if (gp.best_lr) {
            int culled = 0;
            for (int i1 = tid; i1 < n_l; i1 += THREADS) {
                const int32_t i2 = m12s[i1];
                if (i2 >= 0) {
                    const uint32_t k = m21key[i2];
                    const int back = (k == KEY32_ABSENT) ? -1 : static_cast<int>(k & ((1u << GRID_KEY_BITS) - 1));
                    if (back != i1) {
                        m12s[i1] = -1;
                        ++culled;
                    }
                }
            }
            if (culled) atomicSub(&s_count, culled);
            __syncthreads();
        }
    }

    // ---- geometry gates, compaction, back-projection (stereoFrame.cpp:160-183, :359-408) ----------------
    for (int base = 0; base < n_l; base += THREADS) {
        const int i1 = base + tid;
        bool kept = false;
        double disp_s = 0.0, disp_e = 0.0;
        int i2 = -1;
        if (i1 < n_l) {
            i2 = m12s[i1];
            sj.m12[i1] = i2;
            if (i2 >= 0) {
                if (!lines) {
                    const float2 l = reinterpret_cast<const float2 *>(sj.geo_l)[i1];
                    const float2 r = reinterpret_cast<const float2 *>(sj.geo_r)[i2];
                    kept = stereo_point_gate(l, r, cfg.max_dist_epip, cfg.min_disp, disp_s);
                } else {
                    const float4 l = reinterpret_cast<const float4 *>(sj.geo_l)[i1];
                    const float4 r = reinterpret_cast<const float4 *>(sj.geo_r)[i2];
                    kept = stereo_line_gate(l, r, cfg.min_disp, cfg.line_horiz_th, cfg.stereo_overlap_th,
                                            cfg.ls_min_disp_ratio, disp_s, disp_e);
                }
            }
        }
        const unsigned msk = __ballot_sync(0xFFFFFFFFu, kept);
        if (lane == 0) s_part[warp] = __popc(msk);
        __syncthreads();
        int before = s_run;
        for (int w = 0; w < warp; ++w) before += s_part[w];
        const int slot = before + __popc(msk & ((1u << lane) - 1u));
        if (kept) {
            sj.kept_i1[slot] = i1;
            sj.cdesc[2 * slot] = __ldg(sj.d_l + 2 * i1);
            sj.cdesc[2 * slot + 1] = __ldg(sj.d_l + 2 * i1 + 1);
            if (!lines) {
                const float2 l = reinterpret_cast<const float2 *>(sj.geo_l)[i1];
                sj.o0[slot] = disp_s;
                back_projection(cfg, static_cast<double>(l.x), static_cast<double>(l.y), disp_s, sj.o1 + 3 * slot);
            } else {
                const float4 l = reinterpret_cast<const float4 *>(sj.geo_l)[i1];
                const double x1 = l.x, y1 = l.y, x2 = l.z, y2 = l.w;
                sj.o0[2 * slot] = disp_s;
                sj.o0[2 * slot + 1] = disp_e;
                back_projection(cfg, x1, y1, disp_s, sj.o1 + 3 * slot);
                back_projection(cfg, x2, y2, disp_e, sj.o2 + 3 * slot);
                // le_l = sp_l.cross(ep_l) / sqrt(le0^2 + le1^2) with homogeneous endpoints (:366-368)
                const double c0 = __dsub_rn(y1, y2), c1 = __dsub_rn(x2, x1);
                const double c2 = __dsub_rn(__dmul_rn(x1, y2), __dmul_rn(y1, x2));
                const double nrm = __dsqrt_rn(__dadd_rn(__dmul_rn(c0, c0), __dmul_rn(c1, c1)));
                sj.o3[3 * slot] = __ddiv_rn(c0, nrm);
                sj.o3[3 * slot + 1] = __ddiv_rn(c1, nrm);
                sj.o3[3 * slot + 2] = __ddiv_rn(c2, nrm);
            }
        }
        __syncthreads();
        if (tid == 0) {
            int tot = 0;
            for (int w = 0; w < W; ++w) tot += s_part[w];
            s_run += tot;
        }
        __syncthreads();
    }
    if (tid == 0) {
        sj.counts[0] = s_count;
        sj.counts[1] = s_run;
    }
}

// ---- frame-to-frame matching on the compacted descriptors ------------------------------------------------
struct F2FJob {
    const uint4 *d1, *d2;           // compacted left descriptors of the previous / current frame
    const int32_t *n1_ptr, *n2_ptr; // their kept counts (device memory, written by the stereo stage)
    int32_t *m12;                   // out: capacity cap1, entries [0, n1) are written
    int32_t *count;                 // out: StVO::match return value; INT32_MIN where the reference is UB
    int32_t cap1, cap2;
    float nnr;
    int32_t pad_;
};

constexpr uint32_t F2F_INVALID = 0x80000000u; // key bit of lanes without a row; such keys read as absent
constexpr int F2F_KEY_BITS = 22;

__host__ __device__ inline size_t f2f_smem(int cap1, int cap2) {
    return static_cast<size_t>(cap2) * 32 + 2 * grid_align16(static_cast<size_t>(cap2) * 4) +
           grid_align16(static_cast<size_t>(cap1) * 4);
}

// 128-bit shared-memory load the compiler may not hoist or cache (other warps update the words).
__device__ __forceinline__ uint4 lds_volatile_v4(const uint32_t *p) {
    uint4 v;
    const uint32_t a = static_cast<uint32_t>(__cvta_generic_to_shared(p));
    asm volatile("ld.volatile.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
    return v;
}

__device__ __forceinline__ bool nnr_accept_f32(uint32_t k0, uint32_t k1, float nnr) {
    const float d0 = static_cast<float>(static_cast<int>(k0 >> F2F_KEY_BITS));
    const float d1 = static_cast<float>(static_cast<int>(k1 >> F2F_KEY_BITS));
    return d0 < __fmul_rn(d1, nnr); // matching.cpp:54, float arithmetic
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS)
f2f_match_kernel(const F2FJob *__restrict__ jobs, const size_t job_stride, int best_lr) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_count;
    const F2FJob job = *reinterpret_cast<const F2FJob *>(reinterpret_cast<const char *>(jobs) + blockIdx.x * job_stride);
    const int tid = threadIdx.x, lane = tid & 31;
    const int n1 = min(*job.n1_ptr, job.cap1), n2 = min(*job.n2_ptr, job.cap2);
    // matchF2FPoints / Lines return early when either frame has no stereo features
    // (stereoFrameHandler.cpp:164, :187); StVO::match itself needs two rows on the train side(s).
    if (n1 <= 0 || n2 <= 0) {
        if (tid == 0) *job.count = 0;
        return;
    }
    if (n2 < 2 || (best_lr && n1 < 2)) {
        for (int i = tid; i < n1; i += THREADS) job.m12[i] = -1;
        if (tid == 0) *job.count = INT32_MIN;
        return;
    }
    unsigned char *p = smem_raw;
    uint4 *sd2 = reinterpret_cast<uint4 *>(p); p += static_cast<size_t>(job.cap2) * 32;
    uint32_t *cbest = reinterpret_cast<uint32_t *>(p); p += grid_align16(static_cast<size_t>(job.cap2) * 4);
    uint32_t *csecond = reinterpret_cast<uint32_t *>(p); p += grid_align16(static_cast<size_t>(job.cap2) * 4);
    int32_t *m12s = reinterpret_cast<int32_t *>(p);
    stage_bytes(reinterpret_cast<unsigned char *>(sd2), job.d2, static_cast<size_t>(n2) * 32);
    const int n2_pad = (n2 + 3) & ~3;
    for (int i = tid; i < n2_pad; i += THREADS) {
        cbest[i] = KEY32_ABSENT;
        csecond[i] = KEY32_ABSENT;
    }
    if (tid == 0) s_count = 0;
    __syncthreads();
    // 13-LOP3 distance (plm_common.cuh): the staged train rows and every query go through the same GF(2)-linear
    // transform once; the xor of two transformed descriptors already holds the first carry-save level
    for (int r = tid; r < n2; r += THREADS) desc_transform13(sd2[2 * r], sd2[2 * r + 1]);
    __syncthreads();

    int accepted = 0;
    for (int rb = 0; rb < n1; rb += THREADS) {
        if (rb + (tid & ~31) >= n1) continue; // the whole warp is past the last row
        const int i1 = rb + tid;
        const bool valid = i1 < n1;
        Desc a;
        if (valid) {
            a = load_desc(job.d1, i1);
        } else {
            a.lo = make_uint4(0, 0, 0, 0);
            a.hi = a.lo;
        }
        desc_transform13(a.lo, a.hi);
        const uint32_t ck_add = valid ? static_cast<uint32_t>(i1) : (F2F_INVALID | static_cast<uint32_t>(i1));
        uint32_t b0 = KEY32_ABSENT, b1 = KEY32_ABSENT; // row top-2: (d << 22 | i2)
        int j = 0;
        for (; j + 4 <= n2; j += 4) {
            uint32_t ck[4], m0[4];
#pragma unroll
            for (int v = 0; v < 4; ++v) {
                const uint32_t dk = static_cast<uint32_t>(hamming256_t13(a, sd2[2 * (j + v)], sd2[2 * (j + v) + 1])) << F2F_KEY_BITS;
                top2_insert(b0, b1, dk + static_cast<uint32_t>(j + v));
                ck[v] = dk + ck_add;
            }
            if (best_lr) {
#pragma unroll
                for (int v = 0; v < 4; ++v) m0[v] = __reduce_min_sync(0xFFFFFFFFu, ck[v]);
                // column top-2 (d << 22 | i1): only warps that beat the current second best take the slow path
                // The vote makes the branch warp-uniform even if lanes happened to read different snapshots
                // of the (concurrently shrinking) thresholds; a stale larger value only costs a slow path.
                const uint4 sec = lds_volatile_v4(csecond + j);
                if (__any_sync(0xFFFFFFFFu, m0[0] < sec.x || m0[1] < sec.y || m0[2] < sec.z || m0[3] < sec.w)) {
#pragma unroll
                    for (int v = 0; v < 4; ++v) {
                        const uint32_t m1 = __reduce_min_sync(0xFFFFFFFFu, ck[v] == m0[v] ? KEY32_ABSENT : ck[v]);
                        if (lane == 0) {
                            const uint32_t old = atomicMin(&cbest[j + v], m0[v]);
                            atomicMin(&csecond[j + v], max(old, m0[v]));
                            atomicMin(&csecond[j + v], m1);
                        }
                    }
                }
            }
        }
        for (; j < n2; ++j) {
            const uint32_t dk = static_cast<uint32_t>(hamming256_t13(a, sd2[2 * j], sd2[2 * j + 1])) << F2F_KEY_BITS;
            top2_insert(b0, b1, dk + static_cast<uint32_t>(j));
            if (best_lr) {
                const uint32_t ck = dk + ck_add;
                const uint32_t m0 = __reduce_min_sync(0xFFFFFFFFu, ck);
                const uint32_t m1 = __reduce_min_sync(0xFFFFFFFFu, ck == m0 ? KEY32_ABSENT : ck);
                if (lane == 0) {
                    const uint32_t old = atomicMin(&cbest[j], m0);
                    atomicMin(&csecond[j], max(old, m0));
                    atomicMin(&csecond[j], m1);
                }
            }
        }
        if (valid) {
            const bool acc = nnr_accept_f32(b0, b1, job.nnr);
            m12s[i1] = acc ? static_cast<int32_t>(b0 & ((1u << F2F_KEY_BITS) - 1)) : -1;
            accepted += acc ? 1 : 0;
        }
    }
    const unsigned am = __ballot_sync(0xFFFFFFFFu, accepted != 0);
    (void)am;
    if (accepted) atomicAdd(&s_count, accepted);
    __syncthreads();
    if (best_lr) {
        // direction 21 acceptance, in place: cbest[j] <- matches_21[j]
        for (int i2 = tid; i2 < n2; i2 += THREADS) {
            const uint32_t k0 = cbest[i2], k1 = csecond[i2];
            int32_t back = -1;
            if (k0 < F2F_INVALID && k1 < F2F_INVALID && nnr_accept_f32(k0, k1, job.nnr))
                back = static_cast<int32_t>(k0 & ((1u << F2F_KEY_BITS) - 1));
            cbest[i2] = static_cast<uint32_t>(back);
        }
        __syncthreads();
        int culled = 0;
        for (int i1 = tid; i1 < n1; i1 += THREADS) {
            const int32_t i2 = m12s[i1];
            if (i2 >= 0 && static_cast<int32_t>(cbest[i2]) != i1) {
                m12s[i1] = -1;
                ++culled;
            }
        }
        if (culled) atomicSub(&s_count, culled);
        __syncthreads();
    }
    for (int i1 = tid; i1 < n1; i1 += THREADS) job.m12[i1] = m12s[i1];
    if (tid == 0) *job.count = s_count;
}

} // namespace plm
