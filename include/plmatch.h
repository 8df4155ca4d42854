/*
 * plmatch.h -- C ABI of the B200-native descriptor-matching path of PL-inertial-slam.
 *
 * This is the drop-in boundary (SURVEY.md section 8b): every entry point below replaces one
 * function of the reference's matching layer (paths relative to the reference checkout):
 *
 *   plm_hamming256          StVO::distance                 stvo-pl/src/matching.cpp:93-109
 *   plm_knn2                cv::BFMatcher::knnMatch(k=2)   call site stvo-pl/src/matching.cpp:47-48
 *   plm_match_nnr           StVO::matchNNR                 stvo-pl/src/matching.cpp:41-61
 *   plm_match               StVO::match                    stvo-pl/src/matching.cpp:63-91
 *   plm_match_grid_points   StVO::matchGrid (points)       stvo-pl/src/matching.cpp:111-177
 *   plm_match_grid_lines    StVO::matchGrid (lines)        stvo-pl/src/matching.cpp:179-258
 *   plm_stereo_filter_points  gates of matchStereoPoints   stvo-pl/src/stereoFrame.cpp:162-171
 *   plm_stereo_filter_lines   gates of matchStereoLines    stvo-pl/src/stereoFrame.cpp:359-385,
 *                             filterLineSegmentDisparity :416-426, lineSegmentOverlapStereo :484-519
 *   plm_line_pair_filter    overlap / angle filter for matched line pairs: StereoFrame::lineSegmentOverlap
 *                           stvo-pl/src/stereoFrame.cpp:521-627 + the direction test of matching.cpp:221
 *   plm_batch_*             the per-frame loop             app/plslam_dataset.cpp:114-172
 *   plm_frames_*            StereoFrame::matchStereoPoints/Lines + StereoFrameHandler::matchF2FPoints/Lines
 *                           on the device (stereoFrame.cpp:131-184,320-409; stereoFrameHandler.cpp:158-207)
 *   plm_db_* / plm_dev_*    keyframe / local-map database  src/mapHandler.cpp:583-803, 3301-3409
 *   plm_voc_* / plm_bow_*   DBoW2 vocabulary transform + L1 score behind MapHandler::insertKFBowVectorP/L/PL
 *                           src/mapHandler.cpp:3116-3237; 3rdparty/DBoW2/include/DBoW2/TemplatedVocabulary.h:1045-1238,
 *                           3rdparty/DBoW2/src/DBoW2/{BowVector.cpp:31-81, ScoringObject.cpp:25-69, FORB.cpp:78-100}
 *   plm_loopdb_*            loop-closure keyframe database: insertKFBowVectorP/L/PL and isLoopClosure's matching on
 *                           device-resident keyframes   src/mapHandler.cpp:3116-3237, 3325-3378
 *   plm_med_desc / plm_dev_med_desc   PLSLAM::MapPoint / MapLine::updateAverageDescDir (the producer of the
 *                           map's med_desc rows)           src/mapFeatures.cpp:51-93, 121-163
 *   plm_localmap_*          resident local map: map_points / map_lines updated in place and matchMap2KFPoints / Lines
 *                           from the resident rows         src/mapHandler.cpp:583-803, src/mapFeatures.cpp
 *
 * The C++ replacement of stvo-pl/src/matching.cpp that keeps the StVO:: signatures and calls this
 * ABI is pl_inertial_slam_b200/csrc/stvo_matching_gpu.cpp (see INTEGRATION.md).
 *
 * Conventions
 *  - Descriptors are 256-bit (32-byte) rows, `step` bytes apart (cv::Mat::step); step >= 32.
 *  - m12_inout is IN/OUT like the reference's std::vector<int>& matches_12 after
 *    resize(n1, -1): the library writes accepted rows and cross-check culls only, never resets.
 *    Entries >= 0 on input ("stale" matches of the fallback call sites, mapHandler.cpp:325-329)
 *    must be < n2.
 *  - Every function returns a status (PLM_OK or < 0); the reference's int return value (match
 *    count; may be off or negative in the stale-fallback quirk) comes back through n_matches.
 *  - No exception crosses this boundary and there is NO CPU fallback: without a usable CUDA device
 *    every compute entry point returns PLM_E_CUDA.
 *  - A plm_ctx owns one CUDA stream, device scratch and pinned staging.  It may be used by one
 *    host thread at a time; pass NULL to use a lazily created per-thread default context
 *    (re-entrant from any number of host threads, SURVEY 3.4).  A call makes the context's device current for the
 *    calling thread and leaves it current (like cudaSetDevice); callers that run their own CUDA code on another
 *    device on the same thread must switch back themselves.
 *  - Packed top-2 keys: key = (uint64)distance << 32 | train_index, UINT64_MAX when absent;
 *    unsigned min over keys == the reference's lowest-index tie-breaking.
 */
#ifndef PLMATCH_H_
#define PLMATCH_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PLM_VERSION 100

#define PLM_OK             0
#define PLM_E_INVALID     -1 /* null pointer, negative size, step < 32, misaligned device pointer  */
#define PLM_E_SIZE        -2 /* size mismatch: "[matchNNR] Different size for matches and descriptors!",
                                "[matchGrid] Each point/line needs a corresponding descriptor!"      */
#define PLM_E_TRAIN       -3 /* empty train set with a non-empty query: the reference throws
                                "[matchNNR] Different size for matches and descriptors!" (matching.cpp:50-51) */
#define PLM_E_GRID        -4 /* "[GridStructure] invalid dimension" or malformed CSR                  */
#define PLM_E_RATIO       -5 /* matchGrid ratio > 1: the reference's result then depends on
                                unordered_set iteration order                                        */
#define PLM_E_CUDA        -6 /* CUDA runtime failure (see plm_last_error)                            */
#define PLM_E_NOMEM       -7
#define PLM_E_UNSUPPORTED -8 /* size outside what the kernels support (documented per function)      */
#define PLM_E_PEER        -9 /* a device did not arrive at a peer-memory exchange within the spin limit  */

typedef struct plm_ctx plm_ctx;
typedef struct plm_db plm_db;

#define PLM_KEY_ABSENT UINT64_MAX

int plm_version(void);
const char *plm_status_string(int status);
/* Message of the last failing call on this thread (CUDA error string included). */
const char *plm_last_error(void);
int plm_device_count(int *count);

int plm_ctx_create(int device, plm_ctx **out);
int plm_ctx_destroy(plm_ctx *ctx);
/* cudaStream_t the context launches on. */
void *plm_ctx_stream(plm_ctx *ctx);
/* external != 0: launch on the caller's stream (e.g. torch's current stream; a NULL handle is the
 * legacy default stream); external == 0: return to the context's own stream. */
int plm_ctx_set_stream(plm_ctx *ctx, void *cuda_stream, int external);
int plm_ctx_synchronize(plm_ctx *ctx);
/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
uint64_t plm_ctx_launch_count(plm_ctx *ctx);

/* Per-launch CUDA-event timing of the brute-force slice kernel (the roofline kernel): switch it on,
 * run, then read the summed device time and the number of launches since the last read. */
int plm_ctx_set_profiling(plm_ctx *ctx, int on);
int plm_ctx_read_profile(plm_ctx *ctx, double *knn2_slice_ms, int *n_launches);

/* ---- host-buffer entry points (what the StVO:: wrappers call) -------------------------------- */

/* dist[i] = Hamming(a row i, b row i), i < n.  StVO::distance is the n == 1 case. */
int plm_hamming256(plm_ctx *ctx, const uint8_t *a, size_t step_a, const uint8_t *b, size_t step_b,
                   int n, int32_t *dist);

/* Two nearest train rows per query row as packed keys, top2 = n1 x 2 uint64 (best, second).
 * idx_base is added to the train index (database shards).  n2 >= 0 (absent slots = PLM_KEY_ABSENT). */
int plm_knn2(plm_ctx *ctx, const uint8_t *d1, int n1, size_t step1, const uint8_t *d2, int n2,
             size_t step2, uint64_t idx_base, uint64_t *top2);

/* StVO::matchNNR.  Accept row i iff (float)d0 < (float)d1 * nnr (float arithmetic, as :54).
 * Degenerate sizes: n1 == 0 -> 0 matches (as the reference); n2 == 0 with n1 > 0 -> PLM_E_TRAIN (the reference
 * throws); n2 == 1 -> no row has a second neighbour, none is accepted, m12 stays as it was (the reference reads
 * matches_[idx][1] out of bounds there, :54 -- undefined, but it does not throw). */
int plm_match_nnr(plm_ctx *ctx, const uint8_t *d1, int n1, size_t step1, const uint8_t *d2, int n2,
                  size_t step2, float nnr, int32_t *m12_inout, int *n_matches);

/* StVO::match.  best_lr = Config::bestLRMatches(): both directions + mutual check.  One-row sides follow the rule
 * above per direction (with n1 == 1 no reverse match exists, so the mutual check culls every entry of m12). */
int plm_match(plm_ctx *ctx, const uint8_t *d1, int n1, size_t step1, const uint8_t *d2, int n2,
              size_t step2, float nnr, int best_lr, int32_t *m12_inout, int *n_matches);

/* Frame session: the matcher calls of ONE frame as one host <-> device round trip.  Between plm_frame_begin and
 * plm_frame_end the plm_match_nnr / plm_match / plm_match_grid_points / plm_match_grid_lines calls made on this context
 * (NULL = the calling thread's default context) validate their arguments and are RECORDED; plm_frame_end executes them.
 * When every recorded call is frame-sized (matchGrid: n1 <= 2048 and a train side whose work arrays fit shared memory;
 * match: n1, n2 <= 2048; at most 12 calls) the whole session is ONE kernel (frame_fused_kernel, csrc/plm_frame_fused.cuh):
 * all inputs packed into one pinned block, one host -> device copy, one launch -- a cluster of 8 CTAs per matchGrid call,
 * independent CTAs per match call, the job table in the kernel parameters -- and the kernel stores every m12_inout /
 * n_matches straight into the pinned block (no device -> host copy), one synchronisation.  Otherwise each call runs its
 * own copy-in / kernels / copy-out on one of four streams, one synchronisation at the end (option "frame_fused" = 0
 * forces this form).  The recorded pointers (descriptors, grids, m12_inout, n_matches) must stay valid until
 * plm_frame_end returns; results are only defined after it.  This is the stereo (points || lines) + temporal
 * (points || lines) structure of StereoFrame::extractStereoFeatures / StereoFrameHandler::f2fTracking
 * (stereoFrame.cpp:75-76, stereoFrameHandler.cpp:142-143) without host threads.  A stand-alone frame-sized call takes
 * the same kernel as a session of one call.  C++ hosts: StVO::GpuFrame (csrc/stvo_gpu_frame.h). */
int plm_frame_begin(plm_ctx *ctx);
int plm_frame_end(plm_ctx *ctx);
/* 1 while a frame session is open on the context (NULL = the calling thread's default context), else 0. */
int plm_frame_active(plm_ctx *ctx);

/* StVO::matchGrid, points.  xy = n1 x (x, y) grid-cell coordinates of the queries.
 * Grid = CSR of GridStructure over the train features: cell (x, y) has id x * grid_rows + y,
 * cell_start has grid_rows * grid_cols + 1 entries, cell_items the bucket contents.
 * win = { width.first, width.second, height.first, height.second } of GridWindow.
 * ratio = Config::minRatio12P() (double arithmetic, :160); must be <= 1.
 * Supported: n2 <= 32768. */
int plm_match_grid_points(plm_ctx *ctx, const int32_t *xy, const uint8_t *d1, int n1, size_t step1,
                          const int32_t *cell_start, const int32_t *cell_items, int grid_rows,
                          int grid_cols, const uint8_t *d2, int n2, size_t step2,
                          const int32_t win[4], double ratio, int best_lr, int32_t *m12_inout,
                          int *n_matches);

/* StVO::matchGrid, lines.  xyxy = n1 x (start x, start y, end x, end y) cell coordinates;
 * dirs2 = n2 x (dx, dy) unit directions of the train lines; a candidate is skipped when
 * fabs(dot(normalize(end - start), dirs2[i2])) < line_sim_th (NaN passes, :221).
 * ratio = Config::minRatio12P() -- the reference uses the POINT ratio here too (:241). */
int plm_match_grid_lines(plm_ctx *ctx, const int32_t *xyxy, const uint8_t *d1, int n1, size_t step1,
                         const int32_t *cell_start, const int32_t *cell_items, int grid_rows,
                         int grid_cols, const uint8_t *d2, int n2, size_t step2, const double *dirs2,
                         double line_sim_th, const int32_t win[4], double ratio, int best_lr,
                         int32_t *m12_inout, int *n_matches);

/* Epipolar / minimum-disparity gate of matchStereoPoints.  kp_l = n1 x (x, y) float32 pixels,
 * kp_r = n2 x 2.  keep[i1] = 1 iff m12[i1] >= 0 passes; disp[i1] = x_l - x_r of kept rows. */
int plm_stereo_filter_points(plm_ctx *ctx, const float *kp_l, int n1, const float *kp_r, int n2,
                             const int32_t *m12, double max_dist_epip, double min_disp,
                             uint8_t *keep, double *disp, int *n_kept);

/* Overlap / disparity-ratio / horizontal-line gate of matchStereoLines.  ln_* = n x (sx, sy, ex,
 * ey) float32 pixels.  disp_se = n1 x (disp_s, disp_e). */
int plm_stereo_filter_lines(plm_ctx *ctx, const float *ln_l, int n1, const float *ln_r, int n2,
                            const int32_t *m12, double min_disp, double line_horiz_th,
                            double stereo_overlap_th, double ls_min_disp_ratio, uint8_t *keep,
                            double *disp_se, int *n_kept);

/* Opt-in geometric filter for matched line pairs (BASELINE config 2 "NNR line matching with overlap/angle filter").
 * The fork's temporal line matcher applies none (stereoFrameHandler.cpp:182-207); this evaluates the reference's own
 * two tests per matched pair (i1, m12[i1]):
 *   overlap = StereoFrame::lineSegmentOverlap(observed = ln1[i1], other = ln2[m12[i1]])   stereoFrame.cpp:521-627
 *   sim     = |dot(normalize(e1 - s1), normalize(e2 - s2))|   matching.h:39-48, the test of matching.cpp:221
 * keep[i1] = overlap > overlap_th && !(sim < line_sim_th)  (a NaN similarity passes, as in matchGrid); unmatched rows
 * get keep 0, overlap 0, sim 0.  m12 is not modified.  ln1 / ln2 are n x (sx, sy, ex, ey) float pixels. */
int plm_line_pair_filter(plm_ctx *ctx, const float *ln1, int n1, const float *ln2, int n2, const int32_t *m12,
                         double overlap_th, double line_sim_th, uint8_t *keep, double *overlap, double *sim, int *n_kept);

/* ---- batched replay (one launch per stage over a frame arena) -------------------------------- */

/* One brute-force job: rows [off1, off1+n1) x rows [off2, off2+n2) of the descriptor arena;
 * results land at m12_arena[off_m .. off_m + n1). */
typedef struct plm_pair_job {
    int64_t off1, off2, off_m;
    int32_t n1, n2;
} plm_pair_job;

/* One grid job (points when is_lines == 0).  Offsets index the arenas passed to
 * plm_batch_set_match_grid: coords (int32 elements), descriptor rows, CSR arenas, dirs2 (doubles).
 * Every job must be frame-sized: n1 <= 4096 and n2 <= 32768. */
typedef struct plm_grid_job {
    int64_t off_coords; /* into coords arena, int32 units (2 or 4 per query)        */
    int64_t off1, off2; /* descriptor arena rows                                     */
    int64_t off_cell_start, off_cell_items;
    int64_t off_dirs2;  /* into dirs2 arena, double units (lines only)               */
    int64_t off_m;
    int32_t n1, n2, is_lines, pad_;
    int32_t win[4];
} plm_grid_job;

/* A batch owns the device copy of its arenas and job tables, so a replay can be prepared once
 * (set_*), run many times (run: kernels only, enqueued on the context's stream, no host sync) and
 * read back (fetch: device -> host + sync).  run() first restores the uploaded m12 arena, so every
 * run sees the same IN values. */
typedef struct plm_batch plm_batch;
int plm_batch_create(plm_ctx *ctx, plm_batch **out);
int plm_batch_destroy(plm_batch *b);

/* StVO::match for every job; counts[j] = the reference's return value for job j.
 * arena = n_rows x 32 bytes, contiguous.  Jobs with n2 < 2 (or n1 < 2 with best_lr) get
 * counts[j] = INT32_MIN and are skipped (the reference would be UB / throw).
 * m12_arena (n_m entries) is the IN value of every job's match vector. */
int plm_batch_set_match(plm_batch *b, const uint8_t *arena, int64_t n_rows, const plm_pair_job *jobs,
                        int n_jobs, float nnr, int best_lr, const int32_t *m12_arena, int64_t n_m);

/* Same with the descriptor arena ALREADY RESIDENT on the context's device (used in place, never copied; it must stay
 * valid and its rows may be rewritten between runs): the per-keyframe-pair form of loop-closure matching -- StVO::match
 * of one query keyframe against every keyframe of a resident database (isLoopClosure, mapHandler.cpp:3325-3378, at
 * scale; SURVEY 8d "Mode A").  Prepare once with the query rows in a fixed slot of the arena, then per query: rewrite
 * the slot, plm_batch_run, plm_batch_fetch.  m12_arena may be NULL: every match vector then starts at -1.
 * When every live job shares one query range (off1, n1) -- this form -- option "batch_umma" = 1 makes both directions
 * of every pair come from one int8 tensor-core product per 256 query rows x 128 train rows (knn2_umma_pairs_kernel);
 * results are identical either way, and so is the number of launches per run. */
int plm_batch_set_match_dev(plm_batch *b, const void *arena_dev, int64_t n_rows, const plm_pair_job *jobs,
                            int n_jobs, float nnr, int best_lr, const int32_t *m12_arena, int64_t n_m);

/* StVO::matchGrid (points or lines per job) for every job, one CTA per job. */
int plm_batch_set_match_grid(plm_batch *b, const uint8_t *arena, int64_t n_rows, const int32_t *coords,
                             int64_t n_coords, const int32_t *cell_start, int64_t n_cell_start,
                             const int32_t *cell_items, int64_t n_cell_items, const double *dirs2,
                             int64_t n_dirs2, int grid_rows, int grid_cols, const plm_grid_job *jobs,
                             int n_jobs, double ratio, double line_sim_th, int best_lr,
                             const int32_t *m12_arena, int64_t n_m);

int plm_batch_run(plm_batch *b);
int plm_batch_fetch(plm_batch *b, int32_t *m12_arena, int32_t *counts);
/* Bytes the last set_* call copied host -> device / fetch copies device -> host. */
int64_t plm_batch_h2d_bytes(const plm_batch *b);
int64_t plm_batch_d2h_bytes(const plm_batch *b);

/* ---- device-resident stereo-frame pipeline (config 3; SURVEY 8f-1 and 8f-4) --------------------- */
/* The per-frame work of the reference's front end from raw features to tracked features, without a
 * host round trip between the stages:
 *   stereo stage    StereoFrame::matchStereoPoints / matchStereoLines   stvo-pl/src/stereoFrame.cpp:131-184,
 *                   :320-409 -- bucket grid of the right features (GridStructure::at; getLineCoords /
 *                   LineIterator for lines, stvo-pl/src/lineIterator.cpp:34-77), matchGrid with the window
 *                   (matchingSWs, 0) x (0, 0), the geometry gates, compaction of pdesc_l / ldesc_l to the kept
 *                   rows and PinholeStereoCamera::backProjection (pinholeStereoCamera.cpp:229-237)
 *   temporal stage  StereoFrameHandler::matchF2FPoints / matchF2FLines   stvo-pl/src/stereoFrameHandler.cpp:
 *                   158-207 -- StVO::match(prev, curr) on the COMPACTED left descriptors; frame f is matched
 *                   against frame f - 1 of the same upload.
 * Arenas: descriptors n_rows x 32 bytes; keypoints (x, y) float32 pixels (cv::KeyPoint::pt); line segments
 * (startPointX, startPointY, endPointX, endPointY) float32 pixels (cv::line_descriptor::KeyLine). */
typedef struct plm_frame_rec {
    int64_t desc_pl, desc_pr, desc_ll, desc_lr; /* first descriptor-arena row of left/right points, left/right lines */
    int64_t kp_l, kp_r;                         /* first keypoint of the left / right image in the keypoint arena      */
    int64_t ln_l, ln_r;                         /* first segment of the left / right image in the line arena           */
    int32_t n_pl, n_pr, n_ll, n_lr;
} plm_frame_rec;

typedef struct plm_frame_config {
    double inv_width, inv_height; /* GRID_COLS / image cols, GRID_ROWS / image rows (stereoFrame.cpp:47-48)       */
    int32_t grid_rows, grid_cols; /* GRID_ROWS 48, GRID_COLS 64 (stereoFrame.h:51-52)                              */
    int32_t matching_s_ws;        /* Config::matchingSWs()                                                          */
    int32_t best_lr;              /* Config::bestLRMatches()                                                        */
    double min_ratio_12p;         /* matchGrid ratio (points AND lines, matching.cpp:160,241) and the f2f point nnr */
    double min_ratio_12l;         /* f2f line nnr (narrowed to float like the reference's call)                     */
    double line_sim_th, max_dist_epip, min_disp, line_horiz_th, stereo_overlap_th, ls_min_disp_ratio;
    double cam_b, cam_fx, cam_cx, cam_cy; /* PinholeStereoCamera baseline / focal length / principal point         */
} plm_frame_config;

/* Host output buffers; any pointer may be NULL (not copied).  "Left point slots" are the left keypoints of
 * all frames concatenated in frame order (frame f starts at sum of n_pl over earlier frames, NP slots in
 * total); "left line slots" likewise (NL).  Per frame, the first kept rows of a slot range are valid.
 *   stereo_m12_*  matchGrid vector of the stereo stage (index into the frame's right set or -1)
 *   kept_*        kept slot k -> left feature index i1 (the order of stereo_pt / stereo_ls and of the
 *                 compacted descriptors)
 *   pt_disp, pt_P          PointFeature::disp and ::P per kept point (P = 3 doubles)
 *   ls_disp, ls_sP, ls_eP, ls_le   LineFeature::sdisp/edisp (2 doubles), ::sP, ::eP, ::le (3 doubles each)
 *   f2f_m12_*     slot range of frame f holds StVO::match(frame f, frame f + 1): kept index of frame f ->
 *                 kept index of frame f + 1 or -1 (the last frame's range is not written)
 *   counts        n_frames x 6: [0] stereo point matches (matchGrid return), [1] kept points, [2] stereo
 *                 line matches, [3] kept lines, [4] / [5] return value of the f2f point / line match of
 *                 (frame f - 1, frame f); 0 for frame 0 and when either side has no stereo features
 *                 (stereoFrameHandler.cpp:164,187), INT32_MIN where StVO::match would be undefined
 *                 (fewer than two descriptors on a train side). */
typedef struct plm_frames_out {
    int32_t *stereo_m12_p, *stereo_m12_l;
    int32_t *kept_p, *kept_l;
    double *pt_disp, *pt_P;
    double *ls_disp, *ls_sP, *ls_eP, *ls_le;
    int32_t *f2f_m12_p, *f2f_m12_l;
    int32_t *counts;
} plm_frames_out;

typedef struct plm_frames plm_frames;
int plm_frames_create(plm_ctx *ctx, plm_frames **out);
int plm_frames_destroy(plm_frames *fr);
/* Copies the arenas to the device and prepares the job tables (one host -> device copy per arena).
 * Supported: per frame n_pl, n_pr <= 4096 and n_ll, n_lr <= 4096; line segments whose Bresenham walk is
 * longer than grid_rows + grid_cols + 2 cells (far off-image coordinates) are rejected. */
int plm_frames_upload(plm_frames *fr, const uint8_t *desc_arena, int64_t n_rows, const float *kp_arena,
                      int64_t n_kp, const float *ln_arena, int64_t n_ln, const plm_frame_rec *frames,
                      int n_frames, const plm_frame_config *cfg);
/* Stereo stage then temporal stage for every uploaded frame, enqueued on the context's stream. */
int plm_frames_run(plm_frames *fr);
/* Device -> host copy of the requested outputs + stream sync. */
int plm_frames_fetch(plm_frames *fr, const plm_frames_out *out);
/* upload + run + fetch as ONE pipelined call: the frames are cut into chunks of at most chunk_frames
 * consecutive frames (<= 0: 256; the first chunks are shorter so that copying starts early) and the chunks
 * flow through three streams -- host -> device copy of chunk k + 1, the
 * four launches of chunk k and the device -> host copy of chunk k - 1 overlap (both copy engines and the SMs
 * busy at once), and the host-side preparation of a chunk overlaps with the device work of the previous ones.
 * Arenas and outputs should be pinned host memory (pageable memory still works, without the overlap).
 * Returns when every requested output is in host memory. */
int plm_frames_process(plm_frames *fr, const uint8_t *desc_arena, int64_t n_rows, const float *kp_arena,
                       int64_t n_kp, const float *ln_arena, int64_t n_ln, const plm_frame_rec *frames,
                       int n_frames, const plm_frame_config *cfg, const plm_frames_out *out, int chunk_frames);
int64_t plm_frames_h2d_bytes(const plm_frames *fr);
int64_t plm_frames_d2h_bytes(const plm_frames *fr);

/* ---- device-resident entry points (descriptor database shards, multi-GPU merge) -------------- */
/* All *_dev pointers are device pointers on the context's device; descriptor rows are contiguous
 * (32-byte step) and 16-byte aligned.  Work is enqueued on the context's stream, no host sync. */

int plm_dev_knn2(plm_ctx *ctx, const void *d1_dev, int n1, const void *d2_dev, int64_t n2,
                 uint64_t idx_base, uint64_t *top2_dev);
/* top2_out[q] = two smallest keys among parts[p][q][0..1], p < n_parts (parts = n_parts x n1 x 2). */
int plm_dev_top2_merge(plm_ctx *ctx, const uint64_t *parts_dev, int n_parts, int n1,
                       uint64_t *top2_out_dev);
/* matchNNR acceptance from packed top-2: m12[q] = idx0 and ++*count where the ratio test passes. */
int plm_dev_nnr_accept(plm_ctx *ctx, const uint64_t *top2_dev, int n1, float nnr,
                       int32_t *m12_dev_inout, int32_t *count_dev);
/* Mutual check (matching.cpp:80-86): cull m12[i1] >= 0 with m21[m12[i1]] != i1, --*count each. */
int plm_dev_cross_check(plm_ctx *ctx, int32_t *m12_dev_inout, int n1, int64_t i1_base,
                        const int32_t *m21_dev, int64_t n2, int32_t *count_dev);

/* Row-sharded matchGrid (config 4: the local map is desc1, sharded over GPUs; SURVEY 8e).  All
 * pointers are device pointers.  The running per-column minimum of the reference spans shards, so
 * the call is split around ONE exchange:
 *   1. plm_dev_grid_colmin   col_min[i2] = min Hamming distance of this shard's candidate pairs
 *                            (uint16, 0xFFFF = none)
 *   -- caller all-gathers col_min and takes, per column, the min over LOWER-ranked shards = seed --
 *   2. plm_dev_grid_match    matches this shard's rows against thresholds that start at seed
 *                            (NULL = none); accepted rows go to m12_inout, *count += accepts and
 *                            m21key[i2] = min over live pairs of (distance << 32 | i1_base + i1)
 *                            (UINT64_MAX = none)
 *   -- caller min-reduces m21key over shards --
 *   3. plm_dev_m21_from_keys + plm_dev_cross_check finish the mutual check on every shard. */
typedef struct plm_dev_grid_args {
    const int32_t *coords;     /* n1 x 2 (points) or n1 x 4 (lines) */
    const void *d1;            /* n1 x 32 bytes */
    const int32_t *cell_start; /* grid_rows * grid_cols + 1 */
    const int32_t *cell_items;
    const void *d2;            /* n2 x 32 bytes */
    const double *dirs2;       /* n2 x 2, lines only */
    int32_t *m12_inout;        /* n1 */
    int32_t *count;            /* 1 */
    int64_t i1_base;           /* global index of this shard's row 0 */
    double ratio, line_sim_th;
    int32_t n1, n2, grid_rows, grid_cols, is_lines, best_lr;
    int32_t win[4];
} plm_dev_grid_args;
int plm_dev_grid_colmin(plm_ctx *ctx, const plm_dev_grid_args *a, uint16_t *col_min_dev);
int plm_dev_grid_match(plm_ctx *ctx, const plm_dev_grid_args *a, const uint16_t *seed_dev, uint64_t *m21key_dev);
int plm_dev_m21_from_keys(plm_ctx *ctx, const uint64_t *m21key_dev, int n2, int32_t *m21_dev);
/* The complete matchGrid (StVO::matchGrid, matching.cpp:111-258) of device-resident rows against one frame on ONE device
 * as a single call: minima pass, scan, match pass, mutual check -- four launches back to back.  fresh != 0: m12_inout
 * is first filled with -1 and *count zeroed inside the first pass (a new matches_12 vector, as matchMap2KFPoints / Lines
 * build it, mapHandler.cpp:583-803); fresh == 0: both are in/out like the host-buffer entry points. */
int plm_dev_match_grid(plm_ctx *ctx, const plm_dev_grid_args *a, int fresh);

/* ---- top-2 exchange over NVLink peer memory (multi-GPU merge without a gather collective) ------ */
/* The per-query top-2 merge of a row-sharded database (config 5) / local map (config 4) as ONE kernel: every
 * rank pushes its packed keys straight into every other rank's exchange buffer (peer stores over NVLink /
 * NVSwitch), signals, waits for the other ranks' flags and merges -- see csrc/plm_peer.cuh.  Setup, once:
 *   1. each rank:  plm_peer_alloc(ctx, world, q_cap, &buf, handle)      (cudaMalloc + CUDA IPC handle, 64 bytes)
 *   2. the 64-byte handles are exchanged by the caller (any transport; torch.distributed all_gather here)
 *   3. each rank:  plm_peer_open(ctx, handle_of_rank_r, &ptr_r) for r != own rank
 * then per exchange plm_dev_top2_exchange with the same, strictly increasing `epoch` (> 0) on every rank.
 * All ranks must call it with the same n1 <= q_cap.  Results equal plm_dev_top2_merge over an all-gather
 * bit for bit (unsigned min over packed keys). */
#define PLM_PEER_HANDLE_BYTES 64
#define PLM_PEER_MAX_RANKS 16
size_t plm_peer_buffer_bytes(int world, int q_cap);
int plm_peer_alloc(plm_ctx *ctx, int world, int q_cap, void **buf_dev, uint8_t handle[PLM_PEER_HANDLE_BYTES]);
int plm_peer_open(plm_ctx *ctx, const uint8_t handle[PLM_PEER_HANDLE_BYTES], void **buf_dev);
int plm_peer_close(plm_ctx *ctx, void *buf_dev); /* a buffer obtained from plm_peer_open */
int plm_peer_free(plm_ctx *ctx, void *buf_dev);  /* a buffer obtained from plm_peer_alloc */
/* peers[r] = rank r's exchange buffer as mapped in this process (peers[rank] = own).  local_top2_dev: n1 x 2
 * packed keys of this rank.  Outputs (each may be NULL): top2_out_dev n1 x 2 merged keys; m12_dev_inout +
 * count_dev: matchNNR acceptance of the merged keys with ratio nnr (as plm_dev_nnr_accept).  error_dev
 * (int32, required) is set to 1 if a peer did not arrive within ~2 s (nothing is written then). */
int plm_dev_top2_exchange(plm_ctx *ctx, void *const *peers, int rank, int world, int q_cap, uint32_t epoch,
                          const uint64_t *local_top2_dev, int n1, uint64_t *top2_out_dev, float nnr,
                          int32_t *m12_dev_inout, int32_t *count_dev, int32_t *error_dev);

/* Element-wise reductions over the ranks through the same exchange buffers (the two exchanges of the row-sharded
 * matchGrid, see plm_dev_grid_colmin / plm_dev_grid_match above).  src_dev / out_dev hold n_chunks 16-byte chunks
 * (n_chunks <= q_cap; pad the arrays to a multiple of 16 bytes with the identity of the reduction):
 *   PLM_PEER_MIN_U64         out = min over ALL ranks, 2 x uint64 per chunk (pad UINT64_MAX)
 *   PLM_PEER_PREFIX_MIN_U16  out = min over the ranks BELOW this one, 8 x uint16 per chunk; 0xFFFF where there is
 *                            none (pad 0xFFFF)
 * Same epoch / error conventions as plm_dev_top2_exchange (one epoch counter per set of buffers). */
#define PLM_PEER_MIN_U64 0
#define PLM_PEER_PREFIX_MIN_U16 1
int plm_dev_peer_reduce(plm_ctx *ctx, void *const *peers, int rank, int world, int q_cap, uint32_t epoch, int op,
                        const void *src_dev, int n_chunks, void *out_dev, int32_t *error_dev);

/* All-gather of the per-shard match vectors and sum of the per-shard counts (the last step of the row-sharded match /
 * matchGrid) as one kernel over a second set of peer-mapped buffers: plm_peer_gather_bytes(world, n_rows_cap) bytes
 * each, from plm_peer_alloc_bytes (zero-initialised; handles exchanged and opened like the exchange buffers).  Rank r
 * contributes rows [row_lo, row_lo + n_local) of the n_rows-long vector and one count; every rank receives the whole
 * vector in out_dev and the sum of the counts in out_count_dev (may be NULL).  Own epoch counter per set of gather
 * buffers, same conventions as plm_dev_top2_exchange. */
size_t plm_peer_gather_bytes(int world, int64_t n_rows_cap);
int plm_peer_alloc_bytes(plm_ctx *ctx, size_t bytes, void **buf_dev, uint8_t handle[PLM_PEER_HANDLE_BYTES]);
int plm_dev_peer_allgather_i32(plm_ctx *ctx, void *const *peers, int rank, int world, int64_t n_rows_cap, uint32_t epoch,
                               const int32_t *local_dev, int64_t row_lo, int64_t n_local, int64_t n_rows,
                               const int32_t *local_count_dev, int32_t *out_dev, int32_t *out_count_dev,
                               int32_t *error_dev);

/* Single-GPU emulation of the peer kernels, for boxes with fewer GPUs than ranks (tests).  Kernels that wait for one
 * another must never be separate launches on one GPU (nothing guarantees that they run at the same time), so between
 * plm_peer_emulate_begin(world) and plm_peer_emulate_run the calling thread's plm_dev_top2_exchange /
 * plm_dev_peer_reduce / plm_dev_peer_allgather_i32 calls (one per rank, same kind and size, buffers = plain device
 * allocations of that GPU) are recorded instead of launched, and _run executes all of them as ONE cooperative launch
 * (blockIdx.y = rank): every waiting CTA is co-resident with the CTAs it waits for.  world <= 4. */
int plm_peer_emulate_begin(int world);
int plm_peer_emulate_run(plm_ctx *ctx);

/* The whole row-sharded matchGrid of one rank in ONE call (config 4 across GPUs): one minima pass, the prefix-min of the
 * column minima over the lower ranks, the match pass, the min of the per-column best pairs, the mutual check and the
 * all-gather of the match vectors + counts -- ten launches back to back, three of them exchanges over peer memory.
 * `a` describes this rank's shard exactly as for plm_dev_grid_colmin / plm_dev_grid_match (m12_inout = the shard's slice
 * of the in/out vector, count = a zeroed int32).  The call consumes exchange epochs xchg_epoch and xchg_epoch + 1 and
 * gather epoch gather_epoch.  Every rank receives the global vector (n_rows_total) and the global count. */
typedef struct plm_peer_group {
    void *const *xchg;   /* world exchange buffers (plm_peer_alloc), as mapped in this process */
    void *const *gather; /* world gather buffers (plm_peer_alloc_bytes(plm_peer_gather_bytes(..))) */
    int32_t rank, world, q_cap, pad_;
    int64_t n_rows_cap;
    uint32_t xchg_epoch, gather_epoch;
} plm_peer_group;
int plm_dev_sharded_match_grid(plm_ctx *ctx, const plm_dev_grid_args *a, const plm_peer_group *g, int64_t n_rows_total,
                               int32_t *m12_global_dev, int32_t *count_global_dev, int32_t *error_dev);

/* The row-sharded StVO::match of one rank (the brute-force fallback of matchMap2KF*, mapHandler.cpp:645-650, on the same
 * in/out vector) in one call: direction 12 local, direction 21 through the peer-memory top-2 exchange (epoch xchg_epoch),
 * mutual check, all-gather of the match vectors + counts (epoch gather_epoch).  m12_local_inout_dev = this shard's
 * slice of the in/out vector (n1 rows starting at global row i1_base); n2 <= q_cap frame descriptors. */
int plm_dev_sharded_match(plm_ctx *ctx, const void *d1_shard_dev, int n1, int64_t i1_base, const void *d2_dev, int n2,
                          float nnr, int best_lr, int32_t *m12_local_inout_dev, const plm_peer_group *g,
                          int64_t n_rows_total, int32_t *m12_global_dev, int32_t *count_global_dev, int32_t *error_dev);

/* ---- multi-device keyframe database / local map inside ONE process ----------------------------------- */
/* The entry point a single C++ host process (the reference's MapHandler: matchMap2KFPoints / Lines
 * src/mapHandler.cpp:583-803, isLoopClosure :3301-3409) uses to spread the local map or the keyframe database over the
 * GPUs of one box: the library owns the per-device contexts, enables peer access between every pair of devices,
 * allocates the exchange buffers and drives the peer-memory kernels itself -- no launcher, no IPC, no NCCL.
 * Rows are sharded contiguously (shard g = rows [g * per, (g + 1) * per), per = ceil(n_rows / n_devices)); every index
 * in a result is GLOBAL, so results are bit-identical to the single-GPU calls.  devices[] must be distinct and
 * mutually peer-accessible (PLM_E_UNSUPPORTED otherwise); n_devices == 1 is allowed (no exchange).
 * q_cap = the largest query batch / frame (rows) one exchange carries; rows_cap = the largest database / map.
 * One host thread at a time per plm_shard.  A timed-out exchange (option "peer_spin_ms", default ~2 s) makes the
 * current or the next call return PLM_E_PEER and every later one too: outputs are never silently wrong. */
typedef struct plm_shard plm_shard;
int plm_shard_create(const int *devices, int n_devices, int q_cap, int64_t rows_cap, plm_shard **out);
int plm_shard_destroy(plm_shard *s);
int plm_shard_n_devices(const plm_shard *s);
int64_t plm_shard_n_rows(const plm_shard *s);
int plm_shard_range(const plm_shard *s, int i, int64_t *row_lo, int64_t *row_hi);
uint64_t plm_shard_launch_count(const plm_shard *s);
int plm_shard_synchronize(plm_shard *s);
/* (Re)load the database / map: n_rows descriptors `step` bytes apart and, optionally (config 4), the grid-cell
 * coordinates of the same rows: n_rows x coords_per_row int32, 2 = points (x, y), 4 = lines (sx, sy, ex, ey). */
int plm_shard_upload(plm_shard *s, const uint8_t *rows, int64_t n_rows, size_t step, const int32_t *coords, int coords_per_row);
/* Config 5, flat database: StVO::matchNNR / knnMatch(k = 2) of n1 host queries against all rows.  top2 (n1 x 2 packed
 * keys), m12_inout + n_matches may each be NULL.  Batches above q_cap are processed in slices. */
int plm_shard_match_nnr(plm_shard *s, const uint8_t *q, int n1, size_t step, float nnr, uint64_t *top2, int32_t *m12_inout,
                        int *n_matches);
/* Config 4: StVO::matchGrid with the sharded map as desc1 (mapHandler.cpp:637-642, :752-757).  Frame side as in
 * plm_match_grid_points / _lines (lines when the uploaded coordinates have 4 columns; dirs2 then required);
 * m12_inout = the global in/out vector (n_rows). */
int plm_shard_match_grid(plm_shard *s, const int32_t *cell_start, const int32_t *cell_items, int grid_rows, int grid_cols,
                         const uint8_t *d2, int n2, size_t step2, const double *dirs2, double line_sim_th, const int32_t win[4],
                         double ratio, int best_lr, int32_t *m12_inout, int *n_matches);
/* Config 4 fallback: StVO::match(map, frame) on the same in/out vector (mapHandler.cpp:645-650, :760-765). */
int plm_shard_match(plm_shard *s, const uint8_t *d2, int n2, size_t step2, float nnr, int best_lr, int32_t *m12_inout,
                    int *n_matches);

/* A device-resident descriptor database shard (keyframe DB / local map). */
int plm_db_create(plm_ctx *ctx, int64_t capacity_rows, plm_db **out);
int plm_db_destroy(plm_db *db);
/* Copy n rows from host (step bytes apart) to rows [at_row, at_row + n); grows size to cover them. */
int plm_db_upload(plm_db *db, const uint8_t *rows, int64_t n, size_t step, int64_t at_row);
int64_t plm_db_size(const plm_db *db);
void *plm_db_device_ptr(const plm_db *db);
/* knn2 of host queries against the resident shard (H2D queries, D2H packed top-2). */
int plm_db_knn2(plm_db *db, const uint8_t *q, int nq, size_t step, uint64_t idx_base, uint64_t *top2);

/* ---- map landmarks: representative descriptor + mean observation direction -------------------- */
/* PLSLAM::MapPoint::updateAverageDescDir (src/mapFeatures.cpp:51-93) and MapLine::updateAverageDescDir
 * (:121-163), batched over n_lm landmarks.  Observations of landmark l are rows obs_start[l] ..
 * obs_start[l+1]-1 of desc_obs (n_obs x 32 bytes, `step` apart) and of dir_obs (n_obs x 3 doubles, may be
 * NULL together with med_dir).  Per landmark with n observations:
 *   med_idx  = first row i whose value at sorted position int(1 + 0.5*(n-1)) of its Hamming distances to
 *              all n rows (self included) is strictly smallest; 0 for n == 1 (constructor, :29-40),
 *              -1 for an empty list;
 *   med_desc = that descriptor (n_lm x 32 bytes, may be NULL; zeros for an empty list);
 *   med_dir  = (sum of the directions in list order, from zero) / n in fp64 (n_lm x 3, may be NULL).
 * obs_start must be non-decreasing within [0, n_obs] (PLM_E_INVALID otherwise).  Any n is supported;
 * lists of up to 32 observations take the one-warp-per-landmark kernel. */
int plm_med_desc(plm_ctx *ctx, const uint8_t *desc_obs, int64_t n_obs, size_t step, const double *dir_obs,
                 const int32_t *obs_start, int n_lm, int32_t *med_idx, uint8_t *med_desc, double *med_dir);
/* Same on device-resident arenas (all pointers are device pointers, rows contiguous and 16-byte aligned),
 * enqueued on the context's stream without a host sync.  dst_rows_dev (may be NULL) scatters: landmark l
 * writes its descriptor to row dst_rows[l] of med_desc_dev (< 0: not written) -- e.g. straight into the
 * rows of a resident local-map shard.  A malformed obs_start range is treated as an empty list. */
int plm_dev_med_desc(plm_ctx *ctx, const void *desc_obs_dev, int64_t n_obs, const double *dir_obs_dev,
                     const int32_t *obs_start_dev, int n_lm, int32_t *med_idx_dev, void *med_desc_dev,
                     const int32_t *dst_rows_dev, double *med_dir_dev);

/* ---- local-map selection and reprojection gates of matchMap2KF* (SURVEY 8f-1) ------------------- */
/* MapHandler::matchMap2KFPoints / Lines (src/mapHandler.cpp:583-682, :685-803) around the matcher:
 *   select  Pf = R X + t with Twf = [R | t]; pf = (cx + fx Pf0 / Pf2, cy + fy Pf1 / Pf2); a landmark is kept when its
 *           `active` byte is non-zero (local and not yet observed from this keyframe; NULL = all) and pf lies strictly
 *           inside the image with Pf2 > 0 (:602, :705-706; segments: both endpoints).  Kept landmarks are compacted in
 *           order: sel[j] = landmark index, coords[j] = (int)(pf * inv_width), (int)(pf * inv_height) per endpoint
 *           (the matchGrid query coordinates, :605, :709-710), pf[j] = the projection(s) for the gate.
 *   gate    per compacted row i1 with i2 = m12[i1] >= 0: points |pf - pl[i2]| < max_epip (:661-662); lines
 *           le[i2] . (spf, 1) < max_epip && le[i2] . (epf, 1) < max_epip, signed as written (:784-786).
 *           ok[i1] = 1 for an accepted pair, else 0; *count -= rejected pairs (the reference's --matches).
 * X: n x 3 doubles (points) or n x 6 (segment endpoints); feat: n2 x 2 (pl) or n2 x 3 (le).  fp64, every operation
 * rounded separately, the 3x3 product summed left to right (Eigen's own order for it is not reproducible here:
 * these fp64 values are "parity unpinned", DESIGN.md 5). */
typedef struct plm_map_view {
    double T[12];                 /* Twf rows 0..2, row-major: r00 r01 r02 tx | r10 r11 r12 ty | r20 r21 r22 tz */
    double fx, fy, cx, cy;
    double inv_width, inv_height; /* GRID_COLS / image width, GRID_ROWS / image height */
    int32_t width, height;
} plm_map_view;
int plm_map_select(plm_ctx *ctx, int is_lines, const double *X, const uint8_t *active, int n, const plm_map_view *v, int32_t *sel,
                   int32_t *coords, double *pf, int *n_sel);
int plm_map_gate(plm_ctx *ctx, int is_lines, const double *pf, const int32_t *m12, int n_sel, const double *feat, int n2, double max_epip,
                 uint8_t *ok, int *count_inout);
/* Device-resident forms (no host sync; *n_sel_dev is produced / consumed on the device, n_max bounds the launch). */
int plm_dev_map_select(plm_ctx *ctx, int is_lines, const double *X_dev, const uint8_t *active_dev, int n, const plm_map_view *v,
                       int32_t *sel_dev, int32_t *coords_dev, double *pf_dev, int32_t *n_sel_dev);
/* out[j] = rows[sel[j]], j < *n_sel: the representative descriptors of the selected landmarks (:606, :711). */
int plm_dev_gather_rows(plm_ctx *ctx, const void *rows_dev, const int32_t *sel_dev, const int32_t *n_sel_dev, int n_max, void *out_dev);
int plm_dev_map_gate(plm_ctx *ctx, int is_lines, const double *pf_dev, const int32_t *m12_dev, const int32_t *n_sel_dev, int n_max,
                     const double *feat_dev, int n2, double max_epip, uint8_t *ok_dev, int32_t *count_inout_dev);

/* ---- bag-of-words loop-candidate scoring (the reference's vendored DBoW2) ----------------------- */
/* A vocabulary tree as flat arrays, copied to the device once (DBoW2::TemplatedVocabulary::m_nodes,
 * TemplatedVocabulary.h:275-307, 383-408): node 0 is the root; the children of node i are
 * child_ids[child_start[i] .. child_start[i+1]-1] in the reference's vector order (ties in the descent go to
 * the FIRST child, :1225); node_desc is n_nodes x 32 bytes; node_weight the idf / tf weight of a node;
 * node_word[i] >= 0 is the word id of leaf i (-1 on inner nodes).  Requirements (PLM_E_INVALID otherwise):
 * child ids in (parent, n_nodes), every node except the root listed as a child exactly once, leaves carry a
 * word id.  weighting = DBoW2::WeightingType (0 TF_IDF, 1 TF, 2 IDF, 3 BINARY); scoring = DBoW2::ScoringType,
 * only 0 (L1_NORM, the DBoW2 default) is supported (PLM_E_UNSUPPORTED otherwise). */
typedef struct plm_voc plm_voc;
int plm_voc_create(plm_ctx *ctx, int n_nodes, const int32_t *child_start, const int32_t *child_ids,
                   const uint8_t *node_desc, const double *node_weight, const int32_t *node_word, int weighting,
                   int scoring, plm_voc **out);
int plm_voc_destroy(plm_voc *voc);
int plm_voc_words(const plm_voc *voc); /* number of words (max word id + 1) */
/* TemplatedVocabulary::transform(features, BowVector) for n_sets descriptor sets (set s = rows set_start[s] ..
 * set_start[s+1]-1 of desc): the L1-normalised BowVector of set s is written, in ascending word id, to
 * bow_ids / bow_vals at slots set_start[s] .. set_start[s] + bow_len[s] - 1 (so both arrays hold n_rows
 * entries).  Values are bit-identical to the reference's (same order of the fp64 additions).  A set may hold
 * at most 8192 features (PLM_E_UNSUPPORTED). */
int plm_bow_transform(plm_voc *voc, const uint8_t *desc, int64_t n_rows, size_t step, const int32_t *set_start,
                      int n_sets, uint32_t *bow_ids, double *bow_vals, int32_t *bow_len);
/* Same on device pointers (rows contiguous, 16-byte aligned), enqueued on the vocabulary's context stream;
 * max_set >= the largest set. */
int plm_dev_bow_transform(plm_voc *voc, const void *desc_dev, int64_t n_rows, const int32_t *set_start_dev, int n_sets,
                          int max_set, uint32_t *bow_ids_dev, double *bow_vals_dev, int32_t *bow_len_dev);
/* L1Scoring::score(query q, database vector j) for every (q, j): scores[q * n_db + j].  A vector is the
 * entries [start, start + len) of its ids / vals arrays, ids ascending.  This is the loop of
 * insertKFBowVectorP / L (mapHandler.cpp:3129-3137): one query (the new keyframe) against all earlier
 * keyframes; n_q > 1 scores several new keyframes in one launch.  A query may hold at most 8192 entries. */
int plm_bow_score(plm_ctx *ctx, const uint32_t *q_ids, const double *q_vals, const int64_t *q_start,
                  const int32_t *q_len, int n_q, const uint32_t *db_ids, const double *db_vals,
                  const int64_t *db_start, const int32_t *db_len, int n_db, double *scores);
/* Same on device pointers, no host sync; max_q_len >= the longest query; n_words = number of words of the
 * vocabulary (plm_voc_words; sizes the shared-memory membership bitmap of the query -- 0 = unknown: every database
 * entry is then looked up by binary search, same results). */
int plm_dev_bow_score(plm_ctx *ctx, const uint32_t *q_ids_dev, const double *q_vals_dev, const int64_t *q_start_dev,
                      const int32_t *q_len_dev, int n_q, int max_q_len, int64_t n_words, const uint32_t *db_ids_dev,
                      const double *db_vals_dev, const int64_t *db_start_dev, const int32_t *db_len_dev, int n_db,
                      double *scores_dev);

/* ---- loop-closure keyframe database (MapHandler::insertKFBowVectorP / L / PL + isLoopClosure) -------------------- */
/* The keyframes of MapHandler's loop-closure path, resident on the vocabularies' device: each keyframe's left point and
 * line descriptors and its BowVector(s) are uploaded / computed once, when it is inserted; nothing about an earlier
 * keyframe crosses PCIe again.  mode 0 = insertKFBowVectorP (voc_l may be NULL), 1 = insertKFBowVectorL (voc_p may be
 * NULL), 2 = insertKFBowVectorPL (both; they must live on the same device); fixed per database, as one MapHandler uses
 * one strategy.  The database runs on the context of voc_p (mode 1: voc_l).  kf_capacity = keyframes the arenas are
 * first sized for (0 = 64); every arena grows geometrically when needed.  One database object may be used by one host
 * thread at a time. */
typedef struct plm_loopdb plm_loopdb;
int plm_loopdb_create(plm_voc *voc_p, plm_voc *voc_l, int mode, int kf_capacity, plm_loopdb **out);
int plm_loopdb_destroy(plm_loopdb *db);
/* Inserts keyframe kf_idx (larger than every earlier kf_idx; gaps allowed) and scores it as insertKFBowVector* does
 * (mapHandler.cpp:3116-3237): conf_row[j] = score(kf_idx, j) for every live keyframe j < kf_idx, and conf_row[kf_idx] =
 * its self score; every other entry is left untouched.  Scores are bit-identical to plm_bow_transform + plm_bow_score
 * (a score without common words is -0.0).  pdesc / ldesc: the keyframe's left point / line descriptors (both are kept
 * for plm_loopdb_match whatever the mode); a set the mode transforms may hold at most 8192 features
 * (PLM_E_UNSUPPORTED).  blend = {n_pt, std_pt, n_ls, std_ls} of the PL blend for mode 2 (else ignored, may be NULL):
 *   s = 0.0 + (sp * n_pt + sl * n_ls) / (n_pt + n_ls);  s = s + (sp * std_pt + sl * std_ls) / (std_ls + std_pt)
 * in fp64, every operation rounded.  Cost per insert, whatever the database size: one host -> device copy (the
 * descriptors), 2 launches (3 in mode 2), one device -> host copy of the row, one synchronisation.  A failed insert
 * (argument error, PLM_E_UNSUPPORTED, allocation failure) leaves the database unchanged. */
int plm_loopdb_insert(plm_loopdb *db, int kf_idx, const uint8_t *pdesc, int n_p, size_t step_p, const uint8_t *ldesc,
                      int n_l, size_t step_l, const double *blend, double *conf_row);
/* map_keyframes[kf_idx] = NULL: the keyframe is skipped by every later insert and match (its storage is kept).
 * PLM_E_INVALID unless kf_idx is a live keyframe of the database. */
int plm_loopdb_cull(plm_loopdb *db, int kf_idx);
/* The stored BowVector of live keyframe kf_idx (descDBoW_P for which = 0, descDBoW_L for which = 1; the vocabulary
 * must be one the mode scores with): *len entries, ascending word id, to ids / vals, which need room for as many entries
 * as the keyframe's set had features. */
int plm_loopdb_bow(plm_loopdb *db, int kf_idx, int which, uint32_t *ids, double *vals, int32_t *len);
/* isLoopClosure's two StVO::match calls (mapHandler.cpp:3325-3378) for n_pairs candidate pairs, from the resident rows:
 * points of kf0 against points of kf1[k] with nnr_p -> count_pt[k], m12_pt[k * n_p(kf0) ..]; lines with nnr_l ->
 * count_ls[k], m12_ls[k * n_l(kf0) ..] (either match array may be NULL).  Results equal plm_match's on the same rows,
 * including a side with 0 or 1 rows: count 0 and every entry -1 (the reference skips an empty side).  Every keyframe
 * must be live (PLM_E_INVALID otherwise, before any work).  Points and lines run as one batch when nnr_p == nnr_l;
 * with option "batch_umma" = 1 (the tensor-core path of plm_batch_set_match_dev) each kind gets a batch of its own,
 * whose jobs share kf0's rows as the query range. */
int plm_loopdb_match(plm_loopdb *db, int kf0, const int32_t *kf1, int n_pairs, float nnr_p, float nnr_l, int best_lr,
                     int32_t *count_pt, int32_t *count_ls, int32_t *m12_pt, int32_t *m12_ls);
/* Keyframes inserted (culled ones included). */
int64_t plm_loopdb_size(const plm_loopdb *db);
/* Cumulative bytes copied host -> device / device -> host by inserts and matches (inserts: exactly the descriptor
 * rows in, the score row out). */
int64_t plm_loopdb_h2d_bytes(const plm_loopdb *db);
int64_t plm_loopdb_d2h_bytes(const plm_loopdb *db);

/* ---- resident local map (MapHandler's map_points / map_lines + matchMap2KFPoints / Lines) ------------------------ */
/* The landmarks of MapHandler's local-mapping thread, resident on the context's device: positions, the `active` byte of
 * plm_map_select, med_desc / med_dir and every observation (descriptor + direction).  A landmark crosses PCIe once, when
 * it is inserted; later calls send only what changes, and matchMap2KF* runs from the resident rows.  One store holds one
 * kind (is_lines = 0: points, X = 3 doubles; 1: segments, X = 6 doubles), as the reference keeps map_points and
 * map_lines apart.  A landmark's index (slot) is the reference's index into map_points / map_lines: slots are handed
 * out in insertion order and never reused.  lm_capacity / obs_capacity: landmarks / observation rows the arenas are
 * first sized for (0 = 1024 / 4096); every arena grows geometrically.  Each landmark owns a reserved run of
 * observation rows (4 when inserted); a list that outgrows its run moves, device to device, to the tail of the arenas
 * with twice the room.  One store may be used by one host thread at a time.
 *
 * Every call validates its arguments on the host before any device work (argument errors never touch the GPU); a failed
 * call (argument error, invalid or culled slot, duplicate cull, PLM_E_UNSUPPORTED, allocation failure) leaves the store
 * unchanged.  Cost per call, whatever the number of landmarks (n = entries of the call, u = distinct landmarks an
 * observation call touches, n2 = keyframe features, c = grid cells, k = cell_start[c], per = 1 points / 2 segments):
 *   insert            1 host -> device copy of n * (56 + 24 per) bytes, 1 launch
 *   add_observations  1 host -> device copy of 60 n + 20 u bytes (rows, directions, destination rows; per landmark its
 *                     old and new run), 3 launches (append + the two medoid kernels) and a memset
 *   set_positions     1 host -> device copy of n * (4 + 24 per) bytes, 1 launch
 *   set_active        1 host -> device copy of 5 n bytes, 1 launch
 *   cull              1 host -> device copy of 4 n bytes, 1 launch
 * An update call makes no device -> host copy and no synchronisation; it only waits for the host -> device copy of the
 * previous update, whose pinned staging block it reuses.  The cost of plm_localmap_match_kf is stated with it. */
typedef struct plm_localmap plm_localmap;
int plm_localmap_create(plm_ctx *ctx, int is_lines, int lm_capacity, int64_t obs_capacity, plm_localmap **out);
int plm_localmap_destroy(plm_localmap *lm);
/* Appends n landmarks with the next slots (*first_idx = the first; may be NULL): X (n x 3 or n x 6 doubles), one
 * observation each (desc: n x 32 bytes `step` apart, dir: n x 3 doubles), as the MapPoint / MapLine constructors
 * (mapFeatures.cpp:29-40, :99-110): med_desc = desc, med_dir = dir.  New landmarks are active. */
int plm_localmap_insert(plm_localmap *lm, int n, const double *X, const uint8_t *desc, size_t step, const double *dir,
                        int *first_idx);
/* Appends observation i (desc row i, dir row i) to landmark lm_idx[i], in array order (a landmark may appear several
 * times), then recomputes med_desc and med_dir of every touched landmark in one batch of the medoid kernels
 * (plm_med_desc): the result is updateAverageDescDir of the final list, i.e. what the reference leaves after its
 * recompute per append. */
int plm_localmap_add_observations(plm_localmap *lm, int n, const int32_t *lm_idx, const uint8_t *desc, size_t step,
                                  const double *dir);
/* X[idx[i]] = row i of X (e.g. after local bundle adjustment); active[idx[i]] = val[i].  A slot listed twice takes its
 * last entry. */
int plm_localmap_set_positions(plm_localmap *lm, int n, const int32_t *idx, const double *X);
int plm_localmap_set_active(plm_localmap *lm, int n, const int32_t *idx, const uint8_t *val);
/* map_points[idx[i]] = NULL: the slots are never selected again; setting, updating or reading a culled slot, or culling
 * it again (also twice in one call), returns PLM_E_INVALID. */
int plm_localmap_cull(plm_localmap *lm, int n, const int32_t *idx);
/* The keyframe side of plm_localmap_match_kf, from the host: its still unmatched features (desc: n2 x 32 bytes `step`
 * apart), their grid (CSR as plm_match_grid_points takes it: cell_start = grid_rows * grid_cols + 1 entries, cell_items =
 * cell_start[last] entries), dirs2 (n2 x 2, segments only) and feat for the gate: pl (n2 x 2) for points, le (n2 x 3)
 * for segments. */
typedef struct plm_localmap_kf {
    const uint8_t *desc;
    size_t step;
    const int32_t *cell_start;
    const int32_t *cell_items;
    const double *dirs2;
    const double *feat;
    int32_t n2, grid_rows, grid_cols, pad_;
} plm_localmap_kf;
/* The config values matchMap2KF* reads: ratio (matchGrid, Config::minRatio12P), line_sim_th (Config::lineSimTh), max_epip
 * (SlamConfig::maxKFEpipP / L), nnr (the fallback's float ratio), ws (Config::matchingF2FWs: window +-ws),
 * best_lr (Config::bestLRMatches), fast_matching (SlamConfig::fastMatching), min_matches (minPointMatches /
 * minLineMatches). */
typedef struct plm_localmap_params {
    double ratio, line_sim_th, max_epip;
    float nnr;
    int32_t ws, best_lr, fast_matching, min_matches, pad_;
} plm_localmap_params;
/* MapHandler::matchMap2KFPoints / Lines (mapHandler.cpp:583-682, :685-803) from the resident rows in one call: selection
 * (plm_map_select over every slot with its active byte), gather of med_desc of the selected rows, matchGrid with a +-ws
 * window when fast_matching, then StVO::match(nnr) on the same vector (stale entries kept) when
 * n_sel > min_matches && matches < min_matches -- n_sel standing for both feature counts, as the reference passes them
 * -- and the reprojection gate.  Outputs: *n_sel selected slots in order (sel), m12 and ok per selected slot, *count =
 * the reference's match count after the gate; sel / m12 / ok need room for plm_localmap_size entries.  An empty map,
 * n_sel == 0 or n2 == 0 give m12 = -1, ok = 0, count 0.  Results equal plm_map_select + plm_match_grid_* + plm_match +
 * plm_map_gate on the same rows bit for bit.  Synchronises at most three times: for n_sel (it sizes the grid launches),
 * for the grid count (only when fast_matching and n_sel > min_matches) and at the end.  Host -> device: one copy of
 * n2 * (48 + 24 is_lines) + 4 (c + 1 + k) bytes; device -> host: 4 + 9 n_sel + 4 bytes, + 4 with the grid count. */
int plm_localmap_match_kf(plm_localmap *lm, const plm_map_view *v, const plm_localmap_kf *kf, const plm_localmap_params *p,
                          int32_t *sel, int32_t *m12, uint8_t *ok, int *n_sel, int *count);
/* One keyframe's raw features, both kinds, as the reference holds them: points (kp: n_p x 2 float pixels,
 * cv::KeyPoint::pt; pdesc: n_p x 32 bytes `pstep` apart; pl: n_p x 2 doubles for the gate) and segments (segs: n_l x 4
 * float pixels sx, sy, ex, ey; ldesc; le: n_l x 3 doubles for the gate), and the shape of the grid.  Either kind may have
 * no rows. */
typedef struct plm_localmap_kf_raw {
    const float *kp;
    const uint8_t *pdesc;
    size_t pstep;
    const double *pl;
    const float *segs;
    const uint8_t *ldesc;
    size_t lstep;
    const double *le;
    int32_t n_p, n_l, grid_rows, grid_cols;
} plm_localmap_kf_raw;
/* Outputs of one kind, as plm_localmap_match_kf writes them: sel / m12 / ok need room for plm_localmap_size entries. */
typedef struct plm_localmap_out {
    int32_t *sel, *m12;
    uint8_t *ok;
    int32_t n_sel, count;
} plm_localmap_out;
/* p: points, l: segments; h2d_bytes / d2h_bytes / syncs: what the call copied and how often it synchronised. */
typedef struct plm_localmap_pl_out {
    plm_localmap_out p, l;
    int64_t h2d_bytes, d2h_bytes;
    int32_t syncs, pad_;
} plm_localmap_pl_out;
/* The map half of MapHandler::lookForCommonMatches for one keyframe (matchMap2KFPoints, then matchMap2KFLines,
 * mapHandler.cpp:865-871) in one call, from the keyframe's raw features.  The grids are built on the device: points go to
 * cell (trunc(x * inv_width), trunc(y * inv_height)) of the view (off-grid points to no cell), segments to every cell of
 * getLineCoords over the scaled endpoints, with their unit directions; items ascending inside a cell -- the host's
 * GridStructure exactly.  Results equal two plm_localmap_match_kf calls bit for bit, given the host-built grids
 * (grid.csr_from_points over kp * inv_width / height, drivers.line_grid) and the same pl / le; pp / pl are the two kinds'
 * params.  Either store may be NULL (that kind is skipped, its out entries are left alone apart from n_sel = count = 0);
 * both must be on the same context.  Every check is made on the host before any device work (PLM_E_INVALID for stores on
 * different contexts, a store of the wrong kind, null pointers or segment endpoints more than 2^20 cells off the grid;
 * PLM_E_GRID / PLM_E_UNSUPPORTED for grids of no cell or more than 8192 cells); a failed call changes neither store.
 * Cost, whatever the number of landmarks (kinds whose store is NULL or empty count n = 0 and n_sel = 0):
 *   host -> device: one copy of exactly the raw keyframe side, 56 n_p + 72 n_l bytes; no grid crosses PCIe;
 *   device -> host: 8 bytes (both n_sel), + 8 (both grid counts, when a fallback is possible), + 9 (n_sel_p + n_sel_l)
 *   + 8 (sel | m12 | count | ok of both kinds, one copy); with both n_sel 0 the call ends after the first 8 bytes;
 *   synchronisations: at most 3 for the whole keyframe -- both n_sel, both grid counts (only when fast_matching and
 *   n_sel > min_matches for a kind) and the end (besides the wait for the previous update's copy out of the same pinned
 *   block that every call of a store makes);
 *   launches: 1 (both grids, when some kind has landmarks, features and fast_matching) + L_p + L_l, where L_k is what
 *   plm_localmap_match_kf launches for that kind: 3 (selection) + with n_sel > 0 and n2 > 0: 1 (gather) + matchGrid
 *   (1; 4 with best_lr) + the brute-force fallback when it runs (knn2 + accept; twice and a cross check with best_lr)
 *   + 1 (gate); and one device -> device copy of sel of the segments.
 * The output cost goes to each store's h2d / d2h counters by kind (all of it to the one store when one kind runs). */
int plm_localmap_match_kf_pl(plm_localmap *points, plm_localmap *lines, const plm_map_view *v, const plm_localmap_kf_raw *kf,
                             const plm_localmap_params *pp, const plm_localmap_params *pl, plm_localmap_pl_out *out);
/* Reads n slots back: X (n x 3 or 6), med_desc (n x 32 bytes), med_dir (n x 3), n_obs (observations per slot); each may
 * be NULL.  One device -> host copy and one synchronisation. */
int plm_localmap_read(plm_localmap *lm, int n, const int32_t *idx, double *X, uint8_t *med_desc, double *med_dir, int32_t *n_obs);
/* Slots handed out (culled ones included). */
int64_t plm_localmap_size(const plm_localmap *lm);
/* Cumulative bytes copied host -> device / device -> host by every call (the formulas above; read-backs included). */
int64_t plm_localmap_h2d_bytes(const plm_localmap *lm);
int64_t plm_localmap_d2h_bytes(const plm_localmap *lm);

/* Tuning knobs (measurement / A-B tests only; results never depend on them):
 *   "knn_variant"  -1 = automatic (default: 3 for train sets >= 65 536 rows, 5 for short train sides with >= 2^26 pairs,
 *                  else 1), 0 = plain 8-POPC Hamming, 1 = carry-save 5-POPC, 2 = carry-save 4-POPC with blocked top-2
 *                  update, 3 = 13-LOP3 / 4-POPC in the transformed domain (blocked update), 4 = 3 with three lower-bound
 *                  rows per block, 5 = 13-LOP3 with the per-pair update, 7 = the tensor-core kernel (int8 tcgen05 MMA,
 *                  exact) for every single-direction brute force (plm_dev_knn2, plm_knn2, plm_match_nnr, plm_db_knn2);
 *                  automatic mode takes it for train sets >= 65 536 rows with >= 256 queries.  Environment:
 *                  PLM_KNN_VARIANT=popc8|csa5|csa4|t13|mix|t13s|umma.
 *   "batch_umma"   batches of plm_batch_set_match / _dev (and plm_loopdb_match) whose live jobs share one query range:
 *                  1 = both directions of every pair from one int8 tensor-core product (knn2_umma_pairs_kernel),
 *                  0 = the integer list kernels, -1 = automatic (default; today the integer list kernels, which measured
 *                  faster at the loop-closure shapes, DESIGN K1c).  Read when the batch is prepared.  Forcing
 *                  "knn_variant" 0-5 keeps the integer kernels.
 *   "knn_qpt"      2 = long scans with >= 4096 queries keep two queries per thread (default 1).
 *   "knn_fill"     0 = do not fill the last resident CTA slots / share the second-best bound (default 1).
 *   "frame_fused"  1 = frame sessions and stand-alone frame-sized calls run as ONE launch (frame_fused_kernel, default),
 *                  0 = one lane of copies + kernels per call.
 *   "grid_cluster" single matchGrid calls outside the one-launch path: 2 = row-parallel kernel on one 8-CTA thread-block
 *                  cluster (default), 1 = chunk phases on a cluster, 0 = one CTA.
 *   "grid_rows"    1 = map-sized matchGrid uses the row-parallel kernels (default), 0 = warp-per-chunk kernels.
 *   "grid_head"    1 = short CTAs at the start of the map (default), 0 = uniform rows per CTA.
 *   "frames_out_group"  chunks per device -> host copy group of plm_frames_process (default 2).
 *   "frames_threads_p" / "frames_threads_l"  CTA width of the frame pipeline's point chain (256 or 512, default 512)
 *                  and line chain (128 or 256, default 256).
 *   "frames_pairs_p" / "frames_pairs_l"  candidate slots per query row the frame pipeline's pair-list
 *                  matcher is sized for (default 8 / 0; 0 = always use the chunk phases).
 *   "peer_spin_ms" bounded spin of the peer-memory kernels in milliseconds (default ~2000). */
int plm_set_option(const char *key, int value);

/* ---- measurement helpers --------------------------------------------------------------------- */

/* Issue-rate micro-benchmark of the integer pipe on the context's device: giga-instructions/s of
 * independent POPC.32 (*popc_gops) and LOP3.32 (*lop3_gops) per GPU. */
int plm_measure_int_peaks(plm_ctx *ctx, double *popc_gops, double *lop3_gops);
/* Rate of back-to-back int8 tensor-core MMAs (tcgen05.mma kind::i8, 128 x 256 x 32, s32 accumulate) on every SM of the
 * context's device: tera-operations/s (2 per multiply-accumulate) per GPU. */
int plm_measure_mma_i8_peak(plm_ctx *ctx, double *tops);
/* Rate of back-to-back int8 tensor-core MMAs of shape 128 x n x 32 (n = 128 or 256) on every SM, tera-operations/s per
 * GPU.  with_stores != 0: three more warps per SM keep storing to shared memory meanwhile, as the expansion of the
 * tensor-core brute force does.  plm_measure_mma_i8_peak is n = 256 without stores. */
int plm_measure_mma_i8_rate(plm_ctx *ctx, int n, int with_stores, double *tops);

#ifdef __cplusplus
}
#endif
#endif /* PLMATCH_H_ */
