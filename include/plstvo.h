/*
 * plstvo.h — C-ABI of the B200-native PL-StVO frame-to-frame pose engine.
 *
 * Plain C, plain pointers and sizes; no Eigen / OpenCV / torch types cross this
 * boundary.  Every entry point names the reference interface it replaces
 * (paths relative to the rubengooj/stvo-pl checkout).  The reference-side
 * binding a maintainer would add is shown in INTEGRATION.md.
 *
 * Conventions
 *  - all 4x4 / 6x6 matrices are row-major doubles (Eigen is column-major: the
 *    shim transposes on the way in/out);
 *  - descriptors are rows of exactly 32 bytes (ORB and LBD: cv::Mat N x 32
 *    CV_8UC1, continuous) — src/matching.cpp:93-109 hard-codes 8 x int32;
 *  - twist layout x = [t(3); w(3)] (src/auxiliar.cpp:124-141);
 *  - functions return >= 0 on success (a count where the reference returns
 *    one) and a negative PLSTVO_E_* code where the reference throws
 *    (src/matching.cpp:50-51, src/stereoFrameHandler.cpp:1065-1066).
 *    optimizePose never throws in the reference: failure is encoded in the
 *    result exactly as src/stereoFrameHandler.cpp:382-391 does.
 */
#ifndef PLSTVO_H_
#define PLSTVO_H_

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PLSTVO_VERSION        100
#define PLSTVO_DESC_BYTES     32
#define PLSTVO_MAX_FEATURES   65535   /* per frame and feature type (16-bit index in the packed (dist,idx) key) */

/* error codes (negative returns) */
#define PLSTVO_E_INVALID      (-1)  /* bad argument (null pointer, negative size, stride != 32) */
#define PLSTVO_E_TOO_LARGE    (-2)  /* more than PLSTVO_MAX_FEATURES rows */
#define PLSTVO_E_CUDA         (-3)  /* CUDA runtime failure; see plstvo_last_error() */
#define PLSTVO_E_NO_DEVICE    (-4)  /* no sm_100 device: the library never falls back to a CPU path */
#define PLSTVO_E_SIZE         (-5)  /* size mismatch (the reference's std::runtime_error cases) */

/* ---- camera: PinholeStereoCamera getters used by the path
 *      (include/pinholeStereoCamera.h:80-88, src/pinholeStereoCamera.cpp:221-237) */
typedef struct PlCamera {
    double fx, fy, cx, cy, b;
    int32_t width, height;
} PlCamera;

/* ---- the ~15 Config values the path reads (include/config.h:39-105,
 *      defaults src/config.cpp:36-113, KITTI values config/config/config_kitti.yaml) */
typedef struct PlConfig {
    int32_t has_points;        /* Config::hasPoints()      */
    int32_t has_lines;         /* Config::hasLines()       */
    int32_t best_lr_matches;   /* Config::bestLRMatches()  — mutual check in StVO::match */
    int32_t use_motion_model;  /* Config::useMotionModel() */
    int32_t min_features;      /* Config::minFeatures()    */
    int32_t max_iters;         /* Config::maxIters()       */
    int32_t max_iters_ref;     /* Config::maxItersRef()    */
    int32_t solver_mode;       /* `mode` of optimizePose (src/stereoFrameHandler.cpp:329): 0 = GN (the hard-wired value), 1 = GN-robust */
    double  min_ratio_12_p;    /* narrowed to float at the call, src/stereoFrameHandler.cpp:141 */
    double  min_ratio_12_l;    /* src/stereoFrameHandler.cpp:164 */
    double  homog_th;
    double  min_error;
    double  min_error_change;
    double  inlier_k;
    double  lsd_scale;         /* Config::lsdScale(): LineFeature::safeCopy re-applies it (src/stereoFeatures.cpp:117-135) */
} PlConfig;

/* ---- a batch of B stereo frames with pre-extracted features (the contents of
 *      StereoFrame::stereo_pt / stereo_ls / pdesc_l / ldesc_l, include/stereoFrame.h:59-115),
 *      structure-of-arrays, frames concatenated; *_off are prefix sums with B+1 entries.
 *      Arrays the role does not read may be NULL:
 *        as `prev`: pdesc, ldesc, pt_P, pt_sigma2, ls_sP, ls_eP, ls_spl, ls_epl, ls_sigma2, ls_level
 *        as `curr`: pdesc, ldesc, pt_pl, ls_le                                                      */
typedef struct PlFrameBatch {
    int32_t        B;
    const int32_t* pt_off;     /* [B+1] */
    const int32_t* ls_off;     /* [B+1] */
    const uint8_t* pdesc;      /* [n_pt][32]  StereoFrame::pdesc_l */
    const uint8_t* ldesc;      /* [n_ls][32]  StereoFrame::ldesc_l */
    const double*  pt_P;       /* [n_pt][3]   PointFeature::P      (include/stereoFeatures.h:30-58) */
    const double*  pt_pl;      /* [n_pt][2]   PointFeature::pl     */
    const double*  pt_sigma2;  /* [n_pt]      PointFeature::sigma2 */
    const double*  ls_sP;      /* [n_ls][3]   LineFeature::sP      (include/stereoFeatures.h:60-121) */
    const double*  ls_eP;      /* [n_ls][3]   LineFeature::eP      */
    const double*  ls_le;      /* [n_ls][3]   LineFeature::le      */
    const double*  ls_spl;     /* [n_ls][2]   LineFeature::spl     */
    const double*  ls_epl;     /* [n_ls][2]   LineFeature::epl     */
    const double*  ls_sigma2;  /* [n_ls]      LineFeature::sigma2  */
    const int32_t* ls_level;   /* [n_ls]      LineFeature::level   */
} PlFrameBatch;

/* ---- explicit matched lists for B problems (StereoFrameHandler::matched_pt / matched_ls after
 *      f2fTracking, i.e. after safeCopy: sigma2 is used as given) */
typedef struct PlMatchedBatch {
    int32_t        B;
    const int32_t* pt_off;     /* [B+1] */
    const int32_t* ls_off;     /* [B+1] */
    const double*  pt_P;       /* [n][3] */
    const double*  pt_pl_obs;  /* [n][2] */
    const double*  pt_sigma2;  /* [n]    */
    const uint8_t* pt_inlier;  /* [n] or NULL (= all true, as f2fTracking leaves them) */
    const double*  ls_sP;      /* [m][3] */
    const double*  ls_eP;      /* [m][3] */
    const double*  ls_le_obs;  /* [m][3] */
    const double*  ls_spl;     /* [m][2] previous-frame endpoints (src/stereoFrameHandler.cpp:668) */
    const double*  ls_epl;     /* [m][2] */
    const double*  ls_sigma2;  /* [m]    */
    const uint8_t* ls_inlier;  /* [m] or NULL */
} PlMatchedBatch;

/* ---- state of prev_frame read by optimizePose (src/stereoFrameHandler.cpp:317-326, :377-378) */
typedef struct PlPrior {
    double Tfw[16];
    double Tfw_cov[36];
    double DT[16];
    double DT_cov[36];
    double err_norm;
} PlPrior;

/* status: which branch of optimizePose produced the result */
#define PLSTVO_ST_REFINED          0  /* stage 1 ok -> removeOutliers -> stage 2 (src/stereoFrameHandler.cpp:341-350) */
#define PLSTVO_ST_ROBUST_FALLBACK  1  /* stage 1 rejected -> gaussNewtonOptimizationRobust (:357-359) */
#define PLSTVO_ST_FEW_BEFORE       2  /* n_inliers < minFeatures before optimisation (:364-368) */
#define PLSTVO_ST_FEW_AFTER        3  /* n_inliers < minFeatures after removeOutliers (:351-355) */

/* ---- what optimizePose leaves in curr_frame and the handler (src/stereoFrameHandler.cpp:372-391) */
typedef struct PlPoseResult {
    double  DT[16];          /* curr_frame->DT = expmap(logmap(inverse(DT_opt)))  (:374) */
    double  DT_cov[36];      /* curr_frame->DT_cov                                (:375) */
    double  DT_cov_eig[6];   /* ascending                                        (:379-380) */
    double  err_norm;        /* curr_frame->err_norm, -1 on failure               (:376,:387) */
    double  Tfw[16];         /* curr_frame->Tfw                                   (:377,:388) */
    double  Tfw_cov[36];     /* curr_frame->Tfw_cov                               (:378,:389) */
    double  DT_opt[16];      /* the optimised prev->curr transform before inversion (diagnostic) */
    int32_t n_matched_pt;    /* matched_pt.size() */
    int32_t n_matched_ls;    /* matched_ls.size() */
    int32_t n_inliers_pt;
    int32_t n_inliers_ls;
    int32_t n_inliers;
    int32_t good;            /* 1 iff the final isGoodSolution && DT != I branch was taken (:372) */
    int32_t status;          /* PLSTVO_ST_* */
    int32_t iters_stage1;    /* evaluations of optimizeFunctions in the first GN call  */
    int32_t iters_stage2;    /* evaluations in the refinement / robust fallback call   */
    int32_t reserved;
} PlPoseResult;

typedef struct PlContext PlContext;   /* one per GPU; owns streams, device and pinned buffers */
typedef struct PlDeviceBatch PlDeviceBatch; /* inputs resident in HBM (throughput mode) */

/* ---- life cycle ------------------------------------------------------------------------------- */
int         plstvo_version(void);
/* device < 0: use the current device.  Fails with PLSTVO_E_NO_DEVICE when there is no CUDA device. */
int         plstvo_create(int device, PlContext** out);
void        plstvo_destroy(PlContext* ctx);
const char* plstvo_last_error(const PlContext* ctx);
void        plstvo_default_config(PlConfig* cfg);        /* src/config.cpp:36-113 */
void        plstvo_kitti_config(PlConfig* cfg);          /* config/config/config_kitti.yaml */

/* ---- include/matching.h surface --------------------------------------------------------------- */
/* StVO::matchNNR (src/matching.cpp:41-61): m12[i] = index of the nearest row of d2 or -1; returns #accepted.
 * The reference has undefined behaviour for n2 < 2; here every row gets -1. */
int plstvo_match_nnr(PlContext* ctx, const uint8_t* d1, int n1, const uint8_t* d2, int n2,
                     int stride_bytes, float nnr, int32_t* m12);
/* StVO::match (src/matching.cpp:63-91): matchNNR both ways + mutual filter when best_lr_matches != 0. */
int plstvo_match(PlContext* ctx, const uint8_t* d1, int n1, const uint8_t* d2, int n2,
                 int stride_bytes, float nnr, int best_lr_matches, int32_t* m12);
/* Batched form: problem p matches rows [off1[p],off1[p+1]) of d1 against [off2[p],off2[p+1]) of d2.
 * m12 holds indices local to the problem.  counts[p] (optional) = the reference's return value. */
int plstvo_match_batch(PlContext* ctx, int B, const uint8_t* d1, const int32_t* off1,
                       const uint8_t* d2, const int32_t* off2, float nnr, int best_lr_matches,
                       int32_t* m12, int32_t* counts);

/* ---- include/matching.h surface, the stereo (left/right) step: StVO::matchGrid (src/matching.cpp:111-258) ----------
 * SURVEY 8(f)-1, the row next to the hot path: same 256-bit Hamming primitive, candidates restricted to a window of
 * the 64 x 48 bucket grid (GridStructure::get, src/gridStructure.cpp:65-76), the loop-carried gate of
 * Config::bestLRMatches() (a train is only considered by a query if it beats the train's running minimum over all
 * EARLIER queries, :145-150), best / second best with multiplicity, ratio test in double, mutual filter.
 * Batched over B frames: q_off / t_off are prefix offsets of queries (left image) and trains (right image). */
typedef struct PlGridWindow {   /* GridWindow: width = (left, right), height = (up, down), include/gridStructure.h:39-41 */
    int32_t left, right, up, down;
} PlGridWindow;

/* points (src/matching.cpp:111-177; caller src/stereoFrame.cpp:129-146): q_cell / t_cell = integer grid cell (x, y) of
 * every query / train keypoint (kp.pt.x * inv_width, kp.pt.y * inv_height truncated).  m12: problem-local index or -1.
 * counts (optional) = the reference's return value per frame. */
int plstvo_match_grid_points(PlContext* ctx, int B, int grid_rows, int grid_cols, PlGridWindow w, int best_lr_matches,
                             double min_ratio_12_p, const int32_t* q_off, const int32_t* q_cell, const uint8_t* d1,
                             const int32_t* t_off, const int32_t* t_cell, const uint8_t* d2, int32_t* m12,
                             int32_t* counts);
/* lines (src/matching.cpp:179-258; caller src/stereoFrame.cpp:318-345): q_line = integer cells (sp.x, sp.y, ep.x, ep.y) of
 * the query segments; t_line = train segment end points in GRID UNITS as doubles (x1, y1, x2, y2), rasterised into
 * cells exactly like getLineCoords / LineIterator (src/lineIterator.cpp:34-77); t_dir = directions2 (normalised).
 * The reference uses minRatio12P here too (:241). */
int plstvo_match_grid_lines(PlContext* ctx, int B, int grid_rows, int grid_cols, PlGridWindow w, int best_lr_matches,
                            double min_ratio_12_p, double line_sim_th, const int32_t* q_off, const int32_t* q_line,
                            const uint8_t* d1, const int32_t* t_off, const double* t_line, const double* t_dir,
                            const uint8_t* d2, int32_t* m12, int32_t* counts);

/* ---- 3-D lifting of the stereo matches (SURVEY 8(f)-2): the step that turns matchGrid's output into the PointFeature /
 * LineFeature records the solver consumes (src/stereoFrame.cpp:149-172 points, :348-397 lines, filterLineSegmentDisparity
 * :405-415, lineSegmentOverlapStereo :473-508, backProjection src/pinholeStereoCamera.cpp:221-229).  Pure per-feature
 * arithmetic + an ordered compaction (surviving features keep ascending left index, like the reference's push_back loop).
 * Batched over B frames; outputs of frame p are written densely starting at element l_off[p]; counts[p] = survivors. */
typedef struct PlStereoConfig {   /* Config accessors read by this step (include/config.h:72-96, src/config.cpp:58-106) */
    double max_dist_epip, min_disp, ls_min_disp_ratio, line_horiz_th, stereo_overlap_th, orb_scale_factor, lsd_scale;
} PlStereoConfig;
void plstvo_default_stereo_config(PlStereoConfig* c);
/* kp_l / kp_r: cv::KeyPoint::pt (float x, y); octave_l: cv::KeyPoint::octave; m12: matchGrid output (local right index or -1).
 * out: PointFeature::pl, disp, P, sigma2, level; pdesc_out = the surviving rows of desc_l (pdesc_l_aux); src_idx = their i1. */
int plstvo_stereo_lift_points(PlContext* ctx, const PlCamera* cam, const PlStereoConfig* scfg, int B, const int32_t* l_off,
                              const float* kp_l, const int32_t* octave_l, const uint8_t* desc_l, const int32_t* r_off,
                              const float* kp_r, const int32_t* m12, double* pt_pl, double* pt_disp, double* pt_P,
                              double* pt_sigma2, int32_t* pt_level, uint8_t* pdesc_out, int32_t* src_idx, int32_t* counts);
/* seg_l / seg_r: KeyLine start / end points (float sx, sy, ex, ey); angle_l: KeyLine::angle; octave_l: KeyLine::octave.
 * out: LineFeature::spl, epl, sdisp, edisp, sP, eP, le, angle, sigma2, level; ldesc_out, src_idx as for points. */
int plstvo_stereo_lift_lines(PlContext* ctx, const PlCamera* cam, const PlStereoConfig* scfg, int B, const int32_t* l_off,
                             const float* seg_l, const float* angle_l, const int32_t* octave_l, const uint8_t* desc_l,
                             const int32_t* r_off, const float* seg_r, const int32_t* m12, double* ls_spl, double* ls_epl,
                             double* ls_sdisp, double* ls_edisp, double* ls_sP, double* ls_eP, double* ls_le,
                             double* ls_angle, double* ls_sigma2, int32_t* ls_level, uint8_t* ldesc_out, int32_t* src_idx,
                             int32_t* counts);

/* ---- StereoFrame::matchStereoPoints / matchStereoLines (src/stereoFrame.cpp:120-173, :309-398) in one device pass:
 * grid cells from the raw key points / key lines (:129-139, :318-337: x * inv_width truncated, inv_width = grid_cols / image
 * width), matchGrid, and the 3-D lifting, with the match list handed from kernel to kernel in HBM.  Inputs and outputs are
 * those of plstvo_stereo_lift_*; desc_r = right descriptors; m12 (optional) = matchGrid's list per left feature. */
typedef struct PlStereoMatchConfig {   /* include/stereoFrame.h:51-52, src/config.cpp:51, :60, :63, :91 */
    int32_t grid_rows, grid_cols;      /* GRID_ROWS 48, GRID_COLS 64 */
    int32_t matching_s_ws;             /* Config::matchingSWs(): cells to the left of the query, same row */
    int32_t best_lr_matches;
    double  min_ratio_12_p, line_sim_th;
} PlStereoMatchConfig;
void plstvo_default_stereo_match_config(PlStereoMatchConfig* c);
int plstvo_match_stereo_points(PlContext* ctx, const PlCamera* cam, const PlStereoMatchConfig* mcfg, const PlStereoConfig* scfg,
                               int B, const int32_t* l_off, const float* kp_l, const int32_t* octave_l, const uint8_t* desc_l,
                               const int32_t* r_off, const float* kp_r, const uint8_t* desc_r, int32_t* m12, double* pt_pl,
                               double* pt_disp, double* pt_P, double* pt_sigma2, int32_t* pt_level, uint8_t* pdesc_out,
                               int32_t* src_idx, int32_t* counts);
int plstvo_match_stereo_lines(PlContext* ctx, const PlCamera* cam, const PlStereoMatchConfig* mcfg, const PlStereoConfig* scfg,
                              int B, const int32_t* l_off, const float* seg_l, const float* angle_l, const int32_t* octave_l,
                              const uint8_t* desc_l, const int32_t* r_off, const float* seg_r, const uint8_t* desc_r,
                              int32_t* m12, double* ls_spl, double* ls_epl, double* ls_sdisp, double* ls_edisp, double* ls_sP,
                              double* ls_eP, double* ls_le, double* ls_angle, double* ls_sigma2, int32_t* ls_level,
                              uint8_t* ldesc_out, int32_t* src_idx, int32_t* counts);

/* ---- raw stereo features in, pose out: the matching half of StereoFrame::extractStereoFeatures (matchStereoPoints +
 * matchStereoLines, src/stereoFrame.cpp:120-173, :309-398) for the previous and the current frame of B independent pairs, then
 * f2fTracking + optimizePose (src/stereoFrameHandler.cpp:106-180, :307-392) on the lifted records, which never leave HBM.
 * The only host hop in between is the per-frame survivor counts (the tile plan of the descriptor matcher needs them). */
typedef struct PlStereoFeatures {      /* what detectStereoFeatures leaves for B frames (src/stereoFrame.cpp:78-118, :184-307) */
    int32_t        B;
    const int32_t* pl_off;  const int32_t* pr_off;    /* [B+1] left / right key points */
    const float*   kp_l;    const float*   kp_r;      /* [n][2] cv::KeyPoint::pt */
    const int32_t* poct_l;                            /* [n_l] cv::KeyPoint::octave */
    const uint8_t* pdesc_l; const uint8_t* pdesc_r;   /* [n][32] */
    const int32_t* ll_off;  const int32_t* lr_off;    /* [B+1] left / right key lines */
    const float*   seg_l;   const float*   seg_r;     /* [m][4] start / end point */
    const float*   angle_l;                           /* [m_l] KeyLine::angle */
    const int32_t* loct_l;                            /* [m_l] KeyLine::octave */
    const uint8_t* ldesc_l; const uint8_t* ldesc_r;   /* [m][32] */
} PlStereoFeatures;
/* n_stereo (optional): [B][4] = stereo_pt.size(), stereo_ls.size() of the previous and of the current frame. */
int plstvo_track_stereo_batch(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg, const PlStereoMatchConfig* mcfg,
                              const PlStereoConfig* scfg, const PlStereoFeatures* prev, const PlStereoFeatures* curr,
                              const PlPrior* priors, PlPoseResult* results, int32_t* n_stereo);

/* The same for a SEQUENCE: `frames` holds B + 1 consecutive frames, pair p = (frame p, frame p + 1), B results.  Every frame goes
 * through the stereo step once (it is the current frame of one pair and the previous frame of the next, like curr_frame ->
 * prev_frame in updateFrame, src/stereoFrameHandler.cpp:98-100).  Results are per pair with priors[p] as given (NULL: identity):
 * the chaining of Tfw along the sequence (:377-378) is a host-side scan over the B results (plstvo.hpp: chainPoses).
 * n_stereo (optional): [B + 1][2] = stereo_pt.size(), stereo_ls.size() per frame. */
int plstvo_track_stereo_sequence(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg, const PlStereoMatchConfig* mcfg,
                                 const PlStereoConfig* scfg, const PlStereoFeatures* frames, const PlPrior* priors,
                                 PlPoseResult* results, int32_t* n_stereo);

/* Streaming forms: enqueue and return a ticket (0 / 1) like plstvo_track_batch_async; results / n_stereo are valid after
 * plstvo_wait(ctx, ticket).  Two batches may be in flight, so the next batch's uploads run under this batch's kernels; inputs
 * must stay untouched (and should be pinned, plstvo_host_alloc) until the wait returns.
 * NOT fully asynchronous: the call itself blocks (holding the context's lock) until the stereo step of this batch has run on
 * the device, because the number of lifted stereo features per frame — a result of that step — sizes the tracking plan that
 * is built on the host; what overlaps with the caller (and with the other ticket) is the tracking half and the downloads. */
int plstvo_track_stereo_batch_async(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg, const PlStereoMatchConfig* mcfg,
                                    const PlStereoConfig* scfg, const PlStereoFeatures* prev, const PlStereoFeatures* curr,
                                    const PlPrior* priors, PlPoseResult* results, int32_t* n_stereo);
int plstvo_track_stereo_sequence_async(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg, const PlStereoMatchConfig* mcfg,
                                       const PlStereoConfig* scfg, const PlStereoFeatures* frames, const PlPrior* priors,
                                       PlPoseResult* results, int32_t* n_stereo);

/* ---- include/stereoFrameHandler.h surface ----------------------------------------------------- */
/* StereoFrameHandler::f2fTracking (src/stereoFrameHandler.cpp:106-180) for B independent
 * (prev, curr) pairs: descriptor matching for points and lines; m12_* hold problem-local indices
 * (prev row -> curr row or -1).  n_matched[2*p], [2*p+1] = matched_pt.size(), matched_ls.size(). */
int plstvo_f2f_tracking(PlContext* ctx, const PlConfig* cfg, const PlFrameBatch* prev,
                        const PlFrameBatch* curr, int32_t* m12_pt, int32_t* m12_ls, int32_t* n_matched);

/* StereoFrameHandler::optimizePose (src/stereoFrameHandler.cpp:307-392) on explicit matched lists.
 * priors may be NULL (identity Tfw, no motion-model state).  inlier_* (optional) receive the
 * final PointFeature::inlier / LineFeature::inlier flags in list order. */
int plstvo_optimize_pose(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg,
                         const PlMatchedBatch* matched, const PlPrior* priors,
                         PlPoseResult* results, uint8_t* inlier_pt, uint8_t* inlier_ls);

/* insertStereoPair's f2fTracking + optimizePose (app/imagesStVO.cpp:96-97) for B independent pairs,
 * entirely on the device: match -> build matched_pt/ls (ascending prev index, with the
 * LineFeature::safeCopy sigma2 rule) -> optimizePose.  Host buffers in, host buffers out;
 * H2D / compute / D2H are pipelined over chunks of pairs.
 * m12_* / inlier_* are indexed by prev-frame feature (problem-local curr index or -1; 1 = matched and
 * still an inlier after optimizePose).  Any output pointer may be NULL. */
int plstvo_track_batch(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg,
                       const PlFrameBatch* prev, const PlFrameBatch* curr, const PlPrior* priors,
                       PlPoseResult* results, int32_t* m12_pt, int32_t* m12_ls,
                       uint8_t* inlier_pt, uint8_t* inlier_ls);

/* Streaming form of plstvo_track_batch: enqueues the batch (H2D, kernels, D2H) and returns a ticket >= 0 without
 * waiting, so that the caller can submit batch k+1 (its H2D then overlaps the kernels of batch k) before it waits for
 * batch k.  Two batches may be in flight per context; all input AND output buffers of a batch must stay valid and
 * untouched until plstvo_wait(ticket) returned (use plstvo_host_alloc memory: pageable memory makes the copies
 * synchronous).  This is how a video pipeline drives the engine: frame k+1's features go up while pair k solves. */
int plstvo_track_batch_async(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg,
                             const PlFrameBatch* prev, const PlFrameBatch* curr, const PlPrior* priors,
                             PlPoseResult* results, int32_t* m12_pt, int32_t* m12_ls,
                             uint8_t* inlier_pt, uint8_t* inlier_ls);
int plstvo_wait(PlContext* ctx, int ticket);

/* ---- throughput mode: inputs resident in HBM -------------------------------------------------- */
int  plstvo_batch_upload(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg,
                         const PlFrameBatch* prev, const PlFrameBatch* curr, const PlPrior* priors,
                         PlDeviceBatch** out);
/* one pass of the hot path over the resident batch (no host<->device traffic); asynchronous */
int  plstvo_batch_run(PlContext* ctx, PlDeviceBatch* db);
/* run `iters` passes bracketed by CUDA events on the launching stream; *ms_total = elapsed.
 * flush_l2 != 0 writes a buffer larger than L2 between passes (outside the per-pass events, so
 * ms_total only sums the passes). */
int  plstvo_batch_run_timed(PlContext* ctx, PlDeviceBatch* db, int iters, int flush_l2, float* ms_total);
int  plstvo_batch_download(PlContext* ctx, PlDeviceBatch* db, PlPoseResult* results,
                           int32_t* m12_pt, int32_t* m12_ls, uint8_t* inlier_pt, uint8_t* inlier_ls);
void plstvo_batch_free(PlContext* ctx, PlDeviceBatch* db);
int  plstvo_synchronize(PlContext* ctx);

/* pinned host memory for callers that want zero-staging H2D (e2e mode) */
void* plstvo_host_alloc(size_t bytes);
void  plstvo_host_free(void* p);

/* ---- instrumentation -------------------------------------------------------------------------- */
/* kernels launched by this library since the context was created (bench.py's gpu_launches) */
int64_t plstvo_launch_count(const PlContext* ctx);
/* device time of the two stages of one pass over the resident batch, each launched alone `iters` times
 * on the context's stream and bracketed by CUDA events on that stream: *ms_match / *ms_solve = average
 * duration of one K1 (tc_expand + tc_hamming + tc_resolve over the batch) / one K2 (track_solve, one CTA per pair).
 * n_tiles (optional) = matching problems with work (enabled, both sides non-empty); n_pairs (optional) = pairs. */
int     plstvo_batch_kernel_times(PlContext* ctx, PlDeviceBatch* db, int iters, double* ms_match,
                                  double* ms_solve, int32_t* n_tiles, int32_t* n_pairs);
/* The same per stage: ms[0] = operand expansion, ms[1] = distance + top-2 kernel (tcgen05),
 * ms[2] = index resolution, ms[3] = building matched_pt / matched_ls when that is a kernel of its own (the streamed
 * solver; 0 when K2 does it internally), ms[4] = optimizePose (K2, or the streamed solver's
 * GN-loop / outlier / finalize kernels + K2 for the problems it hands back); of ms[4], streamed solver only (0 for K2):
 * ms[5] = the GN loop launch of stage 1, ms[6] = the gate + removeOutliers launch, ms[7] = the GN loop launch of stage 2.
 * counts (optional) = {bit 0: tensor-core matcher, bit 1: streamed solver, bits 8..: problems the streamed solver handed to
 * the fp64 kernel in the last pass; work items of the distance kernel; matching problems; pairs}. */
int     plstvo_batch_stage_times(PlContext* ctx, PlDeviceBatch* db, int iters, double ms[8], int32_t counts[4]);
/* GN evaluation (optimizeFunctions, src/stereoFrameHandler.cpp:549-694) of the resident matched
 * lists at given poses, streamed from HBM: the roofline kernel of config C5.
 * DT: [B][16]; H: [B][36]; g: [B][6]; e: [B]. */
int  plstvo_gn_eval_stream(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg,
                           const PlMatchedBatch* matched, const double* DT, int iters,
                           double* H, double* g, double* e, float* ms_total);
/* test hook: the block-wide radix selection of the streamed solver's outlier pass (solve.cu: block_select_wide) on n_lists
 * caller-supplied lists (values[off[p] .. off[p+1])): out[p] = the k[p]-th smallest value (mode 0), or the k[p]-th smallest of
 * |x - pivot[p]| rounded to float (mode 1: the MAD form of src/auxiliar.cpp:399-402). */
int  plstvo_debug_select(PlContext* ctx, int n_lists, const int32_t* off, const double* values, const int32_t* k,
                         const double* pivot, int mode, double* out);
/* test hook for the on-chip 6x6 routines of the solver (ColPivHouseholderQR solve + log|det|, inverse, symmetric
 * eigenvalues) on n caller-supplied matrices: H [n][36] row-major, g [n][6] -> x [n][6], lad [n], inv [n][36], eig [n][6] */
int  plstvo_debug_algebra(PlContext* ctx, int n, const double* H, const double* g, double* x, double* lad,
                          double* inv, double* eig);
/* POPC issue-rate micro-benchmark: returns 32-bit popcounts per second on this device */
int  plstvo_popc_rate(PlContext* ctx, double* popc_per_s);

#ifdef __cplusplus
}
#endif
#endif /* PLSTVO_H_ */
