/*
 * stlcalib.h — C-ABI of the B200-native calibration cost-evaluation path.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  The reference has no FFI: the
 * three optimisers call plain C++ functions/functors.  Every entry point below
 * names the reference interface it replaces (paths relative to the reference
 * tree).  Plain pointers and sizes only; no C++/torch types cross this line;
 * nothing throws across it (every call returns an stl_status_t).
 *
 *   reference call                                     → C-ABI entry
 *   -------------------------------------------------------------------------
 *   BALoss ctor: builds one KDTree3D per scan          → stl_create + stl_upload_pack
 *     (src/examples/iba_global.cpp:349-367)
 *   BAError(xvec, PointClouds, KdTrees, vTwl, ...)      → stl_eval_batch (B = 1)
 *     (src/examples/iba_global.cpp:169-344,
 *      src/examples/iba_func.cpp:179-354)
 *   iba_func main loop over a Sim3 list                → stl_eval_batch (B = list size)
 *     (src/examples/iba_func.cpp:458-470)
 *   BALoss::eval_x / Nomad eval_block                  → stl_eval_batch + stl_bbo
 *     (src/examples/iba_global.cpp:377-396)
 *   BuildProblem (association at the current estimate) → stl_associate
 *     (src/examples/iba_local.cpp:145-323)
 *   ceres::Problem::Evaluate over IBA_PlaneFactor /    → stl_linearize_batch
 *     Point2Point_Factor / Point2Plane_Factor + Huber
 *     (include/IBACalib2.hpp:152-184,570-584,611-625;
 *      src/examples/iba_local.cpp:263-309)
 *   g2o IBAPlaneEdge computeError/linearizeOplus       → stl_linearize_batch
 *     (include/IBACalib.hpp:74-155)
 *   one LM iteration at x (BAError for monitoring +    → stl_step_batch (reassociate = 1)
 *     BuildProblem + Evaluate, iba_local.cpp:434-446)
 *   the OpenMP reductions of BAError across keyframes  → stl_comm_init: keyframes sharded over GPUs,
 *     (iba_global.cpp:239-251,274-275,318-326)           one NCCL fp64 all-reduce per call
 */
#ifndef STLCALIB_H_
#define STLCALIB_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STL_ABI_VERSION 2
#define STL_MAX_COVIS 10 /* IBAPlaneEdge is fixed at <=10 covisible KFs (IBACalib.hpp:74) */

typedef enum stl_status {
    STL_OK = 0,
    STL_ERR_INVALID = 1,   /* bad argument / inconsistent pack            */
    STL_ERR_CUDA = 2,      /* CUDA runtime error (see stl_last_error)     */
    STL_ERR_NO_DEVICE = 3, /* no usable sm_100 device: there is NO CPU fallback */
    STL_ERR_STATE = 4,     /* call order violated (e.g. eval before upload) */
    STL_ERR_CAPACITY = 5   /* input exceeds a documented limit            */
} stl_status_t;

/*
 * Hot-path parameters: IBAGlobalParams (iba_global.cpp:26-52) and the
 * IBALocalParams members that BuildProblem reads (IBACalib2.hpp:104-137).
 * Defaults set by stl_default_params() are the KITTI-00 YAML values
 * (config/calib/00/iba_calib_global.yml:21-48).
 */
typedef struct stl_params {
    double max_pixel_dist;        /* 1.5   2-D association gate (px)                 */
    double corr_3d_2d_threshold;  /* 40    re-projection gate (px)                   */
    double corr_3d_3d_threshold;  /* 10    3-D/3-D gate (m)                          */
    double norm_radius;           /* 0.6   k-NN radius (m) (= neigh_radius)          */
    double norm_reg_threshold;    /* 0.02  plane regression gate                     */
    double min_diff_dist;         /* 0.2   min extent of the neighbourhood (m)       */
    double err_weight[2];         /* {1,1}                                           */
    double he_threshold;          /* 0.094 (host shim: BBO constraint)               */
    double valid_rate;            /* 0.95  (host shim: BBO constraint)               */
    double max_3d_dist;           /* 1.0   LM path: map-point NN gate (m)            */
    double robust_kernel_delta;   /* 2.98  Huber delta of 3-D/2-D blocks             */
    double robust_kernel_3ddelta; /* 1.0   Huber delta of 3-D/3-D blocks             */
    int32_t num_min_corr;         /* 30    frame skipped below this (iba_global.cpp:203) */
    int32_t norm_max_pts;         /* 30    k of the k-NN (<= 32)                     */
    int32_t norm_min_pts;         /* 5                                               */
    int32_t use_plane;            /* 1                                               */
    /* LM path, depth by Gaussian-process regression for non-planar neighbourhoods
     * (IBA_GPRFactor, IBACalib2.hpp:427-564; call site iba_local.cpp:272-280, commented
     * out in the reference, hence off by default).  Hyper-parameters are fixed per problem
     * (GPRParams.optimize = false); the per-factor L-BFGS fit (GPR::fit, GPR.hpp:350-387)
     * needs Ceres and stays on the host. */
    int32_t use_gpr;              /* 0                                               */
    double gpr_sigma;             /* 10    init_sigma  (IBACalib2.hpp:128)           */
    double gpr_l;                 /* 10    init_l                                    */
    double gpr_sigma_noise;       /* 1e-10 sigma_noise                               */
    /* Index option: precompute the local plane (k-NN, gates, PCA normal, regression error) of EVERY
     * scan point in stl_upload_pack.  The plane fit of ComputeAlignmentDist / BuildProblem is a pure
     * function of (scan, neighbour point, parameters) — it does not depend on the candidate — so it
     * can live in the index like the reference's KD-trees do; evaluations then only look it up.
     * Costs ~36 B per point and a longer upload; results are identical.  On by default; 0 fits every
     * plane at evaluation time (the reference's order of work). */
    int32_t plane_index;          /* 1                                               */
    /* Which BAError the evaluation follows.  0 = src/examples/iba_global.cpp (default).
     * 1 = src/examples/iba_global_stable.cpp: the 2-D queries are the re-projected map points of the
     * keypoints that observe one (:67-80, computed at upload from kp_mappoint and Tcw), a projected
     * scan point is kept when its ROUNDED pixel is inside the image (:92-94), and ComputeAlignmentDist
     * gates on k < 3 before the fit and on the neighbourhood extent after it (:154,:163-171).
     * stl_associate / stl_linearize_* are refused with variant 1 (iba_local.cpp has no such variant);
     * plane_index works with both (the index is then fitted with the stable flavour's gates). */
    int32_t variant;              /* 0                                               */
    /* use_gpr only: fit (sigma, l) of every GPR factor when it is created, as IBA_GPRFactor's constructor does
     * with GPRParams.optimize (IBACalib2.hpp:441-461 -> GPR::fit, GPR.hpp:350-387; IBALocalParams.optimize_gpr).
     * The fit runs on the host inside stl_associate (the reference keeps it on the CPU too); see stl_gpr_fit.
     * 0 keeps gpr_sigma / gpr_l for all factors. */
    int32_t gpr_optimize;         /* 0                                               */
    int32_t gpr_grad_flavour;     /* 0 analytic gradient, 1 the expressions of GPR.hpp:166-171 as coded */
} stl_params_t;

/*
 * KeyFramePack — everything the hot path reads, flattened (SURVEY.md §7.1).
 * All buffers are HOST memory owned by the caller; stl_upload_pack copies.
 * Matrices are row-major 3x4 [R|t].  float32 members are the float32 values
 * ORB-SLAM2 holds (KeyFrame.h:221,228; MapPoint.cc:84-87); scans are the
 * float32 values of the KITTI .bin files (io_tools.h:170-187).
 */
typedef struct stl_pack {
    int32_t n_kf;              /* keyframes in this pack (this rank's shard)        */
    int32_t n_covis;           /* covisible slots per keyframe, <= STL_MAX_COVIS    */
    const int64_t *scan_offset; /* [n_kf+1] first point of each scan in scan_xyz    */
    const float *scan_xyz;     /* [scan_offset[n_kf]][3] LiDAR-frame points         */
    const float *intrinsics;   /* [n_kf][4] fx, fy, cx, cy                          */
    const int32_t *image_wh;   /* [n_kf][2] mnMaxX, mnMaxY                          */
    const int64_t *kp_offset;  /* [n_kf+1] first keypoint of each keyframe          */
    const float *kp_xy;        /* [kp_offset[n_kf]][2] mvKeysUn[i].pt               */
    const float *kp_mappoint;  /* [kp_offset[n_kf]][3] MapPoint::GetWorldPos of the
                                  map point seen at this keypoint; x = NaN if none  */
    const float *Tcw;          /* [n_kf][12] KeyFrame::GetPose                      */
    const float *covis_relpose;/* [n_kf][n_covis][12] Tcw_j * Twc_ref, float32
                                  product, UNSCALED (iba_global.cpp:280)            */
    const uint8_t *covis_valid;/* [n_kf][n_covis] 1 if the slot holds a keyframe    */
    const float *covis_uv;     /* [kp_offset[n_kf]][n_covis][2] (u1,v1) of the keypoint
                                  matched in covisible slot c (GetMatchedKptIds,
                                  KeyFrame.cc:528); u1 = NaN if unmatched           */
    const float *he_Tc;        /* [n_kf][12] Tcw_{i+1} * Twc_i, float32 product
                                  (iba_global.cpp:267)                              */
    const double *he_Tl;       /* [n_kf][12] Twl_{i+1}^-1 * Twl_i (iba_global.cpp:269) */
    const uint8_t *he_valid;   /* [n_kf] 1 iff a next keyframe exists (Fi < F-1,
                                  iba_global.cpp:264); 0 for the globally last one  */
} stl_pack_t;

/*
 * Per-candidate sums returned by stl_eval_batch — exactly the accumulators of
 * BAError (iba_global.cpp:175-186).  Integer counters are carried as doubles
 * (exact below 2^53) so that one fp64 all-reduce covers the whole record.
 */
typedef struct stl_eval_sums {
    double sum_3d2d;    /* corr_3d_2d_err before the division  */
    double sum_3d3d;    /* corr_3d_3d_err before the division  */
    double sum_he;      /* Cval before the division            */
    double cnt_he;      /* Ccnt                                */
    double cnt_3d2d;    /* cnt_3d_2d                           */
    double valid_3d2d;  /* valid_cnt_3d_2d                     */
    double cnt_3d3d;    /* cnt_3d_3d                           */
    double valid_3d3d;  /* valid_cnt_3d_3d                     */
    double valid_pl;    /* valid_pl_3d_3d                      */
    double valid_pt;    /* valid_pt_3d_3d                      */
    double n_frames;    /* frames that passed the num_min_corr gate */
    double n_corr;      /* total 2-D correspondences over kept frames */
} stl_eval_sums_t;
#define STL_EVAL_NSUMS 12

/* What BAError returns (iba_global.cpp:330-343): f1, f2, C, valid, cnt. */
typedef struct stl_ba_error {
    double f1;              /* mean 3-D/2-D error  (DBL_MAX if no valid edge) */
    double f2;              /* mean 3-D/3-D error  (DBL_MAX if no valid edge) */
    double C;               /* mean hand-eye term                            */
    int32_t valid_cnt_3d_2d;
    int32_t cnt_3d_2d;
} stl_ba_error_t;

/*
 * Linearisation of the LM path: sum over all residual blocks of the Huber-
 * corrected cost, gradient J^T r and Gauss-Newton matrix J^T J w.r.t. the raw
 * 7 parameters [omega, upsilon, s] (VertexSim3 oplus is plain addition,
 * g2o_tools.h:21-24).  H is the full symmetric 7x7, row-major.
 */
typedef struct stl_lin_sums {
    double cost;     /* sum 0.5 * rho(||e||^2)                 */
    double g[7];     /* J^T r  (corrected)                     */
    double H[49];    /* J^T J  (corrected)                     */
    double n_blocks_2d; /* IBA_PlaneFactor blocks              */
    double n_blocks_pt; /* Point2Point_Factor blocks           */
    double n_blocks_pl; /* Point2Plane_Factor blocks           */
    double n_residuals; /* total scalar residuals              */
    double n_blocks_gpr; /* IBA_GPRFactor blocks               */
} stl_lin_sums_t;
#define STL_LIN_NSUMS 62

/* One LM iteration's worth of results for one parameter vector: the BAError accumulators followed by the
 * linearisation, contiguous so that ONE all-reduce covers both (stl_step_batch). */
typedef struct stl_step_sums {
    stl_eval_sums_t eval;
    stl_lin_sums_t lin;
} stl_step_sums_t;
#define STL_STEP_NSUMS (STL_EVAL_NSUMS + STL_LIN_NSUMS) /* 74 */

typedef struct stl_ctx stl_ctx_t;

/* ---- life cycle ------------------------------------------------------- */

/* Defaults = config/calib/00/iba_calib_global.yml:21-48. */
void stl_default_params(stl_params_t *p);

/* Creates a context on CUDA device `device` (one context per GPU / process).
 * Fails with STL_ERR_NO_DEVICE if the device is missing or not sm_100:
 * there is no CPU fallback.  Replaces BALoss's constructor state
 * (iba_global.cpp:349-361). */
stl_status_t stl_create(const stl_params_t *params, int32_t device, stl_ctx_t **out);
void stl_destroy(stl_ctx_t *ctx);
const char *stl_last_error(const stl_ctx_t *ctx);
int32_t stl_abi_version(void);

/* Copies the pack to HBM and builds the per-scan 3-D index (replaces the
 * KDTree3D-per-scan build, iba_global.cpp:362-367).  May be called again to
 * replace the pack.
 *
 * Size limits.  A scan holds at most 2^20 points, an image at most 16384 px
 * per side and a keyframe at most 65535 keypoints, but the binding rule is
 * tighter: the K1 tables of the largest keyframe must fit the device's opt-in
 * shared memory per block.  They take 26 B per keypoint (pixel, grid slot,
 * map-point bit, per-keypoint best match) plus the 2 px keypoint bitmap
 * (4 B x ceil((ceil(W/2) + 3) / 32) words x (ceil(H/2) + 3) rows), the 8 px
 * cell grid (2 B per cell) and 2.25 B per 128 points of the largest scan.
 * Measured on an NVIDIA B200 (227 KB opt-in shared memory, 1000 W power
 * limit), 2 keyframes of ~38 k-point scans: 1241 x 376 admits 7694 keypoints,
 * 1920 x 1080 admits 3782; a 3840 x 2160 image admits none (its bitmap alone
 * is 264 KB).  By default a pack over the limit is refused with
 * STL_ERR_CAPACITY and the previously uploaded pack stays in place; with
 * stl_allow_oversize_keyframes(ctx, 1) it is accepted (see there), and only
 * the 65535-keypoint, 16384 px and 2^20-point limits remain. */
stl_status_t stl_upload_pack(stl_ctx_t *ctx, const stl_pack_t *pack);

/* Oversize keyframes.  allow = 1 lets the NEXT stl_upload_pack accept keyframes
 * whose K1 tables do not fit the shared memory of the one-kernel K1; they run
 * on a banded three-kernel K1 whose shared memory does not grow with the image
 * (DESIGN.md §3 "Oversize keyframes"), with bit for bit the results the
 * one-kernel K1 would give.  allow = 0 (the default) refuses such a pack as
 * before.  The call does not touch the resident pack; allow other than 0 / 1
 * -> STL_ERR_INVALID.
 *
 * Routing rule.  The one-kernel K1 keeps a "fitting" set of keyframes whose
 * maxima of keypoints, table bytes and 128-point groups fit the opt-in limit
 * (a sum of maxima, not a maximum of sums).  Keyframes leave that set
 * largest-first, by the shared memory each would need alone (ties: the lower
 * index first), until the set's maxima fit; those that left are the oversize
 * keyframes.  With none the fitting set is the whole pack and nothing changes.
 *
 * Cost: each band of bitmap rows (floor(4096 / words per row) rows, at most
 * 16 KB) streams the scan cells that can project into it, and the K1 keeps its
 * per-keypoint tables, survivors and matches in a workspace sized per
 * (candidate, oversize keyframe): 16 B per keypoint, and per keyframe
 * S = max(4096, min(2 n_kp rounded up to 256, padded scan points)) survivor
 * slots of 4 B and 2 S match slots of 16 B.  A unit that finds more survivors
 * than S falls back to the exact pass over every point (correct, slower;
 * work counter [6]). */
stl_status_t stl_allow_oversize_keyframes(stl_ctx_t *ctx, int32_t allow);

/* Local keyframes of the resident pack that run on the oversize path, in
 * increasing order: up to `cap` of them into kf (may be NULL), their count in
 * *n (even if > cap).  No pack -> STL_ERR_STATE. */
stl_status_t stl_oversize_keyframes(stl_ctx_t *ctx, int32_t *kf, int32_t cap, int32_t *n);

/* ---- Nomad / iba_func path ------------------------------------------- */

/* Evaluates B candidates x[b][7] = [omega, upsilon, s] (Sim3 log as BAError's
 * xvec, iba_global.cpp:188) over this context's keyframes.  HOST in, HOST out;
 * blocking; thread-safe (internally serialised — Nomad calls eval_x from
 * several threads).  sums[b] are this pack's partial sums: with one GPU they
 * are the totals, with keyframe sharding they are all-reduced by the caller
 * (see stl_eval_batch_device). */
stl_status_t stl_eval_batch(stl_ctx_t *ctx, const double *x, int32_t B, stl_eval_sums_t *sums);

/* Same, but leaves the [B][STL_EVAL_NSUMS] fp64 record in DEVICE memory
 * `d_sums` on CUDA stream `stream` (a cudaStream_t; NULL = the context's own
 * stream) without synchronising: the caller all-reduces it (NCCL, sum) and
 * then finalises.  x is HOST memory. */
stl_status_t stl_eval_batch_device(stl_ctx_t *ctx, const double *x, int32_t B, double *d_sums,
                                   void *stream);

/* BAError's epilogue (iba_global.cpp:330-343): sums -> (f1, f2, C, valid, cnt). */
void stl_finalize(const stl_params_t *params, const stl_eval_sums_t *sums, stl_ba_error_t *out);

/* BALoss::eval_x's epilogue (iba_global.cpp:386-388): bbo = {f, C1, C2, C3}. */
void stl_bbo(const stl_params_t *params, const stl_ba_error_t *e, double bbo[4]);

/* ---- Ceres / g2o (LM) path -------------------------------------------- */

/* BuildProblem (iba_local.cpp:145-323): associates at x0[7] and freezes the
 * residual blocks (plane / point-to-point / point-to-plane) on the device.
 * n_blocks[4] receives the block counts {plane 2d, pt, pl, gpr 2d} of this pack; passing NULL makes the
 * call asynchronous (nothing waits on the host; stl_block_counts fetches the numbers later).
 * When x0 is bitwise one of the candidates of the immediately preceding stl_eval_batch, its 2-D
 * correspondences are reused instead of streaming the scans a second time (the reference evaluates
 * BAError(x) and BuildProblem(x) back to back at the same x, iba_global.cpp:201 / iba_local.cpp:191). */
stl_status_t stl_associate(stl_ctx_t *ctx, const double *x0, int64_t n_blocks[4]);

/* Evaluates the frozen blocks at B parameter vectors: cost, J^T r, J^T J
 * (Ceres semantics: Huber via residual/Jacobian rescaling). */
stl_status_t stl_linearize_batch(stl_ctx_t *ctx, const double *x, int32_t B, stl_lin_sums_t *out);
stl_status_t stl_linearize_batch_device(stl_ctx_t *ctx, const double *x, int32_t B, double *d_out,
                                        void *stream);

/* Per-block view of one evaluation, for solvers that want residual blocks rather than normal equations
 * (ceres::CostFunction::Evaluate of IBA_PlaneFactor / Point2Point_Factor / Point2Plane_Factor /
 * IBA_GPRFactor, IBACalib2.hpp:152-184,472-507,570-625; g2o IBAPlaneEdge computeError + linearizeOplus,
 * IBACalib.hpp:103-155): for every frozen block its type (0 plane 3-D/2-D, 1 point-to-point,
 * 2 point-to-plane, 3 GPR), keyframe, keypoint, residual count, the RAW residuals (no robust kernel:
 * the solver applies its own HuberLoss) and their Jacobian rows with respect to the 7 parameters,
 * row-major [block][rmax][7] with a fixed stride of `rmax` rows (>= max(3, 2 * n_covis); g2o's edge is
 * the same layout with rmax = 20).  Blocks are ordered plane, then 3-D/3-D, then GPR, each in keyframe
 * order.  All buffers are host memory sized for `cap_blocks`; *n_blocks_out receives the count. */
stl_status_t stl_eval_blocks(stl_ctx_t *ctx, const double *x, int32_t rmax, int64_t cap_blocks, int32_t *type, int32_t *kf,
                             int32_t *kp, int32_t *n_res, double *residuals, double *jacobians, int64_t *n_blocks_out);

/* ---- GPR hyper-parameters (host; no context, no GPU) -------------------------------------------------
 * The objective of GPR::fit — GPRHyperLoss::Evaluate (GPR.hpp:154-174): negative log marginal likelihood of the
 * depths y[n] observed at pixels x[n][2] under K = sigma^2 exp(-D / 2 l^2) + sigma_noise I — and its gradient
 * with respect to (sigma, l).  flavour 0: the derivative of that objective; flavour 1: the expressions of
 * GPR.hpp:166-171,218-222 exactly as written (dK/dsigma = 2 sigma Kff with the full Kff, dK/dl = (Kff * Dist) / l^3
 * as a matrix product).  Returns STL_ERR_INVALID if the Cholesky factorisation fails (Evaluate returns false). */
stl_status_t stl_gpr_nlml(const double *x, const double *y, int32_t n, double sigma_noise, double sigma, double l, int32_t flavour,
                          double *cost, double grad[2]);
/* GPR::fit (GPR.hpp:350-387): at most max_iter (15 in the reference) quasi-Newton iterations on the objective above
 * from (sigma0, l0).  out = {sigma, l, cost at the start, cost at the end, iterations, objective evaluations}.
 * The reference drives the same objective with ceres::GradientProblemSolver (L-BFGS); its iterate path is not
 * reproducible without Ceres — see csrc/gprfit.hpp. */
stl_status_t stl_gpr_fit(const double *x, const double *y, int32_t n, double sigma_noise, double sigma0, double l0, int32_t max_iter,
                         int32_t flavour, double out[6]);
/* (sigma, l) of the GPR blocks of the last association, in block order ([n_blocks[3]][2]); the per-problem values
 * unless params.gpr_optimize fitted them. */
stl_status_t stl_gpr_hyper(stl_ctx_t *ctx, double *sigma_l, int64_t cap_blocks);

/* Block counts {plane 2d, pt, pl, gpr 2d} of the last association of this context (waits for it). */
stl_status_t stl_block_counts(stl_ctx_t *ctx, int64_t n_blocks[4]);

/* ---- several starts: a PROBLEM SET ------------------------------------------------------------------------
 * Multi-start refinement (refine the best few points of a NOMAD run, or run iba_local from several perturbed initial
 * extrinsics, iba_local.cpp:145-323,434-460) on ONE context: the context freezes P independent BuildProblems, problem p
 * associated at its own x0[p], and evaluates candidate b on the problem it names.  stl_associate(x0) is
 * stl_associate_multi(x0, 1, NULL); every single-problem call keeps its results and meaning on a set of one, and returns
 * STL_ERR_STATE (naming the multi call) while the set holds more than one problem — stl_associate (or stl_step_batch
 * with reassociate != 0) freezes a set of one again.
 * Problem p gives bit for bit what a fresh stl_associate(x0[p]) followed by stl_linearize_batch gives: the same block
 * counts and the same [62] record, whatever P, whichever problems share the call and however the workspace chunks it.
 * With a communicator attached the [B][62] / [P][74] record is exchanged once, like the other records; block counts are
 * this rank's.  Errors: P < 1, a problem index outside [0, P), or a rebuild mask with P different from the size of the
 * frozen set -> STL_ERR_INVALID; P > STL_MAX_PROBLEMS -> STL_ERR_CAPACITY; variant 1 -> STL_ERR_STATE (as stl_associate).
 * A failed allocation leaves no set (the next call starts over). */
#define STL_MAX_PROBLEMS 256   /* = the candidate cap of the evaluation workspace and of the peer-memory record exchange */

/* BuildProblem at x0[p] for p < P (x0 [P][7]).
 * rebuild == NULL: the set is replaced by P new problems.
 * rebuild != NULL: P must equal the current set size; only problems with rebuild[p] != 0 are re-associated (at x0[p]); the
 *   others keep their blocks bit for bit.
 * The 2-D association of the starts comes from the workspace when the preceding evaluation left exactly those x0 there (as
 * stl_associate); all rebuilt problems are associated by the same kernel launches, chunk by chunk of the workspace.
 * With params.gpr_optimize the hyper-parameter fit runs once per rebuilt problem.
 * n_blocks [P][4] as in stl_associate; NULL = asynchronous (read them with stl_block_counts_multi). */
stl_status_t stl_associate_multi(stl_ctx_t *ctx, const double *x0, int32_t P, const uint8_t *rebuild, int64_t *n_blocks);
/* Block counts [P][4] of every problem of the set (waits for the association); cap_problems < P -> STL_ERR_CAPACITY. */
stl_status_t stl_block_counts_multi(stl_ctx_t *ctx, int64_t *n_blocks, int32_t cap_problems);

/* cost, J^T r, J^T J of candidate b (x [B][7]) on problem problem[b] (NULL: B == P and candidate b on problem b), as
 * stl_linearize_batch; the _device twin leaves the [B][62] record in DEVICE memory on `stream`. */
stl_status_t stl_linearize_multi(stl_ctx_t *ctx, const double *x, int32_t B, const int32_t *problem, stl_lin_sums_t *out);
stl_status_t stl_linearize_multi_device(stl_ctx_t *ctx, const double *x, int32_t B, const int32_t *problem, double *d_out, void *stream);

/* One LM iteration for each of P starts (x [P][7]): BAError sums at x[p], BuildProblem at x[p] for the problems flagged in
 * rebuild (NULL = all, which makes a new set), linearisation of problem p at x[p]; ONE [P][74] record, exchanged once.
 * Same bits as stl_eval_batch + stl_associate_multi + stl_linearize_multi.  P = 1 is stl_step_batch(x, 1, rebuild ?
 * rebuild[0] : 1) with its second-stream overlap; a larger set runs the stages one after another on one stream. */
stl_status_t stl_step_multi(stl_ctx_t *ctx, const double *x, int32_t P, const uint8_t *rebuild, stl_step_sums_t *out);
stl_status_t stl_step_multi_device(stl_ctx_t *ctx, const double *x, int32_t P, const uint8_t *rebuild, double *d_out, void *stream);

/* BAError + (optionally) BuildProblem + linearisation in one call — what one LM / g2o iteration at x asks
 * for (iba_local.cpp:434-446 with the BAError value iba_global.cpp:169 logged beside it), or, for a NOMAD
 * poll batch, the cost record and the normal equations of every candidate on the frozen association:
 *   1. the BAError sums of x[0..B)                                        (as stl_eval_batch)
 *   2. reassociate != 0: BuildProblem at x[0], REUSING the 2-D association step 1 just computed for it
 *      (FindProjectCorrespondences at the same extrinsic, iba_global.cpp:201 == iba_local.cpp:191)
 *   3. cost, J^T r, J^T J of the frozen blocks at x[0..B)                  (as stl_linearize_batch)
 * Nothing waits on the host between the stages; with a communicator attached the [B][74] record is
 * all-reduced ONCE.  out[b] = {eval sums, linearisation} of candidate b.
 * With the plane index (the default) stages 2 and 3 run on a second stream of the context beside the 3-D stage of
 * step 1 — BuildProblem needs the 2-D association and the map-point 1-NN of step 1, not its sums — and the map-point
 * 1-NN of BuildProblem is answered inside step 1's search kernel; both streams are joined before the call returns
 * its stream to the caller, so the ordering a caller sees is that of ONE stream.  Same bits as the three calls made
 * one after another. */
stl_status_t stl_step_batch(stl_ctx_t *ctx, const double *x, int32_t B, int32_t reassociate, stl_step_sums_t *out);
/* Same; the [B][STL_STEP_NSUMS] record stays in DEVICE memory `d_out` on `stream`, no synchronisation. */
stl_status_t stl_step_batch_device(stl_ctx_t *ctx, const double *x, int32_t B, int32_t reassociate, double *d_out, void *stream);

/* ---- the two optimisation problems that precede the cost evaluation, on the same 7 parameters (SURVEY 8f N4) ----
 * Hand-eye initialisation, HECalibRobustKernelg2o / HECalibLineProcessg2o (include/NLHECalib.hpp:118-278): one EdgeHE per
 * motion pair (camera motion Ta, LiDAR motion Tb; :27-86) plus the EdgeRegulation on the translation parameters (:88-116).
 * For B parameter vectors x the call returns, in stl_lin_sums_t: cost = sum rho(chi2) (g2o's robust chi2, no factor 1/2),
 * g = J^T rho' Omega e (g2o's b is -g), H = J^T rho' Omega J, n_blocks_2d = edges, n_residuals.  chi2 (optional,
 * [B][n]) receives every edge's e^T Omega e — HECalibLineProcessg2o re-weights its edges from them (:230-241). */
typedef struct stl_he_edges {
    int32_t n;
    const double *Ta;      /* [n][12] camera motions, 3x4 row-major [R|t]                      */
    const double *Tb;      /* [n][12] LiDAR motions                                              */
    const double *info;    /* [n] information scale of each edge (information = info * I); NULL = 1 */
    double huber_delta;    /* g2o::RobustKernelHuber delta (robust_kernel_size, :141-143); <= 0: none */
    double regulation;     /* information scale of the regularisation edge (n * regulation_ratio, :148-150); 0: no such edge */
} stl_he_edges_t;
stl_status_t stl_he_linearize(stl_ctx_t *ctx, const stl_he_edges_t *edges, const double *x, int32_t B, stl_lin_sums_t *out, double *chi2);

/* Calibration bundle adjustment, Optimizer::OptimizeExtrinsicGlobal / Local (src/orb_slam/src/Optimizer.cc:1399-1744):
 * one calibEdge (:65-205) per (keyframe, observed map point): the map point (already in the frame of the first / oldest
 * keyframe) is scaled, taken to the LiDAR frame with the inverse extrinsic, moved by the LiDAR pose of the keyframe,
 * brought back with the extrinsic and projected; error = observation - projection, information = invSigma2 * I,
 * Huber delta = sqrt(5.991).  `level` mirrors setLevel (1 = left out as an outlier, :1513-1524).  Same outputs as
 * stl_he_linearize; chi2 is [B][n_edges] and is also filled for level-1 edges (the reference re-evaluates them, :1509). */
typedef struct stl_calib_edges {
    int32_t n_kf;
    int64_t n_edges;
    const int64_t *edge_offset; /* [n_kf+1] first edge of each keyframe                          */
    const double *Tlw_quat;     /* [n_kf][6] rotation vector and translation of calibEdge::Tlw_quat */
    const float *intrinsics;    /* [n_kf][4] fx, fy, cx, cy                                         */
    const double *Xw;           /* [n_edges][3] calibEdge::Xw                                       */
    const double *obs;          /* [n_edges][2] measurement (undistorted keypoint)                  */
    const float *inv_sigma2;    /* [n_edges] mvInvLevelSigma2[octave]                               */
    const uint8_t *level;       /* [n_edges] or NULL (all active)                                   */
    double huber_delta;
} stl_calib_edges_t;
stl_status_t stl_calib_linearize(stl_ctx_t *ctx, const stl_calib_edges_t *edges, const double *x, int32_t B, stl_lin_sums_t *out, double *chi2);

/* ---- multi-GPU: keyframes sharded over the GPUs of a node (SURVEY.md 8e) -----------------------------
 * One process (or thread) per GPU, each with its own context holding a contiguous block of keyframes
 * (stl_pack_t.n_kf = this rank's shard; covisible data is baked per keyframe, so there is no halo).
 * The only exchange of the path is the sum the reference forms over keyframes
 * (iba_global.cpp:239-251,274-275,318-326): once a communicator is attached, stl_eval_batch,
 * stl_linearize_batch, stl_step_batch and their _device twins finish with ONE ncclAllReduce(sum, fp64) of
 * the [B][12 | 62 | 74] record on the compute stream, and every rank returns the totals.  Every rank must
 * make the same calls with the same x and B.  stl_associate / stl_block_counts report this rank's blocks. */
#define STL_COMM_ID_BYTES 128
/* ncclGetUniqueId: called by one rank; the bytes are handed to the others by the host program (MPI,
 * torch.distributed, a file ...) before stl_comm_init. */
stl_status_t stl_comm_unique_id(uint8_t id[STL_COMM_ID_BYTES]);
/* ncclCommInitRank on the context's device; the context owns the communicator (stl_destroy releases it). */
stl_status_t stl_comm_init(stl_ctx_t *ctx, const uint8_t id[STL_COMM_ID_BYTES], int32_t rank, int32_t n_ranks);
/* rank / size of the attached communicator (0 / 1 when none). */
stl_status_t stl_comm_info(stl_ctx_t *ctx, int32_t *rank, int32_t *n_ranks);
/* How the records are exchanged: out[0] = 1 when every rank could map every other rank's receive buffer (cudaIpc peer
 * memory over NVLink): the kernel that finishes a record then also sums it over the ranks, in rank order, with no separate
 * collective launch (csrc/p2p.cuh); 0 = ncclAllReduce after the last kernel (also used for batches over 256 candidates;
 * STL_NO_P2P=1 forces it).  out[1] = exchanges done through peer memory so far, out[2] = through NCCL. */
stl_status_t stl_comm_stats(stl_ctx_t *ctx, int64_t out[3]);

/* ---- keyframe selection on the resident pack ---------------------------------------------------------
 * A context can restrict every call that walks keyframes to a subset of its pack without a second upload: coarse-to-fine
 * search on every k-th keyframe, a hold-out check, dropping keyframes with moving objects, or the reference's
 * single-frame caller (iba_single_frame.cpp, keyframe 0 only).
 *
 * kf[n]: LOCAL keyframe indices of this context's pack, strictly increasing, inside [0, n_kf); n = 0 (nothing selected) is
 * allowed (kf must then still be non-null).  kf == NULL selects every keyframe: the default, restored by every stl_upload_pack.
 * An invalid list returns STL_ERR_INVALID and leaves the selection as it was; without a pack the call returns STL_ERR_STATE; a
 * CUDA failure returns STL_ERR_CUDA with every keyframe selected.
 *
 * While a selection is set, stl_eval_batch, stl_associate(_multi), stl_step_batch, stl_step_multi (and their _device
 * twins), stl_eval_blocks, the GPR fit, the work counters and the debug getters behave exactly as a context whose pack
 * holds only the selected keyframes' rows (KeyFramePack.select): the same records, bit for bit, and the same block counts.
 * Keyframe f keeps its own rows, among them its hand-eye pair (f, f+1) as he_valid bakes it, whether or not f+1 is
 * selected.  Keyframe indices the library reports (stl_eval_blocks' kf) remain the pack's own.  The debug getters read an
 * unselected keyframe as empty (n = 0, a zero record); stl_knn3d is unaffected.
 *
 * A selection call DROPS the frozen problem set, the reuse of the last evaluation's 2-D association and the batch the
 * debug getters refer to: stl_linearize_*, stl_eval_blocks, stl_block_counts, stl_gpr_hyper and stl_step_* without
 * re-association return STL_ERR_STATE until the next association.
 *
 * With a communicator attached the indices are local to the rank's shard, and every rank must still make every call (with
 * n = 0 where it selects nothing); the record exchange is unchanged. */
stl_status_t stl_select_keyframes(stl_ctx_t *ctx, const int32_t *kf, int32_t n);

/* BAError per keyframe: evaluates B candidates like stl_eval_batch (the same kernels, one workspace chunk at a time) and
 * returns, for every keyframe of the pack, the 13-value record of stl_debug_frame in its order,
 * out[B][n_kf][13] = {sum_3d2d, valid_3d2d, cnt_3d2d, sum_he, cnt_he, kept, n_corr, n_queries,
 *                     sum_3d3d, valid_3d3d, cnt_3d3d, valid_pl, valid_pt}.
 * Rows of unselected keyframes are zero.  With err_weight[1] <= 1e-10 the 3-D columns hold what the record counts for the
 * frame (valid_3d3d = cnt_3d3d = kept, the rest 0), so that the rows of a candidate always sum to its stl_eval_batch
 * record (counters exactly; sums up to the order of the fp64 additions).  There is no exchange: every rank returns its
 * own keyframes.  Like stl_eval_batch, the call leaves its batch to the debug getters and its 2-D association to a
 * following stl_associate at one of its candidates. */
stl_status_t stl_eval_frames(stl_ctx_t *ctx, const double *x, int32_t B, double *out);

/* ---- debug getters (parity tests only) --------------------------------- */

/* 2-D correspondences of keyframe `kf` for the candidate at index `b` of the
 * LAST stl_eval_batch call (FindProjectCorrespondences' corrset,
 * iba_global.cpp:55-96).  Writes up to `cap` pairs ordered by keypoint index;
 * returns the pair count in *n (even if > cap). */
stl_status_t stl_debug_corrset(stl_ctx_t *ctx, int32_t b, int32_t kf, uint32_t *kp_idx,
                               uint32_t *pt_idx, int32_t cap, int32_t *n);

/* Per-query 3-D results of the LAST stl_eval_batch for (b, kf)
 * (ComputeAlignmentDist, iba_global.cpp:111-156): for each correspondence that
 * has a map point, in corrset order: nn index, neighbour count after radius
 * truncation, is_plane, dist.  knn_idx (optional) is [cap][32] neighbour
 * indices in distance order. */
stl_status_t stl_debug_align(stl_ctx_t *ctx, int32_t b, int32_t kf, uint32_t *kp_idx,
                             uint32_t *nn_idx, int32_t *n_neigh, int32_t *is_plane, double *dist,
                             uint32_t *knn_idx, int32_t cap, int32_t *n);

/* Per-keyframe partial record of the LAST stl_eval_batch for (b, kf):
 * out = {sum_3d2d, valid_3d2d, cnt_3d2d, sum_he, cnt_he, kept, n_corr, n_queries,
 *        sum_3d3d, valid_3d3d, cnt_3d3d, valid_pl, valid_pt}. */
stl_status_t stl_debug_frame(stl_ctx_t *ctx, int32_t b, int32_t kf, double out[13]);

/* Stand-alone exact k-NN over scan `kf` (nanoflann findNeighbors,
 * nanoflann.hpp:1588): nq queries q[nq][3] (fp64), k <= 32, radius2 <= 0 means
 * unbounded.  out_idx/out_d2 are [nq][k] sorted ascending by (d2, index);
 * unused slots hold 0xFFFFFFFF / +inf.  HOST in, HOST out. */
stl_status_t stl_knn3d(stl_ctx_t *ctx, int32_t kf, const double *q, int32_t nq, int32_t k,
                       double radius2, uint32_t *out_idx, double *out_d2, int32_t *out_count);

/* The two transcendental calls of the plane fit (std::acos, std::cos in FastEigen3x3_EV, pointcloud.h:404-407) as the
 * device evaluates them — correctly rounded, csrc/crmath.cuh — element-wise on x[n] (acos on x clamped to [-1, 1]).
 * For the parity test against the host libm. */
stl_status_t stl_debug_trig(stl_ctx_t *ctx, const double *x, int32_t n, double *acos_out, double *cos_out);

/* ---- measurement -------------------------------------------------------- */

#define STL_STAGE_ASSOC2D 0  /* K1 transform + project + 2-D association      */
#define STL_STAGE_KNN3D 1    /* K2 3-D 1-NN + k-NN + PCA + gates              */
#define STL_STAGE_REDUCE 2   /* K3 per-candidate reduction                    */
#define STL_STAGE_LINEARIZE 3
#define STL_STAGE_BUILD 4    /* one-off index build of stl_upload_pack        */
#define STL_STAGE_ASSOC_LM 5 /* BuildProblem kernels of stl_associate / stl_step_batch */
#define STL_STAGE_ALLREDUCE 6 /* the NCCL all-reduce of the record (communicator attached) */
#define STL_STAGE_PLANE_INDEX 7 /* plane index part of the build (params.plane_index)  */
#define STL_NSTAGES 8

/* Sets the CUDA stream (a cudaStream_t) on which the calls WITHOUT an explicit stream argument
 * enqueue their work (NULL = the context's own stream).  A context's calls share one workspace:
 * whenever the stream changes from one call to the next, the library makes the new stream wait
 * for the work already queued on the previous one. */
stl_status_t stl_set_stream(stl_ctx_t *ctx, void *stream);

/* When enabled, every stage launch is bracketed by CUDA events on its stream;
 * stl_stage_stats returns accumulated milliseconds / launch counts since the
 * last reset and resets them. */
stl_status_t stl_set_profiling(stl_ctx_t *ctx, int32_t enabled);
stl_status_t stl_stage_stats(stl_ctx_t *ctx, double ms[STL_NSTAGES], int64_t launches[STL_NSTAGES]);

/* Work counters of the last stl_eval_batch or stl_eval_frames (host-side, summed over b):
 * [0] points streamed by K1, [1] 2-D 1-NN queries (= keypoints),
 * [2] 3-D 1-NN queries, [3] 3-D k-NN queries, [4] algorithmic bytes of K1,
 * [5] kernels of this library launched by the context since its creation,
 * [6] (candidate, keyframe) units whose K1 survivor list overflowed and that fell back to the exact
 *     evaluation of every point (cumulative; 0 at the reference's 1.5 px association radius),
 * [7] associations that reused the 2-D correspondences of a preceding evaluation at the same x (cumulative). */
stl_status_t stl_work_counters(stl_ctx_t *ctx, double out[8]);

#ifdef __cplusplus
}
#endif
#endif /* STLCALIB_H_ */
