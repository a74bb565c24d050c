/* tvf.h -- C ABI of libtvf.so: batched linear three-view pose estimation on
 * NVIDIA B200 (sm_100a), a drop-in for the linear hot path of
 * LauraFJulia/TFT_vs_Fund.  Every entry point below replaces one MATLAB
 * function of the reference (file:line cited per function); B = 1 reproduces
 * the reference signature exactly, B > 1 is the batched superset.
 *
 * Conventions
 *   - all data FP64, MATLAB column-major, caller-owned buffers;
 *   - a batch is the trailing dimension: `Corresp` is 6 x n x B (48 contiguous
 *     bytes per point), `CalM` 9 x 3 (shared) or 9 x 3 x B, poses 3 x 4 x B,
 *     tensors 3 x 3 x 3 x B, `Reconst` 3 x n x B;
 *   - plain pointers and sizes only; no exceptions cross the boundary;
 *   - return value: < 0 argument/runtime error (tvf_last_error() has the text),
 *     0 success, > 0 number of problems whose status word is non-zero;
 *   - `status` (int32 per problem, may be NULL) is a bit set, see TVF_ST_*;
 *   - one handle per host thread; a handle drives one GPU (tvf_create) or several
 *     (tvf_create_multi: the host-pointer batched calls shard the batch over the
 *     devices); calls on a handle are serialised by the caller (MATLAB calls MEX on
 *     its interpreter thread only);
 *   - there is no CPU fallback: without a CUDA device tvf_create() fails.
 *
 * Results agree with the reference up to the sign/scale freedom the reference
 * itself leaves open: T and F up to sign (unit Frobenius norm / arbitrary
 * scale), triangulated homogeneous points up to sign.
 */
#ifndef TVF_H_
#define TVF_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct tvf_context* tvf_handle_t;

/* return codes */
#define TVF_OK 0
#define TVF_ERR_ARG (-1)            /* bad pointer / size / unsupported shape            */
#define TVF_ERR_CUDA (-2)           /* CUDA runtime error                                */
#define TVF_ERR_TOO_FEW_POINTS (-3) /* linearF.m:35-37: N < 8 (or N mismatch)            */
#define TVF_ERR_NOMEM (-4)

/* per-problem status bits */
#define TVF_ST_EIG_NOCONV 1    /* inverse iteration hit its cap: the design matrix has no usable spectral gap */
#define TVF_ST_EPIPOLE_ZERO 2  /* sign(V(end)) == 0 at R_t_from_TFT.m:50,55                                   */
#define TVF_ST_NO_POSE_2 4     /* all 4 cheirality votes < 0 or NaN: MATLAB leaves R_f undefined (:91-104)    */
#define TVF_ST_NO_POSE_3 8
#define TVF_ST_NONFINITE 16    /* non-finite value in R_t / reprojection error                                */
#define TVF_ST_BA_NOCONV 32    /* tvf_bundle_adjust: iteration cap reached before the stopping rule held          */
#define TVF_ST_COV_SINGULAR 64 /* tvf_ba_covariance: reduced camera system or a point block not positive definite:
                                  covariance undefined                                                            */

/* the message linearF.m:36 raises; gateways re-raise it verbatim */
#define TVF_LINEARF_ERRMSG \
    "At least 8 correspondences are necessary to compute the fundamental matrix linearly\\n"

/* ---- lifetime ------------------------------------------------------------------------- */
int tvf_version(void);
int tvf_device_count(void);
int tvf_create(tvf_handle_t* out, int device);
/* Group handle over n_dev devices (ids may repeat: two members on one GPU are legal).  Member 0 serves every entry
 * point; the host-pointer batched calls -- pose (tvf_pose, tvf_linear_tft_pose, tvf_linear_f_pose, tvf_optim_f_pose),
 * bundle adjustment (tvf_bundle_adjust) and covariance (tvf_ba_covariance) -- split B into n_dev contiguous ranges,
 * one host thread + one device per range, no exchange between them -- the batched
 * form of the trial loop experiments.m:91-143 / experiments_real.m:75-163.  Results are bit-identical to a one-device call. */
int tvf_create_multi(tvf_handle_t* out, const int* devices, int n_dev);
int tvf_num_devices(tvf_handle_t h);
void tvf_destroy(tvf_handle_t h);
const char* tvf_last_error(tvf_handle_t h); /* h may be NULL: error of the last failed tvf_create */
int tvf_device(tvf_handle_t h);
/* problems per internal chunk (work-space size / pipelining granularity); 0 restores the default */
int tvf_set_chunk(tvf_handle_t h, int64_t problems);
/* stream used by the *_dev entry points: a cudaStream_t (NULL = the legacy default stream).
 * Until this is called -- and again after tvf_use_own_stream() -- the handle's own stream is used. */
int tvf_set_stream(tvf_handle_t h, void* cuda_stream);
int tvf_use_own_stream(tvf_handle_t h);
int tvf_synchronize(tvf_handle_t h);
/* pinned host memory, so the host-pointer entry points overlap copies with compute; placed on the NUMA node of the
 * calling thread's current CUDA device (the thread's CPU affinity is narrowed during the call and restored) */
void* tvf_host_alloc(size_t bytes);
void tvf_host_free(void* p);
/* on != 0: caller buffers >= 1 MiB that are pageable (an mxArray's data) are page-locked with cudaHostRegister for the
 * duration of each host-pointer batched call (pose, bundle adjustment, covariance) and released before it returns;
 * off (default): pageable buffers are staged as tvf_set_host_threads describes */
int tvf_set_host_register(tvf_handle_t h, int on);
/* Pageable caller buffers of the host-pointer batched calls (pose, bundle adjustment, covariance) are otherwise staged
 * chunk by chunk through pinned per-slot buffers, filled and drained by `threads` host threads (0 = automatic: hardware
 * threads / devices of the handle, clamped to 2..8), so the copies still overlap the kernels.  Pinned buffers
 * (tvf_host_alloc, cudaHostRegister) are used in place. */
int tvf_set_host_threads(tvf_handle_t h, int threads);

/* ---- method entry points (host pointers; copies are inside the call) ------------------- */

/* [R_t_2,R_t_3,Reconst,T,iter] = LinearTFTPoseEstimation(Corresp,CalM)
 * TFT_methods/LinearTFTPoseEstimation.m:1,45-62 (iter is the constant 0 and is not returned here).
 * corresp 6 x n x B; calm 9 x 3 (calm_batched = 0) or 9 x 3 x B (1).
 * Outputs (any may be NULL): Rt2, Rt3 3x4xB; reconst 3 x n x B; T 3x3x3xB (pixel coordinates,
 * unit Frobenius norm); repr_err B = ReprError({K1[I|0],K2*R_t_2,K3*R_t_3},Corresp,Reconst)
 * (auxiliar_functions/ReprError.m:39-65, what experiments.m:112-114 evaluates next). */
int tvf_linear_tft_pose(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n,
                        int64_t B, double* Rt2, double* Rt3, double* reconst, double* T, double* repr_err,
                        int32_t* status);

/* [R_t_2,R_t_3,Reconst,T,iter] = LinearFPoseEstimation(Corresp,CalM)
 * F_methods/LinearFPoseEstimation.m:1,42-78.  Same arguments; T = TFT_from_P(...) (:78).
 * F21, F31 (3x3xB each, may be NULL) expose the fundamental matrices of :55-56.
 * n < 8 returns TVF_ERR_TOO_FEW_POINTS (linearF.m:35-37). */
int tvf_linear_f_pose(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n,
                      int64_t B, double* Rt2, double* Rt3, double* reconst, double* T, double* repr_err,
                      double* F21, double* F31, int32_t* status);

/* [R_t_2,R_t_3,Reconst,T,iter] = OptimFPoseEstimation(Corresp,CalM)
 * F_methods/OptimFPoseEstimation.m:1,43-72: both fundamental matrices refined by optimF (Gauss-Helmert
 * minimisation of the reprojection error, Optimization/Gauss_Helmert.m:38-83), then the pose tail of the F method.
 * Same arguments as tvf_linear_f_pose plus iter (B, may be NULL) = it1 + it2 of :49.  F21, F31: the refined
 * matrices of :47-48.  n < 8 -> TVF_ERR_TOO_FEW_POINTS; n > tvf_optim_f_max_n() -> TVF_ERR_ARG (the reference
 * itself forms dense 4N x 4N matrices there). */
int tvf_optim_f_pose(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n,
                     int64_t B, double* Rt2, double* Rt3, double* reconst, double* T, double* repr_err,
                     double* F21, double* F31, int32_t* iter, int32_t* status);
int tvf_optim_f_max_n(void);

/* Generic form of the three method entry points above, with every optional output in one place.
 * method: 1 = LinearTFTPoseEstimation, 7 = LinearFPoseEstimation, 8 = OptimFPoseEstimation (numbering of
 * experiments.m:51-59).  votes (10 x B int32): what recover_R_t computed at R_t_from_TFT.m:91-104 /
 * LinearFPoseEstimation.m:94-107 -- per problem the four cheirality votes of view pair (1,2) in the reference's
 * candidate order (R,t),(R,-t),(Rp,-t),(Rp,t), the four of pair (1,3), then one bit mask per pair of the candidates
 * whose vote is NaN (bit k = candidate k; MATLAB's NaN >= x is false).  Any member may be NULL. */
typedef struct tvf_pose_out {
    double* Rt2;      /* 3 x 4 x B */
    double* Rt3;      /* 3 x 4 x B */
    double* reconst;  /* 3 x n x B */
    double* T;        /* 3 x 3 x 3 x B */
    double* repr_err; /* B */
    double* F21;      /* 3 x 3 x B (methods 7, 8) */
    double* F31;      /* 3 x 3 x B (methods 7, 8) */
    int32_t* iter;    /* B (method 8) */
    int32_t* votes;   /* 10 x B */
    int32_t* status;  /* B */
} tvf_pose_out;
int tvf_pose(tvf_handle_t h, int method, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
             const tvf_pose_out* out);
/* same with device pointers (corresp, calm and every member of out), asynchronous like the other *_dev forms */
int tvf_pose_dev(tvf_handle_t h, int method, const double* corresp, const double* calm, int calm_batched, int n,
                 int64_t B, const tvf_pose_out* out);

/* [F,iter] = optimF(p1,p2)   F_methods/optimF.m:1,34-78.  p1,p2 rows x n x B (rows = 2 or 3); F 3x3xB;
 * iter B (may be NULL).  n < 8 -> TVF_ERR_TOO_FEW_POINTS. */
int tvf_optim_f(tvf_handle_t h, const double* p1, const double* p2, int rows, int n, int64_t B, double* F,
                int32_t* iter, int32_t* status);

/* [T,P1,P2,P3] = linearTFT(p1,p2,p3)   TFT_methods/linearTFT.m:1,36-91.
 * p1,p2,p3: rows x n x B with rows = 2, or 3 for homogeneous points (:39-43).
 * T 3x3x3xB; P2,P3 3x4xB (may be NULL); P1 is eye(3,4) (:88) and is left to the caller. */
int tvf_linear_tft(tvf_handle_t h, const double* p1, const double* p2, const double* p3, int rows, int n,
                   int64_t B, double* T, double* P2, double* P3, int32_t* status);

/* F = linearF(p1,p2)   F_methods/linearF.m:1,32-62.  n < 8 -> TVF_ERR_TOO_FEW_POINTS. */
int tvf_linear_f(tvf_handle_t h, const double* p1, const double* p2, int rows, int n, int64_t B, double* F,
                 int32_t* status);

/* ---- the smaller reference functions, batched ------------------------------------------- */

/* [new_points,N_matrix] = Normalize2Ddata(points)   auxiliar_functions/Normalize2Ddata.m:1,33-39.
 * points 2 x n x B -> new_points 2 x n x B, N_matrix 3 x 3 x B (either may be NULL). */
int tvf_normalize2d(tvf_handle_t h, const double* points, int n, int64_t B, double* new_points, double* N_matrix);

/* T_new = transform_TFT(T_old,M1,M2,M3,inverse)   TFT_methods/transform_TFT.m:1,32-49.
 * M1..M3 3x3 shared (mats_batched = 0) or 3x3xB. */
int tvf_transform_tft(tvf_handle_t h, const double* T_old, const double* M1, const double* M2, const double* M3,
                      int mats_batched, int inverse, int64_t B, double* T_new);

/* [R_t_2,R_t_3] = R_t_from_TFT(T,CalM,Corresp)   TFT_methods/R_t_from_TFT.m:1,40-106.
 * votes (10 x B, may be NULL): the cheirality votes of the local recover_R_t (:91-104), layout as in tvf_pose_out. */
int tvf_rt_from_tft(tvf_handle_t h, const double* T, const double* calm, int calm_batched, const double* corresp,
                    int n, int64_t B, double* Rt2, double* Rt3, int32_t* votes, int32_t* status);

/* T = TFT_from_P(P1,P2,P3)   TFT_methods/TFT_from_P.m:1,25-33.  P* 3x4xB. */
int tvf_tft_from_p(tvf_handle_t h, const double* P1, const double* P2, const double* P3, int64_t B, double* T);

/* space_points = triangulation3D(Pcam,image_points)   auxiliar_functions/triangulation3D.m:1,32-64.
 * P: 3 x 4 x M (cams_batched = 0) or 3 x 4 x M x B; image_points (rows*M) x n x B with rows = 2 or 3;
 * X 4 x n x B unit null vectors (sign arbitrary, as in the reference).  M = 2 or 3 (the only cases
 * on the path); other M return TVF_ERR_ARG. */
int tvf_triangulate(tvf_handle_t h, const double* P, int M, int cams_batched, const double* image_points, int rows,
                    int n, int64_t B, double* X);

/* error = ReprError(ProjM,Corresp,Points3D)   auxiliar_functions/ReprError.m:1,39-65.
 * points3d NULL -> triangulate first (:43-44); else pts_rows = 3 or 4 (:45-48). */
int tvf_repr_error(tvf_handle_t h, const double* P, int M, int cams_batched, const double* corresp, int rows, int n,
                   int64_t B, const double* points3d, int pts_rows, double* err);

/* Corresp = project3Dpoints(Points3D,Pcam)   auxiliar_functions/project3Dpoints.m:1,28-35.
 * points3d 3 x n x B; P 3 x 4 x M (or x B); corresp (2M) x n x B.  Used by the real-data pre-filter
 * (experiments_real.m:94-99). */
int tvf_project3d(tvf_handle_t h, const double* points3d, const double* P, int M, int cams_batched, int n, int64_t B,
                  double* corresp);

/* [rot_err,t_err] = AngError(R_t_true,R_t_est)   auxiliar_functions/AngError.m:1,21-28 (degrees).
 * Rt_true 3x4 (true_batched = 0) or 3x4xB. */
int tvf_ang_error(tvf_handle_t h, const double* Rt_true, int true_batched, const double* Rt_est, int64_t B,
                  double* rot_err, double* t_err);

/* ---- bundle adjustment of the three-view poses ------------------------------------------------------------------
 * Minimises  sum over views m = 1..3 and points i of |pi(K_m (R_m X_i + t_m)) - x_{m,i}|^2  (pixels, no data
 * normalisation; = 3n ReprError^2, auxiliar_functions/ReprError.m:65) over R2, t2, R3, t3 and the points, with camera 1
 * fixed at K1[I|0] and the scale gauge |t2| = 1 (11 + 3n unknowns).  A start with |t2| != 1 is first scaled by 1/|t2|
 * (t2, t3 and the points; the reprojection is unchanged).  This is NOT the reference's BundleAdjustment.m, whose source
 * is not available to check: it normalises the image data first (Normalize2Ddata), which may weight the views
 * differently and then has another minimiser (DESIGN.md section 8).
 *
 * Inputs per problem: corresp 6 x n, calm 9 x 3 (calm_batched = 0: shared) or 9 x 3 x B, the start poses Rt2_0, Rt3_0
 * (3 x 4 x B) and optionally reconst0 (3 x n x B, Euclidean); reconst0 = NULL triangulates the start points with
 * triangulation3D({K1[I|0], K2 Rt2_0, K3 Rt3_0}, corresp), as the pose methods compute Reconst.  n < 4 -> TVF_ERR_ARG.
 * Outputs: Rt2, Rt3 (required), reconst (3 x n x B, Euclidean), repr_err = ReprError of the result, iter = number of
 * linearisations, status (each may be NULL).  Outputs must not overlap inputs.
 *
 * Solver: Levenberg-Marquardt, one warp per problem, the points eliminated by the Schur complement (11 x 11 reduced
 * camera system, Cholesky).  Local chart at every iterate: R <- exp([w]x) R for R2 and R3, t2 moved in its tangent
 * plane and renormalised, t3 and the points additively.  Damping H + mu diag(H), mu_0 = 1e-3; an accepted step (gain
 * ratio rho) sets mu *= max(1/3, 1 - (2 rho - 1)^3), nu = 2; a rejected step (cost not lower, or a damped system that
 * is not positive definite) sets mu *= nu, nu *= 2 and re-solves at the same linearisation.  Only steps that lower the
 * cost are accepted, so repr_err never exceeds the start's.  Stops with status 0 when
 *   |g|_inf <= 1e-12 |g_start|_inf (g = J'r over all 11 + 3n unknowns), or
 *   |step|_2 <= 1e-12 sqrt(sum |X_i|^2 + |t3|^2 + 1), or
 *   an accepted step lowered the cost by at most 1e-15 of it;
 * TVF_ST_BA_NOCONV after 100 linearisations or 400 damped solves without that.  A non-finite input, start point or
 * start cost, or |t2| = 0, gives TVF_ST_NONFINITE with the inputs copied through (reconst = the start points) and
 * iter = 0.  Every sum and test depends on the problem alone: a result is bit-identical whatever its batch, chunk
 * (tvf_set_chunk) or shard.  The host form runs in chunks and shards B over a group handle like tvf_pose; the _dev form
 * takes device pointers (corresp 16-byte aligned) and is asynchronous on the handle's stream. */
int tvf_bundle_adjust(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                      const double* Rt2_0, const double* Rt3_0, const double* reconst0, double* Rt2, double* Rt3,
                      double* reconst, double* repr_err, int32_t* iter, int32_t* status);
int tvf_bundle_adjust_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                          const double* Rt2_0, const double* Rt3_0, const double* reconst0, double* Rt2, double* Rt3,
                          double* reconst, double* repr_err, int32_t* iter, int32_t* status);

/* ---- first-order covariance of the bundle adjustment at a state ------------------------------------------------
 * The uncertainty of tvf_bundle_adjust's result: the inverse of the Gauss-Newton matrix H = J'J of the adjustment's
 * model (pixel residuals, camera 1 = K1[I|0], |t2| = 1), taken at the given state without damping.  The state (Rt2, Rt3
 * 3 x 4 x B, reconst 3 x n x B Euclidean, all required) is usually tvf_bundle_adjust's output, but any state is accepted;
 * it is first put into the adjustment's gauge exactly as tvf_bundle_adjust does (t2, t3 and the points scaled by
 * 1/|t2|).  corresp, calm, calm_batched and n as for tvf_bundle_adjust; n < 4 -> TVF_ERR_ARG.
 *
 * Chart: the adjustment's 11 camera unknowns at the state, R2 <- exp([w2]x) R2, t2 moved by a in its tangent plane
 * (basis u1, u2), R3 <- exp([w3]x) R3, t3 <- t3 + dt3, and the points additively.  The camera block of H^-1 is S^-1,
 * S the 11 x 11 reduced camera system (the points eliminated); the chart covariance C = S^-1 is expanded with
 * G = blkdiag(I3, [u1 u2], I3, I3) to
 *   cov_cam (12 x 12 x B, column-major, may be NULL) = G C G' over [w2 (3), dt2 (3, ambient), w3 (3), dt3 (3)]:
 *           rank 11, null direction (0, t2, 0, 0); independent of the tangent basis;
 *   cov_pts (3 x 3 x n x B, may be NULL): the marginal covariance of each point in the gauge-normalised frame,
 *           V_i^-1 + V_i^-1 W_i' S^-1 W_i V_i^-1 (V_i = the point's 3 x 3 block of H, W_i its 11 x 3 camera block);
 *   sigma2  (B, may be NULL): the a-posteriori noise variance sum r^2 / (3n - 11) (6n residuals, 11 + 3n unknowns).
 * Both covariances are for UNIT pixel noise: multiply by sigma^2 (for example sigma2) for another noise level.
 * status (B, may be NULL): TVF_ST_NONFINITE for a non-finite input, residual or |t2| = 0; TVF_ST_COV_SINGULAR when a
 * point block V_i or S is not positive definite, where a Cholesky pivot counts as positive only above 1e-12 times the
 * matrix's own diagonal entry.  Either way every output of that problem is NaN.  Every sum depends on the problem alone:
 * a result is bit-identical whatever its batch, chunk (tvf_set_chunk), group-handle shard or _dev form.  The host form
 * chunks and shards like tvf_bundle_adjust; the _dev form takes device pointers (corresp 16-byte aligned) and is
 * asynchronous on the handle's stream. */
int tvf_ba_covariance(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                      const double* Rt2, const double* Rt3, const double* reconst, double* cov_cam, double* cov_pts,
                      double* sigma2, int32_t* status);
int tvf_ba_covariance_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                          const double* Rt2, const double* Rt3, const double* reconst, double* cov_cam, double* cov_pts,
                          double* sigma2, int32_t* status);

/* ---- robust pose from raw matches: consensus and RANSAC ----------------------------------------------------------
 * Inlier test of one match x = (x1 y1 x2 y2 x3 y3) under the cameras K1[I|0], K2[R2|t2], K3[R3|t3]: triangulate it as
 * tvf_triangulate does (triangulation3D.m), dehomogenise X(1:3)/X(4), re-project as tvf_project3d does and subtract x
 * (experiments_real.m:94-98).  The match is an inlier iff all six residuals are finite and <= threshold in absolute
 * value.  Unlike the reference, a NaN residual makes the match an outlier.
 *
 * tvf_consensus: that test for every match of corresp (6 x n x B) under one pose per problem (Rt2, Rt3 3 x 4 x B);
 * calm 9 x 3 (calm_batched = 0) or 9 x 3 x B.  inliers (n x B, 0 / 1) and n_inliers (B) may be NULL.  threshold (pixels)
 * must be finite and > 0.  Chunks and shards like tvf_pose; returns 0 or an error. */
int tvf_consensus(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                  const double* Rt2, const double* Rt3, double threshold, uint8_t* inliers, int32_t* n_inliers);

#define TVF_ST_RANSAC_FAILED 128 /* tvf_ransac_pose: every hypothesis of the problem was flagged: no pose           */

/* Pose of each problem from raw matches with outliers: RANSAC over minimal linear solves and the consensus above.
 * method 1: hypotheses from LinearTFTPoseEstimation on s = 7 matches; 7: LinearFPoseEstimation on s = 8 (linearF.m:35-37).
 * Per problem b, with key seeds[b]:
 *   1. hypothesis h = 0 .. hypotheses-1 draws s distinct match indices (below) and solves the method on those columns;
 *   2. its score is its consensus count with `threshold`, or -1 when the method flagged it (status != 0);
 *   3. the best hypothesis has the largest score, ties to the smallest h;
 *   4. the refit solves the method on the consensus columns of the best hypothesis (index order) and is scored again.
 * Result rule: if the best score is >= s, the refit's status is 0 and its count is >= the best score, the refit pose
 * is returned, otherwise the best hypothesis's pose.  inliers (n x B, 0 / 1) and n_inliers (B) are always those of the
 * returned pose; sample (s x B) holds the best hypothesis's indices.  If every hypothesis is flagged, status gets
 * TVF_ST_RANSAC_FAILED, Rt2 and Rt3 are NaN, inliers 0 and sample -1; otherwise status is 0.
 * Sampler (reproducible from NumPy integer for integer): mix64 is splitmix64's output function (z += 0x9E3779B97F4A7C15;
 * z = (z ^ z >> 30) * 0xBF58476D1CE4E5B9; z = (z ^ z >> 27) * 0x94D049BB133111EB; z ^ z >> 31); draw j of hypothesis h is
 * r = mix64(seed ^ mix64((h << 8) | j)); uniform(m) = ((r >> 32) * m) >> 32; the indices come from Floyd's algorithm: for
 * j = 0 .. s-1, m = n - s + j + 1, u = uniform(m), take u, or m - 1 if u was already taken; kept in draw order.
 * The key is per problem, so a result does not depend on its batch, chunk, shard or form (bit-identical).
 * Errors: method other than 1 or 7, hypotheses outside 1 .. 2^24, a threshold that is not finite or <= 0, or n < s
 * (method 7: TVF_ERR_TOO_FEW_POINTS) -> TVF_ERR_ARG.  Outputs may be NULL.  The host form chunks and shards like
 * tvf_pose.  The _dev form takes device pointers (corresp 16-byte aligned) and, unlike the other _dev forms,
 * synchronises the handle's stream once per chunk: the refit groups the problems by consensus size, which it reads back. */
int tvf_ransac_pose(tvf_handle_t h, int method, const double* corresp, const double* calm, int calm_batched, int n,
                    int64_t B, int hypotheses, double threshold, const uint64_t* seeds, double* Rt2, double* Rt3,
                    uint8_t* inliers, int32_t* n_inliers, int32_t* sample, int32_t* status);
int tvf_ransac_pose_dev(tvf_handle_t h, int method, const double* corresp, const double* calm, int calm_batched, int n,
                        int64_t B, int hypotheses, double threshold, const uint64_t* seeds, double* Rt2, double* Rt3,
                        uint8_t* inliers, int32_t* n_inliers, int32_t* sample, int32_t* status);

/* ---- inputs of the measured configurations, generated where they are consumed ------------------------
 * Trials [first_trial, first_trial+B) of experiments.m's sweep: trial j uses noise_levels[j mod L] and
 * seed j div L + 1; each is generateSyntheticScene(n+100, noise, seed, ...) followed by the column
 * sub-sampling of experiments.m:94-95 (auxiliar_functions/generateSyntheticScene.m:75-111).  P: the three
 * scaled 3x4 cameras, ROW-major (36 doubles); (hi_x, hi_y): image size in pixels.  RNG = "TVF scene RNG v2"
 * (MT19937 genrand_res53, polar Gaussian with a reproducible logarithm, NumPy's legacy shuffle): bit-identical
 * to the host generator tft_vs_fund_b200/scene.py; n <= 60.  corresp: 6 x n x B. */
int tvf_generate_sweep(tvf_handle_t h, int64_t first_trial, int64_t B, int n, const double* noise_levels, int L,
                       const double* P, double hi_x, double hi_y, double* corresp);
int tvf_generate_sweep_dev(tvf_handle_t h, int64_t first_trial, int64_t B, int n, const double* noise_levels, int L,
                           const double* P, double hi_x, double hi_y, double* d_corresp);

/* The inner loops of experiments.m:74-124 for one method (1 = LinearTFTPoseEstimation, 7 =
 * LinearFPoseEstimation, 8 = OptimFPoseEstimation; numbering of experiments.m:51-59), entirely device-resident: trials [first_trial, first_trial+B) are generated
 * (as tvf_generate_sweep), solved, and their ReprError / AngError (auxiliar_functions/AngError.m, mean of the
 * two views as in :117-120) summed per noise level in a fixed order.  table: L x 5 row-major =
 * [sum repr_err, sum rot_err, sum t_err, trials counted, trials skipped (no pose / non-finite)].
 * calm 9x3; Rt0_2, Rt0_3: ground-truth 3x4 poses (column-major). */
int tvf_sweep_run(tvf_handle_t h, int method, int64_t first_trial, int64_t B, int n, const double* noise_levels, int L,
                  const double* P, double hi_x, double hi_y, const double* calm, const double* Rt0_2, const double* Rt0_3,
                  double* table);

/* The same loop for any of the four experiments of experiments.m:23-47 ('noise', 'focal', 'points', 'angle'): level l of
 * the swept variable has its own noise, point count N, cameras (focal length / collinearity change K, the centres and
 * the ground truth: generateSyntheticScene.m:45-72,113), CalM and ground-truth poses.  Trial j of [first_trial,
 * first_trial + B) is level j mod L with seed j div L + 1, exactly as in tvf_sweep_run.  table: L x 5 as above; a level
 * the reference skips for lack of matches ((m > 6 && N < 8) || N < 7, experiments.m:99-104) gets +inf sums and count 0.
 * P row-major (as tvf_generate_sweep); calm 9x3 and Rt0_* 3x4 column-major. */
typedef struct tvf_sweep_level {
    double noise;
    int32_t n;
    int32_t reserved;
    double P[36];
    double calm[27];
    double Rt0_2[12];
    double Rt0_3[12];
} tvf_sweep_level;
int tvf_sweep_run_levels(tvf_handle_t h, int method, int64_t first_trial, int64_t B, const tvf_sweep_level* levels, int L,
                         double hi_x, double hi_y, double* table);

/* tvf_sweep_run_levels followed, trial by trial, by the library's bundle adjustment (tvf_bundle_adjust, started from the
 * method's R_t_2, R_t_3 and Reconst, the level's CalM shared): the two column groups of experiments.m:127-141.  Arguments,
 * trial mapping, checks and skipped levels as tvf_sweep_run_levels.  table: L x 11 row-major =
 *   0-4   the method, exactly as tvf_sweep_run_levels;
 *   5-7   after adjustment: sum repr_err (the adjusted ReprError over the trial's n points), sum rot_err, sum t_err;
 *   8     trials counted after adjustment;
 *   9     trials skipped after adjustment (the method's pose skipped, or the adjustment TVF_ST_NONFINITE);
 *   10    sum of the adjustment's `iter` over the trials of column 8.
 * Trials ending with TVF_ST_BA_NOCONV are counted.  A level the reference skips gets +inf in 0-2 and 5-7, 0 elsewhere.
 * Each trial's adjustment is bit-identical to tvf_bundle_adjust's on the same start, whatever the chunk or range. */
int tvf_sweep_run_levels_ba(tvf_handle_t h, int method, int64_t first_trial, int64_t B, const tvf_sweep_level* levels,
                            int L, double hi_x, double hi_y, double* table);

/* ---- device-pointer forms (inputs/outputs already in HBM; asynchronous on the handle's stream,
 *      return 0 without synchronising -- read `status` after tvf_synchronize).  `corresp` must be
 *      16-byte aligned (any cudaMalloc'ed buffer, and any problem boundary inside one, is); otherwise
 *      TVF_ERR_ARG ------------------------------------------------------------------------------ */
int tvf_linear_tft_pose_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n,
                            int64_t B, double* Rt2, double* Rt3, double* reconst, double* T, double* repr_err,
                            int32_t* status);
int tvf_linear_f_pose_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n,
                          int64_t B, double* Rt2, double* Rt3, double* reconst, double* T, double* repr_err,
                          double* F21, double* F31, int32_t* status);
int tvf_optim_f_pose_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n,
                         int64_t B, double* Rt2, double* Rt3, double* reconst, double* T, double* repr_err,
                         double* F21, double* F31, int32_t* iter, int32_t* status);

/* ---- measurement support ------------------------------------------------------------------ */
/* number of kernel launches issued through this handle since creation */
int64_t tvf_launch_count(tvf_handle_t h);
/* per-kernel device time: when enabled every kernel launch of the pose entry points is bracketed by
 * CUDA events on its own stream; tvf_profile_read() returns accumulated milliseconds and launch counts
 * per kernel id (arrays of TVF_NUM_KERNELS). */
#define TVF_K_TFT_STAGE1 0
#define TVF_K_TFT_EPIPOLES 1
#define TVF_K_TFT_STAGE2 2
#define TVF_K_F_STAGE1 3
#define TVF_K_F_FINISH 4
#define TVF_K_CANDIDATES 5
#define TVF_K_VOTES 6
#define TVF_K_SCALE 7
#define TVF_K_FINAL 8
#define TVF_K_TFT_FROM_POSE 9
#define TVF_K_TAIL_FUSED 10
#define TVF_K_TFT_MOMENTS_LARGE 11
#define TVF_K_TFT_STAGE1_SOLVE 12
#define TVF_K_OPTIMF_GH 13
#define TVF_NUM_KERNELS 14
int tvf_profile_enable(tvf_handle_t h, int on);
int tvf_profile_reset(tvf_handle_t h);
int tvf_profile_read(tvf_handle_t h, double* total_ms, int64_t* launches);
const char* tvf_kernel_name(int id);
/* measured FP64 FMA throughput of this device (TFLOP/s; a register-resident DFMA loop on all SMs):
 * the denominator of the FP64 roofline fractions bench.py reports */
double tvf_fp64_peak_tflops(tvf_handle_t h);

#ifdef __cplusplus
}
#endif
#endif /* TVF_H_ */
