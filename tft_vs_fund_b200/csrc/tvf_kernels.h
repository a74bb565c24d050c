// tvf_kernels.h -- internal interface between the C-ABI layer (tvf_api.cu) and
// the kernel translation units.  Not installed; the public contract is include/tvf.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace tvf {

// Where a warp/thread finds the correspondences of problem b, point i.
//   packed != 0 : p1 is `Corresp` 6 x n x B (column-major; 48 contiguous bytes per point)
//   packed == 0 : p1,p2,p3 are rows x n x B each (rows = 2, or 3 for homogeneous input)
struct CoreInput {
    const double* p1;
    const double* p2;
    const double* p3;
    int packed;
    int rows;
    int n;
    long long B;
    int normalize;   // 1: *PoseEstimation path (Normalize2Ddata + undo); 0: estimator called directly
};

// per-problem work-space records (doubles) handed between the estimator stages
constexpr int CORE_WS_TFT = 140;   // 96 moments | 9 normalisation stats (+1) | t1 27 (+1) | e21,e31
constexpr int CORE_WS_F = 36;      // raw f (2 x 9) | outer stats 9 | inner stats 9

// returns 1 when only the moments half ran (split stage 1): the caller then launches launch_tft_stage1_solve
int launch_tft_stage1(const CoreInput& in, double* ws, int* status, int sm_count, cudaStream_t stream);
// large-n stage 1: cluster/TMA moments kernel (returns 0 if the shape is unsupported -> use launch_tft_stage1)
// followed by the solve-only half of stage 1
constexpr int LARGE_N_MIN = 1024;
int launch_tft_moments_large(const double* corresp, int n, long long B, int normalize, double* ws, int sm_count,
                             cudaStream_t stream);
void launch_tft_stage1_solve(long long B, double* ws, int* status, int sm_count, cudaStream_t stream);
void launch_tft_epipoles(double* ws, long long B, cudaStream_t stream);
void launch_tft_stage2(const CoreInput& in, const double* ws, double* T, double* P2, double* P3, int* status,
                       int sm_count, cudaStream_t stream);
void launch_f_stage1(const CoreInput& in, double* ws, int* status, int sm_count, cudaStream_t stream);
// normalize != 0: two pairs per problem (F21, F31 -> F[18*b]); else one (F[9*b])
void launch_f_finish(const double* ws, int normalize, long long B, double* F, cudaStream_t stream);

// ---- Gauss-Helmert refinement of F (optimF.m; tvf_gh_kernels.cu).  ws: f_stage1 records of the pose path
// (two pairs per problem); Fio: 18 x B, receives [F21 F31]; iters: 2 x B.  Returns 0 if n is too large.
int optimf_max_n();
int launch_optimf_gh(const double* corresp, int n, long long B, const double* ws, double* Fio, int* iters, int* status,
                     int sm_count, cudaStream_t stream);
void launch_sum_pairs(const int* in2, long long B, int* out, cudaStream_t stream);

// ---- three-view bundle adjustment (tvf_ba_kernels.cu).  Device pointers; X receives the result and holds the current
// iterate, Xc (3 x n x B) is work space; repr_err, iter, status may be null.  Returns 0 if the launch failed.
struct BaArgs {
    const double* corresp;     // 6 x n x B, 16-byte aligned
    const double* calm;        // 9 x 3 (shared) or 9 x 3 x B
    int calm_batched;
    int n;
    long long B;
    const double* Rt2_0;       // 12 x B
    const double* Rt3_0;       // 12 x B
    const double* X0;          // 3 x n x B, or null: triangulated from the start poses
    double* Rt2;               // 12 x B
    double* Rt3;               // 12 x B
    double* X;                 // 3 x n x B
    double* Xc;                // 3 x n x B
    double* repr_err;          // B
    int* iter;                 // B
    int* status;               // B
};
int launch_bundle_adjust(const BaArgs& a, cudaStream_t stream);

// ---- covariance of the bundle adjustment at a state (tvf_ba_cov_kernels.cu).  Device pointers; cov_cam, cov_pts,
// sigma2 and status may be null.  Returns 0 if the launch failed.
struct BaCovArgs {
    const double* corresp;     // 6 x n x B, 16-byte aligned
    const double* calm;        // 9 x 3 (shared) or 9 x 3 x B
    int calm_batched;
    int n;
    long long B;
    const double* Rt2;         // 12 x B
    const double* Rt3;         // 12 x B
    const double* X;           // 3 x n x B
    double* cov_cam;           // 144 x B
    double* cov_pts;           // 9 x n x B
    double* sigma2;            // B
    int* status;               // B
};
int launch_ba_covariance(const BaCovArgs& a, cudaStream_t stream);

// ---- RANSAC pose (tvf_ransac_kernels.cu).  Device pointers.
// Consensus of Q poses: pose q (Rt2, Rt3 12 x Q) belongs to problem q / H of corresp (6 x n x B) and calm; hstatus (Q,
// may be null): a pose with non-zero status scores -1.  count (Q) must be zeroed before; mask (n x Q, may be null)
// receives the inlier flags.
void launch_ransac_consensus(const double* corresp, const double* calm, int calm_batched, int n, long long Q, int H,
                             const double* Rt2, const double* Rt3, const int* hstatus, double th, int* count,
                             unsigned char* mask, int sm_count, cudaStream_t stream);

// the buffers of one chunk of tvf_ransac_pose: B problems, H hypotheses of s points each
struct RansacArgs {
    const double* corresp;     // 6 x n x B, 16-byte aligned
    const double* calm;        // 9 x 3 (shared) or 9 x 3 x B
    int calm_batched;
    int n;
    long long B;
    const uint64_t* seeds;     // B
    // outputs
    double* Rt2;               // 12 x B
    double* Rt3;               // 12 x B
    unsigned char* inliers;    // n x B
    int* n_inliers;            // B
    int* sample;               // s x B
    int* status;               // B
    // hypotheses (B * H)
    double* gin;               // 6 x s x (B H): the minimal problems
    double* gcalm;             // 27 x (B H) when calm_batched
    double* hRt2; double* hRt3; int* hstatus; int* hcount;
    // per problem: the best hypothesis and the refit
    int* best_h; int* cnt_best; unsigned char* mask_best; double* bestRt2; double* bestRt3;
    int* refst; int* cnt_refit; unsigned char* mask_refit; double* refRt2; double* refRt3;
    double* rin; double* rcalm; int* plist;   // the refit's compacted problems (6 x n x B, 27 x B) and problem list (B)
};
// the s-point minimal problem of every hypothesis (gin, gcalm)
void launch_ransac_sample(const RansacArgs& a, int H, int s, cudaStream_t stream);
// per problem the hypothesis of largest hcount (ties: smallest h) -> best_h (-1: all flagged), bestRt2/3 (NaN then)
void launch_ransac_select(const RansacArgs& a, int H, cudaStream_t stream);
// problems plist[0..m) of refit size k: their consensus columns (mask_best, index order) -> rin (6 x k x m), rcalm
void launch_ransac_gather(const RansacArgs& a, const int* plist, int m, int k, cudaStream_t stream);
// refit results of those problems (Rt2, Rt3, status m each) -> refRt2, refRt3, refst
void launch_ransac_scatter(const RansacArgs& a, const int* plist, int m, const double* Rt2, const double* Rt3,
                           const int* st, cudaStream_t stream);
// the result rule (include/tvf.h, tvf_ransac_pose) -> the outputs
void launch_ransac_finish(const RansacArgs& a, int s, cudaStream_t stream);

// ---- pose tail -----------------------------------------------------------------------------
struct PoseTailArgs {
    const double* corresp;     // 6 x n x B
    const double* calm;        // 9 x 3 (shared) or 9 x 3 x B
    int calm_batched;
    int n;
    long long B;
    // workspace (device)
    double* cand;              // CAND_SIZE x B
    int* votes;                // 10 x B : 8 votes, nanmask pair 2, nanmask pair 3
    double* scale;             // 2 x B : num, den
    // outputs (device; any may be null)
    double* Rt2;               // 12 x B
    double* Rt3;               // 12 x B
    double* reconst;           // 3 x n x B
    double* repr_err;          // B
    int* status;               // B (or-ed into)
};

// mode 0: model = T (27 x B, pixel coordinates); mode 1: model = [F21 F31] (18 x B)
void launch_candidates(int mode, const double* model, const PoseTailArgs& a, cudaStream_t stream);
// TAIL_FUSED_MIN_N <= n <= TAIL_FUSED_MAX_N: votes + scale + final in one launch; otherwise the three kernels below
constexpr int TAIL_FUSED_MIN_N = 7;
constexpr int TAIL_FUSED_MAX_N = 256;
void launch_pose_tail_fused(const PoseTailArgs& a, int sm_count, cudaStream_t stream);
void launch_votes(const PoseTailArgs& a, int sm_count, cudaStream_t stream);
void launch_scale(const PoseTailArgs& a, int sm_count, cudaStream_t stream);
void launch_final(const PoseTailArgs& a, int sm_count, cudaStream_t stream);
// LinearFPoseEstimation.m:78  T = TFT_from_P(K1*eye(3,4), K2*R_t_2, K3*R_t_3)
void launch_tft_from_pose(const double* calm, int calm_batched, const double* Rt2, const double* Rt3,
                          long long B, double* T, cudaStream_t stream);

// ---- stand-alone reference functions (batched) ---------------------------------------------
void launch_normalize2d(const double* pts, int n, long long B, double* out, double* Nmat, cudaStream_t s);
void launch_transform_tft(const double* T, const double* M1, const double* M2, const double* M3, int mats_batched,
                          int inverse, long long B, double* Tout, cudaStream_t s);
void launch_tft_from_p(const double* P1, const double* P2, const double* P3, long long B, double* T, cudaStream_t s);
void launch_triangulate(const double* P, int M, int cams_batched, const double* pts, int rows, int n, long long B,
                        double* X, cudaStream_t s);
void launch_repr_error(const double* P, int M, int cams_batched, const double* corresp, int rows, int n, long long B,
                       const double* pts3d, int pts_rows, double* err, cudaStream_t s);
void launch_project3d(const double* pts3d, const double* P, int M, int cams_batched, int n, long long B, double* out,
                      cudaStream_t s);
void launch_ang_error(const double* Rt_true, int true_batched, const double* Rt_est, long long B, double* rot,
                      double* tr, cudaStream_t s);

// ---- per-noise-level evaluation sums (f3): partial is (L*Q) x 5, table L x 5 = [sum repr, sum rot, sum t, count, skipped].
// status2 != null (bundle adjustment's status, with its iter per trial): a trial flagged in either status word is skipped,
// and partial / table get a sixth column, the sum of iter over the counted trials (finish with ncol = 6).
void launch_sweep_eval_accumulate(const double* Rt2, const double* Rt3, const double* repr, const int* status,
                                  long long first_trial, long long B, int L, int Q, const double* d_Rt0, double* d_partial,
                                  cudaStream_t s, const int* status2 = nullptr, const int* iter = nullptr);
void launch_sweep_eval_finish(const double* d_partial, int L, int Q, double* d_table, cudaStream_t s, int ncol = 5);

// ---- synthetic sweep trials generated on the device (f1) -----------------------------------------------
constexpr int SWEEP_MAX_N = 60;      // n + 100 points per scene must fit the per-thread scratch
void launch_sweep_trials(long long first_trial, long long B, int n, const double* d_noise_levels, int L, const double* d_P,
                         double hi_x, double hi_y, double* d_out, cudaStream_t stream);

}  // namespace tvf
