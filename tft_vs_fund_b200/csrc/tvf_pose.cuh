// tvf_pose.cuh -- per-problem and per-point stages of the pose tail
// (R_t_from_TFT.m:40-106, LinearFPoseEstimation.m:59-78, triangulation3D.m,
// ReprError.m), written as host/device functions so the kernels in
// tvf_pose_kernels.cu and the CPU self-check in tests/hostcheck share one source.
#pragma once
#include "tvf_math.cuh"

// second-chance certificate from the 4 x 4 normal equations (dlt4_depth_signs, round 2 first half) between the ray test
// and the accurate route: off -- what the ray test declines it mostly declines too
#ifndef TVF_VOTE_GRAM_SIGNS
#define TVF_VOTE_GRAM_SIGNS 0
#endif

namespace tvf {

// Per-problem candidate record written by the "candidates" stage and read by
// every point thread of the problem.  For view pair p (0: cameras 1-2, 1: 1-3):
//   R[9] Rp[9] t[3]            -- R_t_from_TFT.m:85-88
//   KR[9] KRp[9] Kt[3]         -- K_v*R, K_v*Rp, K_v*t so that the four candidate
//                                 cameras K_v*[R,+-t] need no further products
constexpr int CAND_PAIR = 42;
constexpr int CAND_SIZE = 2 * CAND_PAIR;
constexpr int OFF_R = 0, OFF_RP = 9, OFF_T = 18, OFF_KR = 21, OFF_KRP = 30, OFF_KT = 39;

// status bits (per problem)
constexpr int ST_EIG_NOCONV = 1;     // inverse iteration hit its cap (ill-conditioned system)
constexpr int ST_EPIPOLE_ZERO = 2;   // sign(V(end))==0 at R_t_from_TFT.m:50/55
constexpr int ST_NO_POSE_2 = 4;      // all four cheirality votes negative/NaN: MATLAB leaves R_f undefined
constexpr int ST_NO_POSE_3 = 8;
constexpr int ST_NONFINITE = 16;     // non-finite value in the outputs
constexpr int ST_TOO_FEW_MATCHES = 256;  // a problem of a ragged batch has fewer matches than the method needs

TVF_HD void fill_pair_(const double* E, const double* K, double* c) {
    decompose_essential(E, c + OFF_R, c + OFF_RP, c + OFF_T);
    mat3_mul(K, c + OFF_R, c + OFF_KR);
    mat3_mul(K, c + OFF_RP, c + OFF_KRP);
    mat3_vec(K, c + OFF_T, c + OFF_KT);
}

// R_t_from_TFT.m:44-58 then :84-88 for both pairs.  T is the TFT in pixel
// coordinates; CalM = [K1;K2;K3] 9x3 column-major.  Returns status bits.
TVF_HD int candidates_from_tft(const double* T, const double* CalM, double* cand) {
    double K1[9], K2[9], K3[9];
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            K1[r + 3 * c] = CalM[r + 9 * c]; K2[r + 3 * c] = CalM[3 + r + 9 * c]; K3[r + 3 * c] = CalM[6 + r + 9 * c];
        }
    double Tc[27];
    transform_tft(T, K1, K2, K3, 1, Tc);                       // :44
    double e21[3], e31[3];
    tft_epipoles(Tc, e21, e31);                                 // :47-55
    int st = 0;
    const double s31 = sign_(e31[2]), s21 = sign_(e21[2]);      // *sign(V(end))
    if (s31 == 0.0 || s21 == 0.0) st |= ST_EPIPOLE_ZERO;
#pragma unroll
    for (int i = 0; i < 3; ++i) { e31[i] *= s31; e21[i] *= s21; }
    // E21 = crossM(e21)*[T1*e31 T2*e31 T3*e31]                  :57
    // E31 = -crossM(e31)*[T1.'*e21 T2.'*e21 T3.'*e21]           :58
    double E21[9], E31[9];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        double a[3], b[3];
        mat3_vec(Tc + 9 * i, e31, a);
        cross3(e21, a, E21 + 3 * i);
        mat3_tvec(Tc + 9 * i, e21, b);
        cross3(e31, b, E31 + 3 * i);
        E31[3 * i] = -E31[3 * i]; E31[3 * i + 1] = -E31[3 * i + 1]; E31[3 * i + 2] = -E31[3 * i + 2];
    }
    fill_pair_(E21, K2, cand);
    fill_pair_(E31, K3, cand + CAND_PAIR);
    return st;
}

// LinearFPoseEstimation.m:86-91 for both pairs (E = K_v.'*F*K1).
TVF_HD int candidates_from_f(const double* F21, const double* F31, const double* CalM, double* cand) {
    double K1[9], K2[9], K3[9];
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            K1[r + 3 * c] = CalM[r + 9 * c]; K2[r + 3 * c] = CalM[3 + r + 9 * c]; K3[r + 3 * c] = CalM[6 + r + 9 * c];
        }
    double tmp[9], E[9];
    mat3_mul_tn(K2, F21, tmp); mat3_mul(tmp, K1, E);
    fill_pair_(E, K2, cand);
    mat3_mul_tn(K3, F31, tmp); mat3_mul(tmp, K1, E);
    fill_pair_(E, K3, cand + CAND_PAIR);
    return 0;
}

TVF_HD void load_K1_as_P1(const double* CalM, double* P1) {      // K1*eye(3,4) == [K1 [0;0;0]]
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int r = 0; r < 3; ++r) P1[r + 3 * c] = CalM[r + 9 * c];
    P1[9] = 0.0; P1[10] = 0.0; P1[11] = 0.0;
}

// candidate k (0..3) of a pair -> camera K*[R|t], rotation third row and t_z
// order (R,t),(R,-t),(Rp,-t),(Rp,t): R_t_from_TFT.m:92-97
TVF_HD void candidate_camera(const double* c, int k, double* P, double* r3, double* tz) {
    const double* KR = (k < 2) ? c + OFF_KR : c + OFF_KRP;
    const double* R = (k < 2) ? c + OFF_R : c + OFF_RP;
    const double sg = (k == 0 || k == 3) ? 1.0 : -1.0;
#pragma unroll
    for (int i = 0; i < 9; ++i) P[i] = KR[i];
    P[9] = sg * c[OFF_KT]; P[10] = sg * c[OFF_KT + 1]; P[11] = sg * c[OFF_KT + 2];
    r3[0] = R[2]; r3[1] = R[5]; r3[2] = R[8];
    *tz = sg * c[OFF_T + 2];
}

// Two-view DLT of one point (triangulation3D.m:51-64 with M=2).
TVF_HD void triangulate2(const double* Pa, const double* Pb, double xa, double ya, double xb, double yb, double* X) {
    double a[4][4];
    dlt_rows(Pa, xa, ya, a[0], a[1]);
    dlt_rows(Pb, xb, yb, a[2], a[3]);
    dlt_null<4>(a, X);
}

TVF_HD void triangulate3(const double* Pa, const double* Pb, const double* Pc, const double* p6, double* X) {
    double a[6][4];
    dlt_rows(Pa, p6[0], p6[1], a[0], a[1]);
    dlt_rows(Pb, p6[2], p6[3], a[2], a[3]);
    dlt_rows(Pc, p6[4], p6[5], a[4], a[5]);
    dlt_null<6>(a, X);
}

// One point's contribution to the votes of a pair (R_t_from_TFT.m:98-100).
// Only candidates (R,t) and (Rp,t) are triangulated: negating t negates the fourth column of the
// candidate camera, which negates the fourth component of every quantity of the Householder QR and of
// the inverse iteration *bit for bit* (all operations are sign-symmetric), so the DLT solution of
// (R,-t) is (X,Y,Z,-W) exactly, both depths change sign, and vote(R,-t) = -vote(R,t),
// vote(Rp,-t) = -vote(Rp,t) -- not an approximation, the same numbers the four separate DLTs give.
// v[0] += vote of (R,t), v[1] += vote of (Rp,t); nanmask bit 0/1 set when that sum is NaN.
// Xa/Xb (may be null) receive the homogeneous solutions for (R,t) and (Rp,t).
// m7 (may be null): dlt_row_minors of (ra, rb).  When the solutions themselves are not asked for, the two depth signs
// come from the certified ray/plane test (dlt4_depth_signs_ray, ~45 FP64 operations) and only the DLTs it declines
// (0.1 % of the sweep's, none at n = 10 000) take the accurate route.
// AFF: m7 comes from dlt_row_minors<true> (view-1 camera K1*[I | 0]).
// the accurate route of one candidate: Householder DLT, the two depth signs (or the NaN flag), optionally the solution.
// Inlined: as an out-of-line function it measured slower (profiles/r02_variants.md).
TVF_HD void cheirality_accurate(const double* ra, const double* rb, const double* rc, const double* rd, const double* r3,
                                      double tz, int q, int* v, int* nanmask, double* dst) {
    double a[4][4];
#pragma unroll
    for (int e = 0; e < 4; ++e) { a[0][e] = ra[e]; a[1][e] = rb[e]; a[2][e] = rc[e]; a[3][e] = rd[e]; }
#if TVF_VOTE_GRAM_SIGNS
    if (dst == nullptr) {
        int sx, sz;
        if (dlt4_depth_signs(a, r3, tz, &sx, &sz)) { v[q] += sx + sz; return; }
    }
#endif
    double X[4];
    dlt_null<4>(a, X);
    // X1./X1(4): one reciprocal, same inf/NaN outcomes as the division (x*inf = +-inf, 0*inf = NaN)
    const double iw = (X[3] != 0.0) ? rcp_(X[3]) : 1.0 / X[3];
    const double X0 = X[0] * iw, X1 = X[1] * iw, X2 = X[2] * iw, X3 = X[3] * iw;
    const double z2 = r3[0] * X0 + r3[1] * X1 + r3[2] * X2 + tz * X3;                      // [R t]*X1
    if (X2 != X2 || z2 != z2) {
        *nanmask |= (1 << q);
    } else {
        v[q] += (int)sign_(X2) + (int)sign_(z2);
    }
    if (dst != nullptr) { dst[0] = X[0]; dst[1] = X[1]; dst[2] = X[2]; dst[3] = X[3]; }
}

template <bool AFF = false>
TVF_HD void cheirality_point(const double* ra, const double* rb, const double* m7, const double* c, double x2, double y2,
                             int* v, int* nanmask, double* Xa, double* Xb) {
#pragma unroll 1
    for (int q = 0; q < 2; ++q) {
        double P[12], r3[3], tz;
        candidate_camera(c, q == 0 ? 0 : 3, P, r3, &tz);
        double rc[4], rd[4];
        dlt_rows(P, x2, y2, rc, rd);
        double* dst = (q == 0) ? Xa : Xb;
        if (dst == nullptr) {          // only the two depth signs are needed: certified shortcut, else the accurate route
            int sx, sz;
            if (m7 != nullptr && dlt4_depth_signs_ray<AFF>(m7, rc, rd, r3, tz, &sx, &sz)) { v[q] += sx + sz; continue; }
        }
        cheirality_accurate(ra, rb, rc, rd, r3, tz, q, v, nanmask, dst);
    }
}

// votes of the four candidates in the reference's order (R,t),(R,-t),(Rp,-t),(Rp,t) from the two sums
TVF_HD void expand_votes(const int* v2, int nan2, int* vote4, int* nan4) {
    vote4[0] = v2[0]; vote4[1] = -v2[0]; vote4[2] = -v2[1]; vote4[3] = v2[1];
    *nan4 = ((nan2 & 1) ? 3 : 0) | ((nan2 & 2) ? 12 : 0);
}

// R_t_from_TFT.m:91-104: `>=` with num_points_seen starting at 0, later ties win.
// Returns 0..3 or -1 when nothing is ever assigned (MATLAB: undefined R_f).
TVF_HD int select_candidate(const int* vote, int nanmask) {
    int best = 0, sel = -1;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (!((nanmask >> k) & 1) && vote[k] >= best) { sel = k; best = vote[k]; }
    }
    return sel;
}

// selected pose of a pair: Rt (3x4 column-major, [R t]) and camera K*[R t]
TVF_HD void selected_pose(const double* c, int k, double* Rt, double* P) {
    const double* R = (k < 2) ? c + OFF_R : c + OFF_RP;
    const double* KR = (k < 2) ? c + OFF_KR : c + OFF_KRP;
    const double sg = (k == 0 || k == 3) ? 1.0 : -1.0;
#pragma unroll
    for (int i = 0; i < 9; ++i) { Rt[i] = R[i]; P[i] = KR[i]; }
#pragma unroll
    for (int i = 0; i < 3; ++i) { Rt[9 + i] = sg * c[OFF_T + i]; P[9 + i] = sg * c[OFF_KT + i]; }
}

// One point's contribution to the t3 scale (R_t_from_TFT.m:68-73):
// num += dot(p3 x X3, p3 x u3), den += |p3 x u3|^2, X3 = K3*R3*X, u3 = K3*t3.
TVF_HD void scale_point(const double* P1, const double* P2, const double* KR3, const double* u3,
                        const double* p6, double* num, double* den) {
    double X[4];
    triangulate2(P1, P2, p6[0], p6[1], p6[2], p6[3], X);
    const double iw = 1.0 / X[3];
    const double Xc[3] = {X[0] * iw, X[1] * iw, X[2] * iw};
    double X3[3];
    mat3_vec(KR3, Xc, X3);
    const double p3[3] = {p6[4], p6[5], 1.0};
    double c1[3], c2[3];
    cross3(p3, X3, c1);
    cross3(p3, u3, c2);
    *num = c1[0] * c2[0] + c1[1] * c2[1] + c1[2] * c2[2];
    *den = c2[0] * c2[0] + c2[1] * c2[1] + c2[2] * c2[2];
}

// Final three-view DLT + this point's squared reprojection residual over the
// three views (LinearTFTPoseEstimation.m:59-60, ReprError.m:60-65).
TVF_HD double final_point(const double* P1, const double* P2, const double* P3, const double* p6, double* Xout) {
    double X[4];
    triangulate3(P1, P2, P3, p6, X);
    const double iw = 1.0 / X[3];
    const double Xe[4] = {X[0] * iw, X[1] * iw, X[2] * iw, 1.0};
    Xout[0] = Xe[0]; Xout[1] = Xe[1]; Xout[2] = Xe[2];
    double sq = 0.0;
    const double* Ps[3] = {P1, P2, P3};
#pragma unroll
    for (int v = 0; v < 3; ++v) {
        double x[3];
        cam_apply(Ps[v], Xe, x);
        const double iz = 1.0 / x[2];
        const double dx = x[0] * iz - p6[2 * v], dy = x[1] * iz - p6[2 * v + 1];
        sq += dx * dx + dy * dy;
    }
    return sq;
}

// final_point with the third camera given as K3*R3 (first nine entries of P3) and a separately held translation column
// (the fused tail scales t3 in registers): the same operations on the same values as final_point on [K3*R3 | t3s].
TVF_HD double final_point_kt(const double* P1, const double* P2, const double* P3, const double* t3s, const double* p6,
                             double* Xout) {
    double a[6][4];
    dlt_rows(P1, p6[0], p6[1], a[0], a[1]);
    dlt_rows(P2, p6[2], p6[3], a[2], a[3]);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        a[4][c] = p6[5] * P3[2 + 3 * c] - P3[1 + 3 * c];
        a[5][c] = P3[0 + 3 * c] - p6[4] * P3[2 + 3 * c];
    }
    a[4][3] = p6[5] * t3s[2] - t3s[1];
    a[5][3] = t3s[0] - p6[4] * t3s[2];
    double X[4];
    dlt_null<6>(a, X);
    const double iw = 1.0 / X[3];
    const double Xe[4] = {X[0] * iw, X[1] * iw, X[2] * iw, 1.0};
    Xout[0] = Xe[0]; Xout[1] = Xe[1]; Xout[2] = Xe[2];
    double sq = 0.0;
#pragma unroll
    for (int v = 0; v < 3; ++v) {
        double x[3];
        if (v < 2) {
            cam_apply(v == 0 ? P1 : P2, Xe, x);
        } else {
#pragma unroll
            for (int r = 0; r < 3; ++r) x[r] = P3[r] * Xe[0] + P3[r + 3] * Xe[1] + P3[r + 6] * Xe[2] + t3s[r] * Xe[3];
        }
        const double iz = 1.0 / x[2];
        const double dx = x[0] * iz - p6[2 * v], dy = x[1] * iz - p6[2 * v + 1];
        sq += dx * dx + dy * dy;
    }
    return sq;
}

}  // namespace tvf
