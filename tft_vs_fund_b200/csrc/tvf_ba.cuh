// tvf_ba.cuh -- per-point algebra of the three-view bundle adjustment (tvf_bundle_adjust, tvf_ba_kernels.cu).
// `__host__ __device__` like tvf_math.cuh: the same source is inlined into the kernel and compiled with g++ for the
// CPU tests (tests/test_bundle_adjust_cpu.py).
//
// Objective: sum over views m and points i of |pi(K_m (R_m X_i + t_m)) - x_{m,i}|^2 in pixels, camera 1 = K1[I|0],
// |t2| = 1.  The solver linearises in a LOCAL chart around the current iterate; the 11 camera unknowns are
//     c = [w2 (3), a (2), w3 (3), dt3 (3)]:  R2 <- exp([w2]x) R2,  t2 <- (t2 + a0 u1 + a1 u2) / |.|,
//                                            R3 <- exp([w3]x) R3,  t3 <- t3 + dt3,
// with {t2, u1, u2} = onb3(t2), and each point has its 3 coordinates.  Residuals of one point are ordered
// (view 1 x, y, view 2 x, y, view 3 x, y).
#pragma once
#include "tvf_math.cuh"

namespace tvf {

constexpr int BA_NC = 11;                 // camera unknowns
constexpr int BA_NSUM = 66 + 3 * BA_NC;   // per-point sums: reduced matrix (upper triangle, row-major), reduced right-hand
                                          // side, diag(H_cc), g_c
constexpr int BA_RED_RHS = 66, BA_DIAG = 77, BA_GC = 88;

// Levenberg-Marquardt schedule and stopping rule (documented with tvf_bundle_adjust in include/tvf.h)
constexpr double BA_MU0 = 1e-3;           // initial damping: H + mu diag(H)
constexpr double BA_GTOL = 1e-12;         // stop: |g|_inf <= BA_GTOL |g_start|_inf
constexpr double BA_XTOL = 1e-12;         // stop: |step| <= BA_XTOL sqrt(|X|^2 + |t3|^2 + 1)
constexpr double BA_FTOL = 1e-15;         // stop: accepted step lowers the cost by <= BA_FTOL of it
constexpr int BA_IT_MAX = 100;            // linearisations
constexpr int BA_SOLVE_MAX = 4 * BA_IT_MAX;   // damped solves in all (rejected steps included)
constexpr int ST_BA_NOCONV = 32;          // TVF_ST_BA_NOCONV

struct BaCams {
    double K1[9], K2[9], K3[9];           // column-major
    double R2[9], t2[3], R3[9], t3[3];
    double u1[3], u2[3];                  // tangent basis of the unit sphere at t2
};

// one point's residuals and Jacobian blocks; the rows of view 1 carry no camera unknowns, view 2 only the first five
// (w2, a), view 3 only the last six (w3, dt3)
struct BaPoint {
    double r[6];
    double Jp[6][3];                      // d r / d X
    double J2[2][5];                      // d r(view 2) / d (w2, a)
    double J3[2][6];                      // d r(view 3) / d (w3, dt3)
};

// the point's share of the elimination at damping mu
struct BaElim {
    double L[6];                          // Cholesky factor of H_pp + mu diag(H_pp): l00 l10 l11 l20 l21 l22
    double W[3][12];                      // L^-1 [H_pc | g_p]
    double d[3];                          // diag(H_pp) (undamped)
    double g[3];                          // g_p = Jp' r
};

TVF_HD int ba_tri(int a, int b) { return a * BA_NC - (a * (a - 1)) / 2 + (b - a); }   // a <= b < 11

// CalM 9 x 3 and [R|t] 3 x 4, column-major -> cameras (t2 taken as given; u1, u2 from it)
TVF_HD void ba_load_cams(const double* calm, const double* Rt2, const double* Rt3, BaCams& c) {
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            c.K1[r + 3 * k] = calm[r + 9 * k]; c.K2[r + 3 * k] = calm[3 + r + 9 * k]; c.K3[r + 3 * k] = calm[6 + r + 9 * k];
        }
#pragma unroll
    for (int q = 0; q < 9; ++q) { c.R2[q] = Rt2[q]; c.R3[q] = Rt3[q]; }
#pragma unroll
    for (int q = 0; q < 3; ++q) { c.t2[q] = Rt2[9 + q]; c.t3[q] = Rt3[9 + q]; }
    onb3(c.t2, c.u1, c.u2);
}

// pixel residual of one view at camera coordinates Y, and A = d pixel / d Y (2 x 3)
TVF_HD void ba_view(const double* K, const double* Y, double x, double y, double* r, double (*A)[3]) {
    double h[3];
    mat3_vec(K, Y, h);
    const double iz = 1.0 / h[2];
    const double px = h[0] * iz, py = h[1] * iz;
    r[0] = px - x; r[1] = py - y;
    if (A) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            A[0][k] = (K[3 * k] - px * K[2 + 3 * k]) * iz;
            A[1][k] = (K[1 + 3 * k] - py * K[2 + 3 * k]) * iz;
        }
    }
}

// sum of the six squared residuals of one point
TVF_HD double ba_point_cost(const BaCams& c, const double* X, const double* x6) {
    double Y[3], v[3], r[2], s = 0.0;
    ba_view(c.K1, X, x6[0], x6[1], r, nullptr);
    s += r[0] * r[0] + r[1] * r[1];
    mat3_vec(c.R2, X, v);
    Y[0] = v[0] + c.t2[0]; Y[1] = v[1] + c.t2[1]; Y[2] = v[2] + c.t2[2];
    ba_view(c.K2, Y, x6[2], x6[3], r, nullptr);
    s += r[0] * r[0] + r[1] * r[1];
    mat3_vec(c.R3, X, v);
    Y[0] = v[0] + c.t3[0]; Y[1] = v[1] + c.t3[1]; Y[2] = v[2] + c.t3[2];
    ba_view(c.K3, Y, x6[4], x6[5], r, nullptr);
    s += r[0] * r[0] + r[1] * r[1];
    return s;
}

// residuals and Jacobian blocks of one point.  d(exp([w]x) R X)/dw at w = 0 is -[R X]x, so the row of a rotation
// block is (R X) x A(row); d t2 / d a = [u1 u2].
TVF_HD void ba_point_jac(const BaCams& c, const double* X, const double* x6, BaPoint& p) {
    double A[2][3], Y[3], v[3];
    ba_view(c.K1, X, x6[0], x6[1], p.r, A);
#pragma unroll
    for (int k = 0; k < 2; ++k)
#pragma unroll
        for (int j = 0; j < 3; ++j) p.Jp[k][j] = A[k][j];
    // view 2
    mat3_vec(c.R2, X, v);
    Y[0] = v[0] + c.t2[0]; Y[1] = v[1] + c.t2[1]; Y[2] = v[2] + c.t2[2];
    ba_view(c.K2, Y, x6[2], x6[3], p.r + 2, A);
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const double* a = A[k];
#pragma unroll
        for (int j = 0; j < 3; ++j) p.Jp[2 + k][j] = a[0] * c.R2[3 * j] + a[1] * c.R2[1 + 3 * j] + a[2] * c.R2[2 + 3 * j];
        p.J2[k][0] = v[1] * a[2] - v[2] * a[1];
        p.J2[k][1] = v[2] * a[0] - v[0] * a[2];
        p.J2[k][2] = v[0] * a[1] - v[1] * a[0];
        p.J2[k][3] = a[0] * c.u1[0] + a[1] * c.u1[1] + a[2] * c.u1[2];
        p.J2[k][4] = a[0] * c.u2[0] + a[1] * c.u2[1] + a[2] * c.u2[2];
    }
    // view 3
    mat3_vec(c.R3, X, v);
    Y[0] = v[0] + c.t3[0]; Y[1] = v[1] + c.t3[1]; Y[2] = v[2] + c.t3[2];
    ba_view(c.K3, Y, x6[4], x6[5], p.r + 4, A);
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const double* a = A[k];
#pragma unroll
        for (int j = 0; j < 3; ++j) p.Jp[4 + k][j] = a[0] * c.R3[3 * j] + a[1] * c.R3[1 + 3 * j] + a[2] * c.R3[2 + 3 * j];
        p.J3[k][0] = v[1] * a[2] - v[2] * a[1];
        p.J3[k][1] = v[2] * a[0] - v[0] * a[2];
        p.J3[k][2] = v[0] * a[1] - v[1] * a[0];
        p.J3[k][3] = a[0]; p.J3[k][4] = a[1]; p.J3[k][5] = a[2];
    }
}

// camera Jacobian entry (row k of the 6 residuals, column j of the 11 unknowns)
TVF_HD double ba_jc(const BaPoint& p, int k, int j) {
    if (k >= 2 && k < 4 && j < 5) return p.J2[k - 2][j];
    if (k >= 4 && j >= 5) return p.J3[k - 4][j - 5];
    return 0.0;
}

// H_pp = Jp'Jp, H_pc = Jp'Jc, g_p = Jp'r; the damped point block H_pp + mu diag(H_pp) = L L' is eliminated:
// W = L^-1 [H_pc | g_p].  False if the damped block is not (numerically) positive definite.
TVF_HD bool ba_point_eliminate(const BaPoint& p, double mu, BaElim& e) {
    double H[3][3], B[3][12];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < 6; ++k) s += p.Jp[k][i] * p.Jp[k][j];
            H[i][j] = s;
        }
        double g = 0.0;
#pragma unroll
        for (int k = 0; k < 6; ++k) g += p.Jp[k][i] * p.r[k];
        B[i][11] = g; e.g[i] = g; e.d[i] = H[i][i];
#pragma unroll
        for (int j = 0; j < 5; ++j) B[i][j] = p.Jp[2][i] * p.J2[0][j] + p.Jp[3][i] * p.J2[1][j];
#pragma unroll
        for (int j = 0; j < 6; ++j) B[i][5 + j] = p.Jp[4][i] * p.J3[0][j] + p.Jp[5][i] * p.J3[1][j];
    }
    const double h00 = H[0][0] * (1.0 + mu), h11 = H[1][1] * (1.0 + mu), h22 = H[2][2] * (1.0 + mu);
    const double l00 = sqrt(h00);
    const double l10 = H[1][0] / l00, l20 = H[2][0] / l00;
    const double q11 = h11 - l10 * l10;
    const double l11 = sqrt(q11);
    const double l21 = (H[2][1] - l20 * l10) / l11;
    const double q22 = h22 - l20 * l20 - l21 * l21;
    const double l22 = sqrt(q22);
    e.L[0] = l00; e.L[1] = l10; e.L[2] = l11; e.L[3] = l20; e.L[4] = l21; e.L[5] = l22;
#pragma unroll
    for (int j = 0; j < 12; ++j) {
        const double w0 = B[0][j] / l00;
        const double w1 = (B[1][j] - l10 * w0) / l11;
        const double w2 = (B[2][j] - l20 * w0 - l21 * w1) / l22;
        e.W[0][j] = w0; e.W[1][j] = w1; e.W[2][j] = w2;
    }
    // !(x > 0) is also true for NaN
    return (h00 > 0.0) && (q11 > 0.0) && (q22 > 0.0) && fabs(l22) <= 1.79769313486231570e308;
}

// adds the point's BA_NSUM sums to acc: (H_cc - W'W) upper triangle | g_c - W' W(:,11) | diag(H_cc) | g_c,
// where H_cc and g_c are this point's camera-block normal equations (block diagonal in the two cameras)
TVF_HD void ba_point_accumulate(const BaPoint& p, const BaElim& e, double* acc) {
    double gc[BA_NC];
#pragma unroll
    for (int j = 0; j < 5; ++j) gc[j] = p.J2[0][j] * p.r[2] + p.J2[1][j] * p.r[3];
#pragma unroll
    for (int j = 0; j < 6; ++j) gc[5 + j] = p.J3[0][j] * p.r[4] + p.J3[1][j] * p.r[5];
#pragma unroll
    for (int a = 0; a < BA_NC; ++a) {
#pragma unroll
        for (int b = a; b < BA_NC; ++b) {
            double hcc = 0.0;
            if (b < 5) hcc = p.J2[0][a] * p.J2[0][b] + p.J2[1][a] * p.J2[1][b];
            else if (a >= 5) hcc = p.J3[0][a - 5] * p.J3[0][b - 5] + p.J3[1][a - 5] * p.J3[1][b - 5];
            const double ww = e.W[0][a] * e.W[0][b] + e.W[1][a] * e.W[1][b] + e.W[2][a] * e.W[2][b];
            acc[ba_tri(a, b)] += hcc - ww;
            if (a == b) acc[BA_DIAG + a] += hcc;
        }
        const double wg = e.W[0][a] * e.W[0][11] + e.W[1][a] * e.W[1][11] + e.W[2][a] * e.W[2][11];
        acc[BA_RED_RHS + a] += gc[a] - wg;
        acc[BA_GC + a] += gc[a];
    }
}

// back-substitution of one point: dX = -(H_pp + mu diag(H_pp))^-1 (g_p + H_pc dc) = -L^-T (W(:,11) + W(:,0:11) dc)
TVF_HD void ba_point_step(const BaElim& e, const double* dc, double* dX) {
    double y[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        double s = e.W[k][11];
#pragma unroll
        for (int j = 0; j < BA_NC; ++j) s += e.W[k][j] * dc[j];
        y[k] = s;
    }
    const double z2 = y[2] / e.L[5];
    const double z1 = (y[1] - e.L[4] * z2) / e.L[2];
    const double z0 = (y[0] - e.L[1] * z1 - e.L[3] * z2) / e.L[0];
    dX[0] = -z0; dX[1] = -z1; dX[2] = -z2;
}

// R <- exp([w]x) R by Rodrigues' formula, exp([w]x) = I + s [w]x + q [w]x^2 with s = sin(th)/th and
// q = (1 - cos th)/th^2 = 2 sin^2(th/2)/th^2 (series below 1e-4 rad: no cancellation at any angle)
TVF_HD void ba_rotate(const double* w, double* R) {
    const double th2 = w[0] * w[0] + w[1] * w[1] + w[2] * w[2];
    double s, q;
    if (th2 < 1e-8) {
        s = 1.0 - th2 / 6.0 + th2 * th2 / 120.0;
        q = 0.5 - th2 / 24.0 + th2 * th2 / 720.0;
    } else {
        const double th = sqrt(th2);
        const double sh = sin(0.5 * th);
        s = sin(th) / th;
        q = 2.0 * sh * sh / th2;
    }
    const double W[9] = {0.0, w[2], -w[1], -w[2], 0.0, w[0], w[1], -w[0], 0.0};    // [w]x, column-major
    double W2[9], E[9], Rn[9];
    mat3_mul(W, W, W2);
#pragma unroll
    for (int k = 0; k < 9; ++k) E[k] = s * W[k] + q * W2[k];
    E[0] += 1.0; E[4] += 1.0; E[8] += 1.0;
    mat3_mul(E, R, Rn);
#pragma unroll
    for (int k = 0; k < 9; ++k) R[k] = Rn[k];
}

// the camera update of one step dc (11 unknowns, ordered as in the header comment); u1, u2 follow the new t2
TVF_HD void ba_update_cams(const double* dc, BaCams& c) {
    ba_rotate(dc, c.R2);
    double t[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) t[k] = c.t2[k] + dc[3] * c.u1[k] + dc[4] * c.u2[k];
    const double inv = 1.0 / sqrt(t[0] * t[0] + t[1] * t[1] + t[2] * t[2]);
#pragma unroll
    for (int k = 0; k < 3; ++k) c.t2[k] = t[k] * inv;
    onb3(c.t2, c.u1, c.u2);
    ba_rotate(dc + 5, c.R3);
#pragma unroll
    for (int k = 0; k < 3; ++k) c.t3[k] += dc[8 + k];
}

// Cholesky solve of the damped reduced camera system (the sums of ba_point_accumulate over all points, plus
// mu * diag(H_cc) on the diagonal): dc = -(S + mu D)^-1 rhs.  Factors in place: entries [0, 77) of `red` are destroyed,
// diag(H_cc) and g_c are kept.  False if not positive definite or the step is not finite.
TVF_HD bool ba_solve_reduced(double* red, double mu, double* dc) {
#pragma unroll 1
    for (int i = 0; i < BA_NC; ++i) {                          // red(j, i), j <= i, becomes U(j, i) of S + mu D = U'U
#pragma unroll 1
        for (int j = 0; j <= i; ++j) {
            double s = red[ba_tri(j, i)] + ((i == j) ? mu * red[BA_DIAG + i] : 0.0);
            for (int k = 0; k < j; ++k) s -= red[ba_tri(k, i)] * red[ba_tri(k, j)];
            if (i == j) {
                if (!(s > 0.0)) return false;
                red[ba_tri(i, i)] = sqrt(s);
            } else {
                red[ba_tri(j, i)] = s / red[ba_tri(j, j)];
            }
        }
    }
    double* y = red + BA_RED_RHS;
#pragma unroll 1
    for (int i = 0; i < BA_NC; ++i) {                          // U' y = -rhs
        double s = -y[i];
        for (int k = 0; k < i; ++k) s -= red[ba_tri(k, i)] * y[k];
        y[i] = s / red[ba_tri(i, i)];
    }
    bool finite = true;
#pragma unroll 1
    for (int i = BA_NC - 1; i >= 0; --i) {                     // U dc = y
        double s = y[i];
        for (int k = i + 1; k < BA_NC; ++k) s -= red[ba_tri(i, k)] * dc[k];
        dc[i] = s / red[ba_tri(i, i)];
        finite = finite && fabs(dc[i]) <= 1.79769313486231570e308;
    }
    return finite;
}

// ---- first-order covariance at a state (tvf_ba_covariance, tvf_ba_cov_kernels.cu) -------------------------------
// H = J'J at mu = 0.  The camera block of H^-1 is S^-1 (S = the reduced matrix of ba_point_accumulate); point i's block
// is V_i^-1 + V_i^-1 H_pc,i S^-1 H_cp,i V_i^-1 = L^-T (I + W S^-1 W') L^-1 with V_i = L L' and W = L^-1 H_pc,i.
// A pivot of a Cholesky factorisation (of a V_i or of S) counts as positive only if it exceeds BA_COV_PIVOT times the
// matrix's own diagonal entry: below that, 1/pivot carries fewer than ~4 correct digits and the covariance is undefined.
constexpr double BA_COV_PIVOT = 1e-12;
constexpr int ST_COV_SINGULAR = 64;       // TVF_ST_COV_SINGULAR

// the point block V = H_pp of ba_point_eliminate(p, 0, e) passes the relative pivot floor (e.L[0]^2 = e.d[0])
TVF_HD bool ba_cov_point_ok(const BaElim& e) {
    return (e.L[0] > 0.0) && (e.L[2] * e.L[2] > BA_COV_PIVOT * e.d[1]) && (e.L[5] * e.L[5] > BA_COV_PIVOT * e.d[2]);
}

// Cholesky S = U'U in place on the 66 upper-triangle entries of the reduced matrix; false if a pivot is not above
// BA_COV_PIVOT times S's diagonal entry (or is NaN)
TVF_HD bool ba_cov_factor(double* U) {
#pragma unroll 1
    for (int i = 0; i < BA_NC; ++i) {
#pragma unroll 1
        for (int j = 0; j <= i; ++j) {
            double s = U[ba_tri(j, i)];
            for (int k = 0; k < j; ++k) s -= U[ba_tri(k, i)] * U[ba_tri(k, j)];
            if (i == j) {
                if (!(s > 0.0 && s > BA_COV_PIVOT * U[ba_tri(i, i)])) return false;
                U[ba_tri(i, i)] = sqrt(s);
            } else {
                U[ba_tri(j, i)] = s / U[ba_tri(j, j)];
            }
        }
    }
    return true;
}

// column j of S^-1 from the factor of ba_cov_factor: U'y = e_j, U x = y
TVF_HD void ba_cov_column(const double* U, int j, double* x) {
    double y[BA_NC];
#pragma unroll 1
    for (int i = 0; i < BA_NC; ++i) {
        double s = (i == j) ? 1.0 : 0.0;
        for (int k = 0; k < i; ++k) s -= U[ba_tri(k, i)] * y[k];
        y[i] = s / U[ba_tri(i, i)];
    }
#pragma unroll 1
    for (int i = BA_NC - 1; i >= 0; --i) {
        double s = y[i];
        for (int k = i + 1; k < BA_NC; ++k) s -= U[ba_tri(i, k)] * x[k];
        x[i] = s / U[ba_tri(i, i)];
    }
}

// entry (i, j) of G C G', G = blkdiag(I3, [u1 u2], I3, I3) (12 x 11): the chart covariance C (11 x 11, column-major)
// in the basis-free coordinates [w2, dt2 (ambient), w3, dt3].  Callers form i <= j and mirror, so the result is
// symmetric bit for bit.
TVF_HD double ba_cov_expand(const double* C, const double* u1, const double* u2, int i, int j) {
    double gi[2], gj[2];
    int ci = i < 3 ? i : (i < 6 ? 3 : i - 1), cj = j < 3 ? j : (j < 6 ? 3 : j - 1);   // first chart column of the row
    const int ni = (i >= 3 && i < 6) ? 2 : 1, nj = (j >= 3 && j < 6) ? 2 : 1;
    gi[0] = ni == 2 ? u1[i - 3] : 1.0; gi[1] = ni == 2 ? u2[i - 3] : 0.0;
    gj[0] = nj == 2 ? u1[j - 3] : 1.0; gj[1] = nj == 2 ? u2[j - 3] : 0.0;
    double s = 0.0;
    for (int a = 0; a < ni; ++a)
        for (int b = 0; b < nj; ++b) s += gi[a] * C[(ci + a) + BA_NC * (cj + b)] * gj[b];
    return s;
}

// point i's 3 x 3 marginal covariance (column-major, symmetric bit for bit) from its elimination at mu = 0 and the
// camera covariance C = S^-1 (11 x 11, column-major): L^-T (I + W C W') L^-1
TVF_HD void ba_cov_point(const BaElim& e, const double* C, double* cov) {
    double T[3][BA_NC], M[3][3], Li[3][3];
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll 1
        for (int b = 0; b < BA_NC; ++b) {
            double s = 0.0;
            for (int a = 0; a < BA_NC; ++a) s += e.W[k][a] * C[a + BA_NC * b];
            T[k][b] = s;
        }
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int l = k; l < 3; ++l) {
            double s = (k == l) ? 1.0 : 0.0;
#pragma unroll 1
            for (int b = 0; b < BA_NC; ++b) s += T[k][b] * e.W[l][b];
            M[k][l] = s; M[l][k] = s;
        }
    const double l00 = e.L[0], l10 = e.L[1], l11 = e.L[2], l20 = e.L[3], l21 = e.L[4], l22 = e.L[5];
    Li[0][0] = 1.0 / l00; Li[1][1] = 1.0 / l11; Li[2][2] = 1.0 / l22;
    Li[1][0] = -l10 * Li[0][0] * Li[1][1];
    Li[2][1] = -l21 * Li[1][1] * Li[2][2];
    Li[2][0] = -(l20 * Li[0][0] + l21 * Li[1][0]) * Li[2][2];
    Li[0][1] = 0.0; Li[0][2] = 0.0; Li[1][2] = 0.0;
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = a; b < 3; ++b) {
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < 3; ++k)
#pragma unroll
                for (int l = 0; l < 3; ++l) s += Li[k][a] * M[k][l] * Li[l][b];
            cov[a + 3 * b] = s; cov[b + 3 * a] = s;
        }
}

}  // namespace tvf
