// tvf_math.cuh -- thread-level FP64 building blocks of the linear three-view
// pose path.  Everything here is `__host__ __device__` so the *same source* is
// (a) inlined into the sm_100a kernels and (b) compiled with g++ into a
// test-only library (tests/hostcheck) and checked against the oracle on CPU.
//
// Conventions: MATLAB column-major everywhere.  A 3x3 matrix is double[9] with
// M(r,c) = M[r + 3*c]; a 3x4 camera is double[12] with P(r,c) = P[r + 3*c];
// a trifocal tensor is double[27] with T(j,k,i) = T[j + 3*k + 9*i]
// (TFT_methods/linearTFT.m:67).
#pragma once
#include <math.h>

#if defined(__CUDACC__)
#define TVF_HD __host__ __device__ __forceinline__
#else
#define TVF_HD inline
#endif

namespace tvf {

// 1/sqrt(x) for normal positive x.  Device: MUFU.RSQ64H seed (~20 bits) + two Newton steps (full double precision,
// not correctly rounded, no special-case path: 8 instructions instead of the ~16 of CUDA's rsqrt()).  x = 0 gives
// NaN (CUDA: +inf); every caller multiplies the result into a vector that is then 0*inf = NaN as well, or guards x > 0.
TVF_HD double rsqrt_(double x) {
#if defined(__CUDA_ARCH__)
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double h = 0.5 * x;
    double e = fma(-h * y, y, 0.5);
    y = fma(y, e, y);
    e = fma(-h * y, y, 0.5);
    return fma(y, e, y);
#else
    return 1.0 / sqrt(x);
#endif
}

// 1/x and sqrt(x) for normal positive/any-sign finite x.  Device: MUFU seed + Newton steps (full double
// precision, not correctly rounded, no slow path) -- ~7 instructions instead of ~20 for the IEEE forms.
// Host (test build): the exact operations.  Used where a last-ulp difference is immaterial (QR, Jacobi
// rotations, normalisations); inv3/transform keep IEEE division.
TVF_HD double rcp_(double x) {
#if defined(__CUDA_ARCH__)
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    e = fma(-x, r, 1.0);
    return fma(r, e, r);
#else
    return 1.0 / x;
#endif
}

TVF_HD double sqrt_(double x) {        // x >= 0; sqrt(0) = 0
#if defined(__CUDA_ARCH__)
    const double r = rsqrt_(x);
    return (x > 0.0) ? x * r : 0.0;
#else
    return sqrt(x);
#endif
}

TVF_HD double sign_(double x) {  // MATLAB sign(): sign(0)=0, sign(NaN)=NaN
    return (x > 0.0) ? 1.0 : ((x < 0.0) ? -1.0 : x);
}

// ------------------------------------------------------------------ 3x3 basics
TVF_HD void mat3_mul(const double* A, const double* B, double* C) {  // C = A*B
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int r = 0; r < 3; ++r)
            C[r + 3 * c] = A[r] * B[3 * c] + A[r + 3] * B[1 + 3 * c] + A[r + 6] * B[2 + 3 * c];
}

TVF_HD void mat3_mul_tn(const double* A, const double* B, double* C) {  // C = A.'*B
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int r = 0; r < 3; ++r)
            C[r + 3 * c] = A[3 * r] * B[3 * c] + A[3 * r + 1] * B[1 + 3 * c] + A[3 * r + 2] * B[2 + 3 * c];
}

TVF_HD void mat3_mul_nt(const double* A, const double* B, double* C) {  // C = A*B.'
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int r = 0; r < 3; ++r)
            C[r + 3 * c] = A[r] * B[c] + A[r + 3] * B[c + 3] + A[r + 6] * B[c + 6];
}

TVF_HD void mat3_vec(const double* A, const double* x, double* y) {  // y = A*x
#pragma unroll
    for (int r = 0; r < 3; ++r) y[r] = A[r] * x[0] + A[r + 3] * x[1] + A[r + 6] * x[2];
}

TVF_HD void mat3_tvec(const double* A, const double* x, double* y) {  // y = A.'*x
#pragma unroll
    for (int r = 0; r < 3; ++r) y[r] = A[3 * r] * x[0] + A[3 * r + 1] * x[1] + A[3 * r + 2] * x[2];
}

TVF_HD double det3(const double* M) {
    return M[0] * (M[4] * M[8] - M[7] * M[5]) - M[3] * (M[1] * M[8] - M[7] * M[2]) +
           M[6] * (M[1] * M[5] - M[4] * M[2]);
}

TVF_HD void inv3(const double* M, double* Mi) {  // inv(M) by adjugate (transform_TFT.m:37,43)
    const double c00 = M[4] * M[8] - M[7] * M[5];
    const double c01 = M[7] * M[2] - M[1] * M[8];
    const double c02 = M[1] * M[5] - M[4] * M[2];
    const double d = M[0] * c00 + M[3] * c01 + M[6] * c02;
    const double id = 1.0 / d;
    Mi[0] = c00 * id; Mi[1] = c01 * id; Mi[2] = c02 * id;
    Mi[3] = (M[6] * M[5] - M[3] * M[8]) * id;
    Mi[4] = (M[0] * M[8] - M[6] * M[2]) * id;
    Mi[5] = (M[3] * M[2] - M[0] * M[5]) * id;
    Mi[6] = (M[3] * M[7] - M[6] * M[4]) * id;
    Mi[7] = (M[6] * M[1] - M[0] * M[7]) * id;
    Mi[8] = (M[0] * M[4] - M[3] * M[1]) * id;
}

TVF_HD void cross3(const double* a, const double* b, double* c) {
    c[0] = a[1] * b[2] - a[2] * b[1];
    c[1] = a[2] * b[0] - a[0] * b[2];
    c[2] = a[0] * b[1] - a[1] * b[0];
}

// ------------------------------------------------- one-sided Jacobi SVD, 3 cols
// Hestenes rotations on the columns of A (3x3, column-major, overwritten by A*V)
// accumulating V.  On return the columns are sorted by descending norm s[0..2];
// V(:,2) is MATLAB's V(:,end).  Replaces svd() at linearTFT.m:71-79,
// R_t_from_TFT.m:47-55,85 and linearF.m:61.
TVF_HD void jacobi_rot_(double* ap, double* aq, double* vp, double* vq, bool& rotated) {
    const double alpha = ap[0] * ap[0] + ap[1] * ap[1] + ap[2] * ap[2];
    const double beta = aq[0] * aq[0] + aq[1] * aq[1] + aq[2] * aq[2];
    const double gamma = ap[0] * aq[0] + ap[1] * aq[1] + ap[2] * aq[2];
    // converged pair: |gamma| <= 1e-15*sqrt(alpha*beta) (~4.5 eps: below that a rotation only moves rounding noise)
    if (!(gamma * gamma > 1.0e-30 * (alpha * beta)) || fabs(gamma) < 1e-300) return;
    rotated = true;
    const double zeta = (beta - alpha) * rcp_(2.0 * gamma);
    const double t = copysign(1.0, zeta) * rcp_(fabs(zeta) + sqrt_(1.0 + zeta * zeta));
    const double c = rsqrt_(1.0 + t * t);
    const double s = c * t;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const double x = ap[i], y = aq[i];
        ap[i] = c * x - s * y; aq[i] = s * x + c * y;
        const double u = vp[i], w = vq[i];
        vp[i] = c * u - s * w; vq[i] = s * u + c * w;
    }
}

TVF_HD void swap_cols_(double* a, double* b, double* va, double* vb, double& sa, double& sb) {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        double t = a[i]; a[i] = b[i]; b[i] = t;
        t = va[i]; va[i] = vb[i]; vb[i] = t;
    }
    double t = sa; sa = sb; sb = t;
}

TVF_HD void jacobi_svd3(double* A, double* V, double* s, int* sweeps = nullptr) {
#pragma unroll
    for (int i = 0; i < 9; ++i) V[i] = (i % 4 == 0) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 30; ++sweep) {
        bool rotated = false;
        jacobi_rot_(A + 0, A + 3, V + 0, V + 3, rotated);
        jacobi_rot_(A + 0, A + 6, V + 0, V + 6, rotated);
        jacobi_rot_(A + 3, A + 6, V + 3, V + 6, rotated);
        if (sweeps) *sweeps = sweep + 1;
        if (!rotated) break;
    }
    s[0] = sqrt_(A[0] * A[0] + A[1] * A[1] + A[2] * A[2]);
    s[1] = sqrt_(A[3] * A[3] + A[4] * A[4] + A[5] * A[5]);
    s[2] = sqrt_(A[6] * A[6] + A[7] * A[7] + A[8] * A[8]);
    if (s[0] < s[1]) swap_cols_(A + 0, A + 3, V + 0, V + 3, s[0], s[1]);
    if (s[1] < s[2]) swap_cols_(A + 3, A + 6, V + 3, V + 6, s[1], s[2]);
    if (s[0] < s[1]) swap_cols_(A + 0, A + 3, V + 0, V + 3, s[0], s[1]);
}

// V(:,end) of svd(M) for a 3x3 M (column-major; `transpose`: of M.'), by Householder QR + inverse iteration with R -- the
// route of dlt_null: the conditioning is that of the SVD, and one null vector costs ~240 FP64 operations instead of the
// ~650 of a converged one-sided Jacobi SVD.  The iteration converges at the rate (s3/s2)^2: <= 3e-3 for the slices of a
// linear TFT estimate at 3 px noise, 0 for a valid (calibrated, constrained) tensor -- two to five steps.  Returns false
// when it has not converged in NULL3_MAX_IT steps (two nearly equal smallest singular values); the caller then takes
// the Jacobi route, which does not care.
constexpr int NULL3_MAX_IT = 12;
TVF_HD bool null3_qr(const double* M, bool transpose, double* v) {
    double a[3][3];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) a[r][c] = transpose ? M[c + 3 * r] : M[r + 3 * c];
    double rr[3][3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        if (k == 2) { rr[2][2] = -a[2][2]; break; }       // 1 x 1 reflection: alpha = -x1 exactly
        double sig = 0.0;
#pragma unroll
        for (int i = k; i < 3; ++i) sig += a[i][k] * a[i][k];
        const double nrm = sqrt_(sig);
        const double x1 = a[k][k];
        const double alpha = -copysign(nrm, x1);
        const double den = sig - alpha * x1;               // = v'v / 2 >= 0
        const double f = (den > 0.0) ? rcp_(den) : 0.0;
        const double vk = x1 - alpha;
#pragma unroll
        for (int c = k + 1; c < 3; ++c) {
            double sdot = vk * a[k][c];
#pragma unroll
            for (int i = k + 1; i < 3; ++i) sdot += a[i][k] * a[i][c];
            sdot *= f;
            a[k][c] -= sdot * vk;
#pragma unroll
            for (int i = k + 1; i < 3; ++i) a[i][c] -= sdot * a[i][k];
        }
        rr[k][k] = alpha;
#pragma unroll
        for (int c = k + 1; c < 3; ++c) rr[k][c] = a[k][c];
    }
    const double rmax = fmax(fabs(rr[0][0]), fmax(fabs(rr[1][1]), fabs(rr[2][2])));
    if (!(rmax > 0.0) || !(rmax < 1.0e300)) return false;            // zero matrix, NaN, Inf: the Jacobi route decides
    const double tiny = 1e-300 + 1e-18 * rmax;
    double d[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double p = (fabs(rr[k][k]) < tiny) ? copysign(tiny, rr[k][k]) : rr[k][k];
        d[k] = rcp_(p);
    }
    double x2 = d[2];
    double x1 = -(rr[1][2] * x2) * d[1];
    double x0 = -(rr[0][1] * x1 + rr[0][2] * x2) * d[0];
    double inv = rsqrt_(x0 * x0 + x1 * x1 + x2 * x2);
    x0 *= inv; x1 *= inv; x2 *= inv;
    double dprev = 0.0;
    bool ok = false;
    for (int it = 0; it < NULL3_MAX_IT; ++it) {
        const double y0 = x0 * d[0];
        const double y1 = (x1 - rr[0][1] * y0) * d[1];
        const double y2 = (x2 - rr[0][2] * y0 - rr[1][2] * y1) * d[2];
        double z2 = y2 * d[2];
        double z1 = (y1 - rr[1][2] * z2) * d[1];
        double z0 = (y0 - rr[0][1] * z1 - rr[0][2] * z2) * d[0];
        inv = rsqrt_(z0 * z0 + z1 * z1 + z2 * z2);
        z0 *= inv; z1 *= inv; z2 *= inv;
        // as in dlt_null: stop on a change below 1e-13, or as soon as the error LEFT (change x rate) is below 1e-14
        const double e0 = z0 - x0, e1 = z1 - x1, e2 = z2 - x2;
        const double d2 = e0 * e0 + e1 * e1 + e2 * e2;
        x0 = z0; x1 = z1; x2 = z2;
        if (!(d2 > 1e-26) || !(d2 * d2 > 1e-28 * dprev)) { ok = (d2 == d2); break; }
        dprev = d2;
    }
    v[0] = x0; v[1] = x1; v[2] = x2;
    return ok;
}

// V(:,end) of svd(M) for a 3x3 M (column-major); M is not modified.
TVF_HD void null3(const double* M, double* v) {
    if (null3_qr(M, false, v)) return;
    double A[9], V[9], s[3];
#pragma unroll
    for (int i = 0; i < 9; ++i) A[i] = M[i];
    jacobi_svd3(A, V, s);
    v[0] = V[6]; v[1] = V[7]; v[2] = V[8];
}
// same for M.' without forming the transpose in memory
TVF_HD void null3_t(const double* M, double* v) {
    if (null3_qr(M, true, v)) return;
    double A[9], V[9], s[3];
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int r = 0; r < 3; ++r) A[r + 3 * c] = M[c + 3 * r];
    jacobi_svd3(A, V, s);
    v[0] = V[6]; v[1] = V[7]; v[2] = V[8];
}

// Full SVD of a (nearly) rank-2 3x3: U(:,1:2) from A*V/s, U(:,3) = u1 x u2.
TVF_HD void svd3_full(const double* M, double* U, double* s, double* V) {
    double A[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) A[i] = M[i];
    jacobi_svd3(A, V, s);
    const double i0 = rcp_(s[0]), i1 = rcp_(s[1]);
#pragma unroll
    for (int i = 0; i < 3; ++i) { U[i] = A[i] * i0; U[3 + i] = A[3 + i] * i1; }
    cross3(U, U + 3, U + 6);
}

// Epipoles of a TFT: e31 = common right null direction of the slices, e21 =
// common left null direction (linearTFT.m:71-79 / R_t_from_TFT.m:47-55).
// `slice_nulls` lets the warp kernel spread the six independent slice problems
// over lanes; the thread-level version below does all eight.
TVF_HD void epipole_from_nulls(const double* v0, const double* v1, const double* v2, double* e) {
    // rows of the stacked matrix are v_i.'  -> column-major M(r,c) = v_r[c]
    double M[9];
#pragma unroll
    for (int c = 0; c < 3; ++c) { M[0 + 3 * c] = v0[c]; M[1 + 3 * c] = v1[c]; M[2 + 3 * c] = v2[c]; }
    null3(M, e);
}

TVF_HD void tft_epipoles(const double* T, double* e21, double* e31) {
    double v[9];
    null3(T, v); null3(T + 9, v + 3); null3(T + 18, v + 6);
    epipole_from_nulls(v, v + 3, v + 6, e31);
    null3_t(T, v); null3_t(T + 9, v + 3); null3_t(T + 18, v + 6);
    epipole_from_nulls(v, v + 3, v + 6, e21);
}

// Branch-free orthonormal completion {e,u1,u2} of a unit vector (Duff et al. 2017).
TVF_HD void onb3(const double* e, double* u1, double* u2) {
    const double sg = copysign(1.0, e[2]);
    const double a = -rcp_(sg + e[2]);                 // |sg + e2| >= 1: no special cases (IEEE 1/x on the host build)
    const double b = e[0] * e[1] * a;
    u1[0] = 1.0 + sg * e[0] * e[0] * a; u1[1] = sg * b; u1[2] = -sg * e[0];
    u2[0] = b; u2[1] = sg + e[1] * e[1] * a; u2[2] = -e[1];
}

// ------------------------------------------------------------- transform_TFT
// TFT_methods/transform_TFT.m:36-49.  inverse!=0: T_new(:,:,i) = inv(M2)*(sum_r
// M1(r,i) T(:,:,r))*inv(M3).'; inverse==0: M2*(sum_r inv(M1)(r,i) T(:,:,r))*M3.'.
// Always renormalised to unit Frobenius norm (:49).
TVF_HD void transform_tft(const double* T, const double* M1, const double* M2, const double* M3,
                          int inverse, double* Tn) {
    double A1[9], A2[9], A3[9];
    if (inverse) {
#pragma unroll
        for (int i = 0; i < 9; ++i) A1[i] = M1[i];
        inv3(M2, A2); inv3(M3, A3);
    } else {
        inv3(M1, A1);
#pragma unroll
        for (int i = 0; i < 9; ++i) { A2[i] = M2[i]; A3[i] = M3[i]; }
    }
    double nrm = 0.0;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        double S[9], L[9];
#pragma unroll
        for (int e = 0; e < 9; ++e)
            S[e] = A1[0 + 3 * i] * T[e] + A1[1 + 3 * i] * T[9 + e] + A1[2 + 3 * i] * T[18 + e];
        mat3_mul(A2, S, L);
        mat3_mul_nt(L, A3, Tn + 9 * i);
#pragma unroll
        for (int e = 0; e < 9; ++e) nrm += Tn[9 * i + e] * Tn[9 * i + e];
    }
    const double inv = 1.0 / sqrt(nrm);
#pragma unroll
    for (int e = 0; e < 27; ++e) Tn[e] *= inv;
}

// ------------------------------------------------------------------ TFT_from_P
TVF_HD double det4_rows(const double* a, const double* b, const double* c, const double* d) {
    // determinant of the 4x4 whose rows are a,b,c,d
    const double s0 = a[0] * b[1] - a[1] * b[0], s1 = a[0] * b[2] - a[2] * b[0];
    const double s2 = a[0] * b[3] - a[3] * b[0], s3 = a[1] * b[2] - a[2] * b[1];
    const double s4 = a[1] * b[3] - a[3] * b[1], s5 = a[2] * b[3] - a[3] * b[2];
    const double c5 = c[2] * d[3] - c[3] * d[2], c4 = c[1] * d[3] - c[3] * d[1];
    const double c3 = c[1] * d[2] - c[2] * d[1], c2 = c[0] * d[3] - c[3] * d[0];
    const double c1 = c[0] * d[2] - c[2] * d[0], c0 = c[0] * d[1] - c[1] * d[0];
    return s0 * c5 - s1 * c4 + s2 * c3 + s3 * c2 - s4 * c1 + s5 * c0;
}

// TFT_methods/TFT_from_P.m:25-33; P* are 3x4 column-major.
TVF_HD void tft_from_p(const double* P1, const double* P2, const double* P3, double* T) {
    double r1[3][4], r2[3][4], r3[3][4];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) { r1[r][c] = P1[r + 3 * c]; r2[r][c] = P2[r + 3 * c]; r3[r][c] = P3[r + 3 * c]; }
    double nrm = 0.0;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const int ra = (i == 0) ? 1 : 0, rb = (i == 2) ? 1 : 2;
        const double sg = (i == 1) ? -1.0 : 1.0;
#pragma unroll
        for (int j = 0; j < 3; ++j)
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const double d = sg * det4_rows(r1[ra], r1[rb], r2[j], r3[k]);
                T[j + 3 * k + 9 * i] = d; nrm += d * d;
            }
    }
    const double inv = 1.0 / sqrt(nrm);
#pragma unroll
    for (int e = 0; e < 27; ++e) T[e] *= inv;
}

// --------------------------------------------------------------------- DLT
// Smallest right singular vector of an Mx4 system (triangulation3D.m:55-62):
// Householder QR, then inverse iteration with R (never forms A'A, so the
// conditioning is that of the SVD route).  rows[r][c]; destroyed.
template <int M>
TVF_HD void dlt_null(double (&a)[M][4], double* x, int* iters = nullptr) {
    double r[4][4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (M == 4 && k == 3) {          // a 1 x 1 reflection: alpha = -x1 exactly, nothing left to update (saves a sqrt and a reciprocal)
            r[3][3] = -a[3][3];
            break;
        }
        double sig = 0.0;
#pragma unroll
        for (int i = k; i < M; ++i) sig += a[i][k] * a[i][k];
        const double nrm = sqrt_(sig);
        const double x1 = a[k][k];
        const double alpha = -copysign(nrm, x1);
        const double den = sig - alpha * x1;          // = v'v / 2 >= 0
        const double f = (den > 0.0) ? rcp_(den) : 0.0;
        const double vk = x1 - alpha;
#pragma unroll
        for (int c = k + 1; c < 4; ++c) {
            double sdot = vk * a[k][c];
#pragma unroll
            for (int i = k + 1; i < M; ++i) sdot += a[i][k] * a[i][c];
            sdot *= f;
            a[k][c] -= sdot * vk;
#pragma unroll
            for (int i = k + 1; i < M; ++i) a[i][c] -= sdot * a[i][k];
        }
        r[k][k] = alpha;
#pragma unroll
        for (int c = k + 1; c < 4; ++c) r[k][c] = a[k][c];
    }
    // guard exactly singular pivots
    const double rmax = fmax(fmax(fabs(r[0][0]), fabs(r[1][1])), fmax(fabs(r[2][2]), fabs(r[3][3])));
    const double tiny = 1e-300 + 1e-18 * rmax;
    double d[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const double p = (fabs(r[k][k]) < tiny) ? copysign(tiny, r[k][k]) : r[k][k];
        d[k] = rcp_(p);
    }
    // start vector: R x = e4
    double x0, x1, x2, x3;
    x3 = d[3];
    x2 = -(r[2][3] * x3) * d[2];
    x1 = -(r[1][2] * x2 + r[1][3] * x3) * d[1];
    x0 = -(r[0][1] * x1 + r[0][2] * x2 + r[0][3] * x3) * d[0];
    double inv = rsqrt_(x0 * x0 + x1 * x1 + x2 * x2 + x3 * x3);
    x0 *= inv; x1 *= inv; x2 *= inv; x3 *= inv;
    int it = 0;
    double dprev = 0.0;               // squared change of the previous step (0: no rate estimate yet)
    for (; it < 40; ++it) {
        const double y0 = x0 * d[0];
        const double y1 = (x1 - r[0][1] * y0) * d[1];
        const double y2 = (x2 - r[0][2] * y0 - r[1][2] * y1) * d[2];
        const double y3 = (x3 - r[0][3] * y0 - r[1][3] * y1 - r[2][3] * y2) * d[3];
        double z3 = y3 * d[3];
        double z2 = (y2 - r[2][3] * z3) * d[2];
        double z1 = (y1 - r[1][2] * z2 - r[1][3] * z3) * d[1];
        double z0 = (y0 - r[0][1] * z1 - r[0][2] * z2 - r[0][3] * z3) * d[0];
        inv = rsqrt_(z0 * z0 + z1 * z1 + z2 * z2 + z3 * z3);
        z0 *= inv; z1 *= inv; z2 *= inv; z3 *= inv;
        // squared change d2 = |z - x|^2.  Inverse iteration converges linearly with rate rho = (s4/s3)^2 ~ d2/dprev
        // (in squares: rho^2), so the error LEFT in z is ~ |z - x| * rho: stop as soon as that product is below 1e-14
        // instead of running one more step only to see a change below 1e-13.  (All terms are squares: sign symmetric.)
        const double e0 = z0 - x0, e1 = z1 - x1, e2 = z2 - x2, e3 = z3 - x3;
        const double d2 = e0 * e0 + e1 * e1 + e2 * e2 + e3 * e3;
        x0 = z0; x1 = z1; x2 = z2; x3 = z3;
        if (!(d2 > 1e-26) || !(d2 * d2 > 1e-28 * dprev)) { ++it; break; }
        dprev = d2;
    }
    x[0] = x0; x[1] = x1; x[2] = x2; x[3] = x3;
    if (iters) *iters = it;
}

// ------------------------------------------------- certified depth signs of a two-view DLT
// The cheirality test of recover_R_t (R_t_from_TFT.m:98-100) uses only the SIGNS of two depths of the DLT solution X:
// sign(X3/X4) and sign(([R t] X)_3 / X4).  This routine gets them from the 4 x 4 normal equations (Cholesky + inverse
// iteration: ~45 % fewer FP64 operations than the Householder route of dlt_null) and CERTIFIES them: it answers only
// when (a) the three leading Cholesky pivots are >= 1e-3 of the largest diagonal entry, which bounds lambda_3(A'A) from
// below by 1e-9/9 of it (interlacing) and with it the error of the squared-condition route by ~4e-6 in the unit vector
// X; (b) the iteration has visibly converged (change of the last step <= 1e-5, i.e. a spectral gap is present); and (c)
// both sign-deciding products are at least 1e-3 away from zero (|X| = 1).  Otherwise it returns false and the caller
// runs the accurate dlt_null.  The votes are therefore the ones the accurate route gives -- checked integer for integer
// against it on the host (tests/test_hostcheck.py) and against the oracle on the GPU.
TVF_HD bool dlt4_depth_signs(const double (&a)[4][4], const double* r3, double tz, int* s_x, int* s_z) {
    double g[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) g[i][j] = a[0][i] * a[0][j] + a[1][i] * a[1][j] + a[2][i] * a[2][j] + a[3][i] * a[3][j];
    const double gmax = fmax(fmax(g[0][0], g[1][1]), fmax(g[2][2], g[3][3]));
    const double pmin = 1.0e-3 * gmax;
    if (!(g[0][0] >= pmin)) return false;                         // also catches NaN
    const double i0 = rsqrt_(g[0][0]);
    const double l10 = g[1][0] * i0, l20 = g[2][0] * i0, l30 = g[3][0] * i0;
    const double p1 = g[1][1] - l10 * l10;
    if (!(p1 >= pmin)) return false;
    const double i1 = rsqrt_(p1);
    const double l21 = (g[2][1] - l20 * l10) * i1, l31 = (g[3][1] - l30 * l10) * i1;
    const double p2 = g[2][2] - l20 * l20 - l21 * l21;
    if (!(p2 >= pmin)) return false;
    const double i2 = rsqrt_(p2);
    const double l32 = (g[3][2] - l30 * l20 - l31 * l21) * i2;
    double p3 = g[3][3] - l30 * l30 - l31 * l31 - l32 * l32;
    p3 = (p3 >= 1.0e-14 * gmax) ? p3 : 1.0e-14 * gmax;            // noise-free data: A'A is singular, X is its null vector
    const double i3 = rsqrt_(p3);
    // start: L' x = e4, then inverse iteration x <- (L L')^-1 x
    double x3 = i3;
    double x2 = -(l32 * x3) * i2;
    double x1 = -(l21 * x2 + l31 * x3) * i1;
    double x0 = -(l10 * x1 + l20 * x2 + l30 * x3) * i0;
    double inv = rsqrt_(x0 * x0 + x1 * x1 + x2 * x2 + x3 * x3);
    x0 *= inv; x1 *= inv; x2 *= inv; x3 *= inv;
    double d2 = 1.0;
#pragma unroll
    for (int it = 0; it < 2; ++it) {
        const double y0 = x0 * i0;
        const double y1 = (x1 - l10 * y0) * i1;
        const double y2 = (x2 - l20 * y0 - l21 * y1) * i2;
        const double y3 = (x3 - l30 * y0 - l31 * y1 - l32 * y2) * i3;
        double z3 = y3 * i3;
        double z2 = (y2 - l32 * z3) * i2;
        double z1 = (y1 - l21 * z2 - l31 * z3) * i1;
        double z0 = (y0 - l10 * z1 - l20 * z2 - l30 * z3) * i0;
        inv = rsqrt_(z0 * z0 + z1 * z1 + z2 * z2 + z3 * z3);
        z0 *= inv; z1 *= inv; z2 *= inv; z3 *= inv;
        const double e0 = z0 - x0, e1 = z1 - x1, e2 = z2 - x2, e3 = z3 - x3;
        d2 = e0 * e0 + e1 * e1 + e2 * e2 + e3 * e3;
        x0 = z0; x1 = z1; x2 = z2; x3 = z3;
        if (d2 <= 1.0e-10) break;
    }
    if (!(d2 <= 1.0e-10)) return false;
    const double q1 = x2 * x3;                                    // sign(X3 / X4)
    const double zc = r3[0] * x0 + r3[1] * x1 + r3[2] * x2 + tz * x3;
    const double q2 = zc * x3;                                    // sign(([R t] X)_3 / X4)
    if (!(fabs(q1) >= 1.0e-3) || !(fabs(q2) >= 1.0e-3)) return false;
    *s_x = (q1 > 0.0) ? 1 : -1;
    *s_z = (q2 > 0.0) ? 1 : -1;
    return true;
}

// ------------------------------------------------- depth signs from the ray / plane intersection, certified
// A cheaper certificate for the same two signs, tried first.  Let B = the first three rows of the 4 x 4 DLT system A (both
// rows of view 1 and the first row of the candidate view) and rd its fourth row.  The 4-D cross product Xt of B's rows is
// the null vector of B -- geometrically the point where the ray of view 1 meets the plane that rd's sibling row
// back-projects -- and costs twelve multiply-adds from the 2 x 2 minors of the view-1 rows, which all four candidates of
// a point share.  With xh = Xt/|Xt| and v the smallest right singular vector of A:
//   |A xh| = |rd.Xt| / |Xt|                                    (B xh = 0),
//   |A xh|^2 = sum_i sigma_i^2 (v_i.xh)^2 >= sigma_3(A)^2 sin^2(angle(xh, v))
//   sigma_3(A) >= s_3(B)                                        (interlacing: B is A without a row)
//   s_3(B) = |Xt| / (s_1 s_2) >= 2 |Xt| / |B|_F^2               (|Xt| = s_1 s_2 s_3, AM-GM)
// so sin(angle) <= eta = |rd.Xt| |B|_F^2 / (2 |Xt|^2).  For eta <= 0.2 the distance between the unit vectors is
// <= 1.01 eta =: d, the sign-deciding products move by at most  |D(x3 x4)| <= d + d^2/2  and
// |D(z x4)| <= sqrt(2) d (2 + d)  (|[r3 tz]| <= sqrt 2), and the routine answers only when both products of xh exceed
// 2.1 d resp. 3.2 d plus an absolute 1e-6 (rounding of the cofactors, guarded by |Xt|^2 >= 1e-12 |B|_F^6, and of the
// accurate route itself).  Everything is written without a division; any NaN fails a comparison and returns false.
// m7: minors M01, M02, M03, M12, M13, M23 of the view-1 rows (M_jk = a_j b_k - a_k b_j) and |a|^2 + |b|^2.
// AFF: the view-1 camera is K1*[I | 0] (always, in this pipeline), so both of its rows end in an exact zero: the three minors
// with index 3 vanish and three of the four cofactors are single products -- the same values as the general form.
template <bool AFF = false>
TVF_HD void dlt_row_minors(const double* ra, const double* rb, double* m7) {
    m7[0] = ra[0] * rb[1] - ra[1] * rb[0]; m7[1] = ra[0] * rb[2] - ra[2] * rb[0];
    m7[3] = ra[1] * rb[2] - ra[2] * rb[1];
    if (AFF) {
        m7[2] = 0.0; m7[4] = 0.0; m7[5] = 0.0;
        m7[6] = (ra[0] * ra[0] + ra[1] * ra[1] + ra[2] * ra[2]) + (rb[0] * rb[0] + rb[1] * rb[1] + rb[2] * rb[2]);
    } else {
        m7[2] = ra[0] * rb[3] - ra[3] * rb[0]; m7[4] = ra[1] * rb[3] - ra[3] * rb[1]; m7[5] = ra[2] * rb[3] - ra[3] * rb[2];
        m7[6] = (ra[0] * ra[0] + ra[1] * ra[1] + ra[2] * ra[2] + ra[3] * ra[3]) + (rb[0] * rb[0] + rb[1] * rb[1] + rb[2] * rb[2] + rb[3] * rb[3]);
    }
}
template <bool AFF = false>
TVF_HD bool dlt4_depth_signs_ray(const double* m7, const double* rc, const double* rd, const double* r3, double tz,
                                 int* s_x, int* s_z) {
    const double M01 = m7[0], M02 = m7[1], M03 = m7[2], M12 = m7[3], M13 = m7[4], M23 = m7[5];
    const double X0 = AFF ? rc[3] * M12 : rc[1] * M23 - rc[2] * M13 + rc[3] * M12;
    const double X1 = AFF ? -(rc[3] * M02) : -(rc[0] * M23 - rc[2] * M03 + rc[3] * M02);
    const double X2 = AFF ? rc[3] * M01 : rc[0] * M13 - rc[1] * M03 + rc[3] * M01;
    const double X3 = -(rc[0] * M12 - rc[1] * M02 + rc[2] * M01);
    const double xx = X0 * X0 + X1 * X1 + X2 * X2 + X3 * X3;
    const double b2 = m7[6] + (rc[0] * rc[0] + rc[1] * rc[1] + rc[2] * rc[2] + rc[3] * rc[3]);
    const double rho = rd[0] * X0 + rd[1] * X1 + rd[2] * X2 + rd[3] * X3;
    const double rb2 = fabs(rho) * b2;                            // = 2 eta |Xt|^2
    if (!(rb2 < 0.4 * xx)) return false;                          // eta < 0.2 (also catches NaN and xx = 0)
    if (!(xx >= 1.0e-12 * (b2 * b2 * b2))) return false;          // cofactors not dominated by cancellation
    const double q1 = X2 * X3;                                    // sign(X3 / X4), times |Xt|^2
    const double zc = r3[0] * X0 + r3[1] * X1 + r3[2] * X2 + tz * X3;
    const double q2 = zc * X3;                                    // sign(([R t] X)_3 / X4), times |Xt|^2
    const double floor_ = 1.0e-6 * xx;
    if (!(fabs(q1) >= 1.0605 * rb2 + floor_)) return false;       // 2.1 * 1.01 eta
    if (!(fabs(q2) >= 1.616 * rb2 + floor_)) return false;        // 3.2 * 1.01 eta
    *s_x = (q1 > 0.0) ? 1 : -1;
    *s_z = (q2 > 0.0) ? 1 : -1;
    return true;
}

// rows of the DLT system contributed by one view (triangulation3D.m:58-59):
// [0 -1 y; 1 0 -x]*P  ->  (-P(2,:) + y*P(3,:) ; P(1,:) - x*P(3,:)).  P 3x4 column-major.
TVF_HD void dlt_rows(const double* P, double x, double y, double* row_a, double* row_b) {
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        row_a[c] = y * P[2 + 3 * c] - P[1 + 3 * c];
        row_b[c] = P[0 + 3 * c] - x * P[2 + 3 * c];
    }
}

// x = P*[X;1]-style product for a homogeneous 4-vector: out = P*X4
TVF_HD void cam_apply(const double* P, const double* X, double* out) {
#pragma unroll
    for (int r = 0; r < 3; ++r)
        out[r] = P[r] * X[0] + P[r + 3] * X[1] + P[r + 6] * X[2] + P[r + 9] * X[3];
}

// ------------------------------------------------------- essential -> R, Rp, t
// R_t_from_TFT.m:84-88 / LinearFPoseEstimation.m:87-91.
TVF_HD void decompose_essential(const double* E, double* R, double* Rp, double* t) {
    double U[9], s[3], V[9];
    svd3_full(E, U, s, V);
    // U*W = [u2, -u1, u3];  U*W.' = [-u2, u1, u3]
    double UW[9], UWt[9];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        UW[i] = U[3 + i]; UW[3 + i] = -U[i]; UW[6 + i] = U[6 + i];
        UWt[i] = -U[3 + i]; UWt[3 + i] = U[i]; UWt[6 + i] = U[6 + i];
    }
    mat3_mul_nt(UW, V, R);
    mat3_mul_nt(UWt, V, Rp);
    const double sr = sign_(det3(R)), sp = sign_(det3(Rp));
#pragma unroll
    for (int i = 0; i < 9; ++i) { R[i] *= sr; Rp[i] *= sp; }
    t[0] = U[6]; t[1] = U[7]; t[2] = U[8];
}

// --------------------------------------------------------------------- AngError
// auxiliar_functions/AngError.m:25,28 incl. MATLAB's complex acos for |x|>1.
TVF_HD double matlab_abs_acos(double x) {
    if (x > 1.0) return log(x + sqrt(x * x - 1.0));                    // |i*acosh(x)|
    if (x < -1.0) {
        const double a = log(-x + sqrt(x * x - 1.0));
        return sqrt(3.14159265358979323846 * 3.14159265358979323846 + a * a);
    }
    return acos(x);
}

TVF_HD void ang_error(const double* Rt_true, const double* Rt_est, double* rot_err, double* t_err) {
    double tr = 0.0;
#pragma unroll
    for (int i = 0; i < 9; ++i) tr += Rt_true[i] * Rt_est[i];          // trace(R_true.'*R_est)
    const double k = 180.0 / 3.14159265358979323846;
    *rot_err = fabs(k * matlab_abs_acos((tr - 1.0) / 2.0));
    const double* a = Rt_est + 9; const double* b = Rt_true + 9;
    const double na = sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
    const double nb = sqrt(b[0] * b[0] + b[1] * b[1] + b[2] * b[2]);
    const double d = (a[0] / na) * (b[0] / nb) + (a[1] / na) * (b[1] / nb) + (a[2] / na) * (b[2] / nb);
    *t_err = fabs(k * matlab_abs_acos(d));
}

}  // namespace tvf
