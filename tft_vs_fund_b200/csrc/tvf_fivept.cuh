// tvf_fivept.cuh -- the calibrated five-point minimal three-view pose (tvf_five_point_pose, RANSAC method 9): Nistér's
// five-point essential matrix for views 1-2 (Sturm sequences on the degree-10 polynomial), the F path's decomposition
// and two-view DLT, and a Lambda Twist P3P for view 3.  Host/device functions, so five_point_pose_kernel and the CPU
// check in tests/hostcheck/five_point_hostcheck.cpp share one source.  The rules are written out in include/tvf.h.
#pragma once
#include "tvf_pose.cuh"

namespace tvf {

constexpr int FP_MAX_E = 10;          // real roots of the degree-10 polynomial, at most

// ---------------------------------------------------------------- polynomials in one variable, p[i] of x^i
TVF_HD double fp_horner(const double* p, int d, double x) {
    double v = p[d];
    for (int i = d - 1; i >= 0; --i) v = v * x + p[i];
    return v;
}

// c (degree da + db) = a (degree da) * b (degree db)
TVF_HD void fp_pmul(const double* a, int da, const double* b, int db, double* c) {
    for (int i = 0; i <= da + db; ++i) c[i] = 0.0;
    for (int i = 0; i <= da; ++i)
        for (int j = 0; j <= db; ++j) c[i + j] += a[i] * b[j];
}

// sign changes of the Sturm sequence s[0..m-1] (degrees deg[]) at x; zeros are skipped
TVF_HD int fp_sturm_changes(const double (*s)[11], const int* deg, int m, double x) {
    int changes = 0;
    double prev = 0.0;
    for (int k = 0; k < m; ++k) {
        const double v = fp_horner(s[k], deg[k], x);
        if (v != 0.0) {
            if (prev != 0.0 && ((v > 0.0) != (prev > 0.0))) ++changes;
            prev = v;
        }
    }
    return changes;
}

// The distinct real roots of p (degree d <= 10), ascending; returns their count.  Leading coefficients below 1e-14 of
// the largest are dropped.  The Sturm sequence of the monic polynomial isolates the roots by bisection; a root alone in
// its interval with a sign change is polished by safeguarded Newton steps, and one without (an even multiplicity) by
// Sturm bisection to the last bits.  Roots that stay together down to a width of 1e-15 relative are reported once each
// at that interval's midpoint.
TVF_HD int fp_real_roots(const double* p_in, int d, double* roots) {
    double s[11][11];
    int deg[11];
    double mx = 0.0;
    for (int i = 0; i <= d; ++i) mx = fmax(mx, fabs(p_in[i]));
    if (!(mx > 0.0) || !isfinite(mx)) return 0;
    while (d > 0 && fabs(p_in[d]) <= 1e-14 * mx) --d;
    if (d < 1) return 0;
    for (int i = 0; i <= d; ++i) s[0][i] = p_in[i] / p_in[d];
    deg[0] = d;
    double bound = 0.0;                                   // Cauchy: every root lies within 1 + max |a_i / a_d|
    for (int i = 0; i < d; ++i) bound = fmax(bound, fabs(s[0][i]));
    bound += 1.0;
    for (int i = 1; i <= d; ++i) s[1][i - 1] = i * s[0][i] / d;
    deg[1] = d - 1;
    int m = 2;
    while (deg[m - 1] > 0) {                              // s[m] = -rem(s[m-2], s[m-1]), scaled to max |coefficient| 1
        double r[11];
        const int da = deg[m - 2], db = deg[m - 1];
        double amax = 0.0;
        for (int i = 0; i <= da; ++i) { r[i] = s[m - 2][i]; amax = fmax(amax, fabs(r[i])); }
        for (int k = da - db; k >= 0; --k) {
            const double q = r[k + db] / s[m - 1][db];
            for (int j = 0; j <= db; ++j) r[k + j] -= q * s[m - 1][j];
            r[k + db] = 0.0;
        }
        int dr = db - 1;
        double rmax = 0.0;
        for (int i = 0; i <= dr; ++i) rmax = fmax(rmax, fabs(r[i]));
        if (!(rmax > 1e-13 * amax)) break;                // the remainder vanishes: s[m-1] is the gcd (a multiple root)
        while (dr > 0 && fabs(r[dr]) <= 1e-13 * rmax) --dr;
        for (int i = 0; i <= dr; ++i) s[m][i] = -r[i] / rmax;
        deg[m] = dr;
        ++m;
    }
    // intervals (lo, hi] holding at least one root, on a stack: at most one pending interval per root
    double slo[11], shi[11];
    int svlo[11], svhi[11], top = 0, count = 0;
    slo[0] = -bound; shi[0] = bound;
    svlo[0] = fp_sturm_changes(s, deg, m, -bound); svhi[0] = fp_sturm_changes(s, deg, m, bound);
    if (svlo[0] - svhi[0] > 0) top = 1;
    while (top > 0 && count < d) {
        --top;
        double lo = slo[top], hi = shi[top];
        int vlo = svlo[top], vhi = svhi[top];
        const int k = vlo - vhi;
        const double width_tol = 1e-15 * fmax(fabs(lo), fabs(hi)) + 1e-300;
        if (k > 1) {
            if (hi - lo <= width_tol) {
                for (int j = 0; j < k && count < d; ++j) roots[count++] = 0.5 * (lo + hi);
                continue;
            }
            const double mid = 0.5 * (lo + hi);
            const int vm = fp_sturm_changes(s, deg, m, mid);
            if (vm - vhi > 0 && top < 11) { slo[top] = mid; shi[top] = hi; svlo[top] = vm; svhi[top] = vhi; ++top; }
            if (vlo - vm > 0 && top < 11) { slo[top] = lo; shi[top] = mid; svlo[top] = vlo; svhi[top] = vm; ++top; }
            continue;
        }
        double flo = fp_horner(s[0], d, lo), fhi = fp_horner(s[0], d, hi);
        double x;
        if (flo == 0.0 || fhi == 0.0 || (flo > 0.0) == (fhi > 0.0)) {
            // no sign change: an even multiplicity (or the root sits on an end), so bisect the Sturm count
            for (int it = 0; it < 200 && hi - lo > 1e-15 * fmax(fabs(lo), fabs(hi)) + 1e-300; ++it) {
                const double mid = 0.5 * (lo + hi);
                if (vlo - fp_sturm_changes(s, deg, m, mid) > 0) hi = mid; else { lo = mid; vlo = fp_sturm_changes(s, deg, m, mid); }
            }
            x = 0.5 * (lo + hi);
        } else {
            x = 0.5 * (lo + hi);
            for (int it = 0; it < 200; ++it) {
                double f = s[0][d], df = 0.0;
                for (int i = d - 1; i >= 0; --i) { df = df * x + f; f = f * x + s[0][i]; }
                if (f == 0.0) break;
                if ((f > 0.0) == (flo > 0.0)) lo = x; else hi = x;
                double xn = x - f / df;
                if (!(xn > lo && xn < hi)) xn = 0.5 * (lo + hi);
                const bool done = fabs(xn - x) <= 4e-16 * fabs(x) + 1e-300 || hi - lo <= 4e-16 * fmax(fabs(lo), fabs(hi));
                x = xn;
                if (done) break;
            }
        }
        roots[count++] = x;
    }
    return count;
}

// ---------------------------------------------------------------- polynomials in x, y, z of degree <= 3
// The 20 monomials in Nistér's order: the first 10 are eliminated, rows 4..9 of the reduced matrix lead with
// x^2 z, x^2, y^2 z, y^2, xyz, xy.  FP_MUL[i][v]: the index of monomial i times x, y, z (v = 0, 1, 2), -1 above degree 3.
//   0 x3  1 y3  2 x2y  3 xy2  4 x2z  5 x2  6 y2z  7 y2  8 xyz  9 xy  10 xz2  11 xz  12 x  13 yz2  14 yz  15 y
//   16 z3  17 z2  18 z  19 1
constexpr int FP_X = 12, FP_Y = 15, FP_Z = 18, FP_ONE = 19;
TVF_HD int fp_mul_index(int i, int v) {
    constexpr signed char T[20][3] = {
        {-1, -1, -1}, {-1, -1, -1}, {-1, -1, -1}, {-1, -1, -1}, {-1, -1, -1}, {0, 2, 4}, {-1, -1, -1}, {3, 1, 6},
        {-1, -1, -1}, {2, 3, 8}, {-1, -1, -1}, {4, 8, 10}, {5, 9, 11}, {-1, -1, -1}, {8, 6, 13}, {9, 7, 14},
        {-1, -1, -1}, {10, 13, 16}, {11, 14, 17}, {12, 15, 18}};
    return T[i][v];
}

// out += a * l, a of degree <= 2 in the 20-basis, l = (lx, ly, lz, l1) linear
TVF_HD void fp_mul_lin(const double* a, const double* l, double* out) {
    for (int i = 5; i < 20; ++i) {
        const double c = a[i];
        if (c == 0.0) continue;
        for (int v = 0; v < 3; ++v) {
            const int j = fp_mul_index(i, v);
            if (j >= 0) out[j] += c * l[v];
        }
        out[i] += c * l[3];
    }
}

// the linear entry E(e) = x X(e) + y Y(e) + z Z(e) + W(e) as a 20-basis polynomial
TVF_HD void fp_lin20(const double* l, double* a) {
    for (int i = 0; i < 20; ++i) a[i] = 0.0;
    a[FP_X] = l[0]; a[FP_Y] = l[1]; a[FP_Z] = l[2]; a[FP_ONE] = l[3];
}

// The essential matrices of five calibrated rays q1, q2 (5 x 3 each, q2' E q1 = 0): up to 10, each 3 x 3 column-major,
// unit Frobenius norm, the largest-magnitude entry positive (the first of equal ones), ordered by ascending root z; the
// rest NaN.  *nE: the number of real roots.  Returns false when the elimination meets a zero (or NaN) pivot.
TVF_HD bool five_point_essentials(const double (*q1)[3], const double (*q2)[3], double* Eout, int* nE) {
    for (int e = 0; e < 9 * FP_MAX_E; ++e) Eout[e] = (double)NAN;
    *nE = 0;
    // 1. null space of the 5 x 9 epipolar system: Householder QR of its transpose M (9 x 5), Q's last four columns
    double M[9][5], v[5][9];
    for (int j = 0; j < 5; ++j)
        for (int c = 0; c < 3; ++c)
            for (int r = 0; r < 3; ++r) M[r + 3 * c][j] = q2[j][r] * q1[j][c];
    for (int k = 0; k < 5; ++k) {
        double sig = 0.0;
        for (int i = k; i < 9; ++i) sig += M[i][k] * M[i][k];
        const double alpha = -copysign(sqrt(sig), M[k][k]);
        for (int i = 0; i < 9; ++i) v[k][i] = i < k ? 0.0 : M[i][k];
        v[k][k] -= alpha;
        double vv = 0.0;
        for (int i = k; i < 9; ++i) vv += v[k][i] * v[k][i];
        const double f = vv > 0.0 ? 2.0 / vv : 0.0;
        for (int c = k; c < 5; ++c) {
            double dot = 0.0;
            for (int i = k; i < 9; ++i) dot += v[k][i] * M[i][c];
            dot *= f;
            for (int i = k; i < 9; ++i) M[i][c] -= dot * v[k][i];
        }
        for (int i = 0; i < 9; ++i) v[k][i] *= sqrt(f);         // H_k = I - v v'
    }
    double N[4][9];                                            // X, Y, Z, W = Q e_5 .. Q e_8
    for (int j = 0; j < 4; ++j) {
        for (int i = 0; i < 9; ++i) N[j][i] = (i == j + 5) ? 1.0 : 0.0;
        for (int k = 4; k >= 0; --k) {
            double dot = 0.0;
            for (int i = k; i < 9; ++i) dot += v[k][i] * N[j][i];
            for (int i = k; i < 9; ++i) N[j][i] -= dot * v[k][i];
        }
    }
    // 2. the ten cubic constraints det E = 0 and 2 E E' E - tr(E E') E = 0 as a 10 x 20 matrix
    double L[9][4];
    for (int e = 0; e < 9; ++e)
        for (int j = 0; j < 4; ++j) L[e][j] = N[j][e];
    double A[10][20];
    for (int r = 0; r < 10; ++r)
        for (int c = 0; c < 20; ++c) A[r][c] = 0.0;
    {   // det E = sum_c E(0,c) * cofactor(0,c)
        for (int c = 0; c < 3; ++c) {
            const int c1 = (c + 1) % 3, c2 = (c + 2) % 3;
            double a[20], cof[20];
            fp_lin20(L[1 + 3 * c1], a);
            for (int i = 0; i < 20; ++i) cof[i] = 0.0;
            fp_mul_lin(a, L[2 + 3 * c2], cof);
            fp_lin20(L[1 + 3 * c2], a);
            for (int i = 0; i < 20; ++i) a[i] = -a[i];
            fp_mul_lin(a, L[2 + 3 * c1], cof);
            fp_mul_lin(cof, L[0 + 3 * c], A[0]);
        }
    }
    double EEt[6][20];                                         // (0,0) (1,1) (2,2) (0,1) (0,2) (1,2)
    const int pr[6] = {0, 1, 2, 0, 0, 1}, pc[6] = {0, 1, 2, 1, 2, 2};
    for (int k = 0; k < 6; ++k) {
        for (int i = 0; i < 20; ++i) EEt[k][i] = 0.0;
        for (int c = 0; c < 3; ++c) {
            double a[20];
            fp_lin20(L[pr[k] + 3 * c], a);
            fp_mul_lin(a, L[pc[k] + 3 * c], EEt[k]);
        }
    }
    double tr[20];
    for (int i = 0; i < 20; ++i) tr[i] = EEt[0][i] + EEt[1][i] + EEt[2][i];
    for (int c = 0; c < 3; ++c)
        for (int r = 0; r < 3; ++r) {
            double* row = A[1 + r + 3 * c];
            for (int k = 0; k < 3; ++k) {                      // 2 (E E')(r,k) E(k,c)
                const int a = r < k ? r : k, b = r < k ? k : r;
                const int idx = a == b ? a : (a == 0 ? (b == 1 ? 3 : 4) : 5);
                double t[20];
                for (int i = 0; i < 20; ++i) t[i] = 2.0 * EEt[idx][i];
                fp_mul_lin(t, L[k + 3 * c], row);
            }
            double t[20];
            for (int i = 0; i < 20; ++i) t[i] = -tr[i];
            fp_mul_lin(t, L[r + 3 * c], row);
        }
    // 3. Gauss-Jordan with partial pivoting on the first ten columns
    for (int c = 0; c < 10; ++c) {
        int p = c;
        double best = 0.0;
        for (int r = c; r < 10; ++r)
            if (fabs(A[r][c]) > best) { best = fabs(A[r][c]); p = r; }
        if (!(best > 0.0)) return false;
        if (p != c)
            for (int j = 0; j < 20; ++j) { const double t = A[c][j]; A[c][j] = A[p][j]; A[p][j] = t; }
        const double inv = 1.0 / A[c][c];
        for (int j = c; j < 20; ++j) A[c][j] *= inv;
        for (int r = 0; r < 10; ++r) {
            if (r == c) continue;
            const double f = A[r][c];
            if (f == 0.0) continue;
            for (int j = c; j < 20; ++j) A[r][j] -= f * A[c][j];
        }
    }
    // 4. <k> = <e> - z<f>, <l> = <g> - z<h>, <m> = <i> - z<j>: a 3 x 3 matrix B(z) acting on (x, y, 1); columns are
    // polynomials in z of degrees 3, 3, 4
    double B[3][3][5];
    for (int r = 0; r < 3; ++r) {
        const double* e = A[4 + 2 * r];
        const double* f = A[5 + 2 * r];
        const double px[2][3] = {{e[12], e[11], e[10]}, {f[12], f[11], f[10]}};
        const double py[2][3] = {{e[15], e[14], e[13]}, {f[15], f[14], f[13]}};
        const double p1[2][4] = {{e[19], e[18], e[17], e[16]}, {f[19], f[18], f[17], f[16]}};
        for (int i = 0; i < 5; ++i) { B[r][0][i] = 0.0; B[r][1][i] = 0.0; B[r][2][i] = 0.0; }
        for (int i = 0; i < 3; ++i) { B[r][0][i] += px[0][i]; B[r][0][i + 1] -= px[1][i]; B[r][1][i] += py[0][i]; B[r][1][i + 1] -= py[1][i]; }
        for (int i = 0; i < 4; ++i) { B[r][2][i] += p1[0][i]; B[r][2][i + 1] -= p1[1][i]; }
    }
    const int dB[3] = {3, 3, 4};
    double poly[11];
    for (int i = 0; i < 11; ++i) poly[i] = 0.0;
    for (int c = 0; c < 3; ++c) {                              // det B = sum_c B(0,c) * cofactor(0,c)
        const int c1 = (c + 1) % 3, c2 = (c + 2) % 3;
        double t1[8], t2[8], cof[8], term[11];
        fp_pmul(B[1][c1], dB[c1], B[2][c2], dB[c2], t1);
        fp_pmul(B[1][c2], dB[c2], B[2][c1], dB[c1], t2);
        const int dc = dB[c1] + dB[c2];
        for (int i = 0; i <= dc; ++i) cof[i] = t1[i] - t2[i];
        fp_pmul(B[0][c], dB[c], cof, dc, term);
        for (int i = 0; i <= 10; ++i) poly[i] += term[i];
    }
    double zs[10];
    const int nz = fp_real_roots(poly, 10, zs);
    *nE = nz;
    // 5. an E per root: (x, y, 1) spans the null space of B(z), the largest cross product of two of its rows
    for (int k = 0; k < nz; ++k) {
        const double z = zs[k];
        double Bz[3][3];
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) Bz[r][c] = fp_horner(B[r][c], dB[c], z);
        double best[3] = {0.0, 0.0, 0.0}, bn = -1.0;
        for (int pair = 0; pair < 3; ++pair) {
            const int a = pair == 2 ? 1 : 0, b = pair == 0 ? 1 : 2;
            double cr[3];
            cross3(Bz[a], Bz[b], cr);
            const double nn = cr[0] * cr[0] + cr[1] * cr[1] + cr[2] * cr[2];
            if (nn > bn) { bn = nn; best[0] = cr[0]; best[1] = cr[1]; best[2] = cr[2]; }
        }
        const double x = best[0] / best[2], y = best[1] / best[2];
        double E[9], nrm = 0.0;
        for (int e = 0; e < 9; ++e) { E[e] = x * N[0][e] + y * N[1][e] + z * N[2][e] + N[3][e]; nrm += E[e] * E[e]; }
        int big = 0;
        for (int e = 1; e < 9; ++e)
            if (fabs(E[e]) > fabs(E[big])) big = e;
        const double sc = copysign(1.0 / sqrt(nrm), E[big]);
        for (int e = 0; e < 9; ++e) Eout[9 * k + e] = E[e] * sc;
    }
    return true;
}

// ---------------------------------------------------------------- P3P (Lambda Twist)
// Camera poses (R, t: x_cam = R X + t) that map the three points X (3 x 3, one per row) onto the rays y (unit vectors,
// one per row) with positive depths: up to 4, returned count.  With cos c_ij = y_i . y_j and a_ij = |X_i - X_j|^2 the
// depths satisfy lambda' M_ij lambda = a_ij; D0 = (a23 M12 - a12 M23) + g (a13 M23 - a23 M13) is made singular by the
// root g of a cubic at which D0 is most indefinite, so lambda' D0 lambda = 0 splits into two planes (eigenvectors of
// D0); on each plane a13 f12 - a12 f13 = 0 is a homogeneous quadratic, and f12 = a12 sets the scale.
TVF_HD void fp_sym_null(const double (*D)[3], double* v) {          // unit null vector of a rank-2 3 x 3 matrix
    double bn = -1.0;
    for (int pair = 0; pair < 3; ++pair) {
        const int a = pair == 2 ? 1 : 0, b = pair == 0 ? 1 : 2;
        double cr[3];
        cross3(D[a], D[b], cr);
        const double nn = cr[0] * cr[0] + cr[1] * cr[1] + cr[2] * cr[2];
        if (nn > bn) { bn = nn; v[0] = cr[0]; v[1] = cr[1]; v[2] = cr[2]; }
    }
    const double s = 1.0 / sqrt(bn);
    v[0] *= s; v[1] *= s; v[2] *= s;
}

TVF_HD double fp_quad(const double (*G)[3], const double* a, const double* b) {
    double s = 0.0;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) s += a[i] * G[i][j] * b[j];
    return s;
}

TVF_HD int p3p_lambda_twist(const double (*X)[3], const double (*y)[3], double (*R)[9], double (*t)[3]) {
    double d[3][3];
    for (int i = 0; i < 3; ++i) { d[0][i] = X[0][i] - X[1][i]; d[1][i] = X[0][i] - X[2][i]; d[2][i] = X[1][i] - X[2][i]; }
    const double a12 = d[0][0] * d[0][0] + d[0][1] * d[0][1] + d[0][2] * d[0][2];
    const double a13 = d[1][0] * d[1][0] + d[1][1] * d[1][1] + d[1][2] * d[1][2];
    const double a23 = d[2][0] * d[2][0] + d[2][1] * d[2][1] + d[2][2] * d[2][2];
    const double c12 = y[0][0] * y[1][0] + y[0][1] * y[1][1] + y[0][2] * y[1][2];
    const double c13 = y[0][0] * y[2][0] + y[0][1] * y[2][1] + y[0][2] * y[2][2];
    const double c23 = y[1][0] * y[2][0] + y[1][1] * y[2][1] + y[1][2] * y[2][2];
    const double M12[3][3] = {{1.0, -c12, 0.0}, {-c12, 1.0, 0.0}, {0.0, 0.0, 0.0}};
    const double M13[3][3] = {{1.0, 0.0, -c13}, {0.0, 0.0, 0.0}, {-c13, 0.0, 1.0}};
    const double M23[3][3] = {{0.0, 0.0, 0.0}, {0.0, 1.0, -c23}, {0.0, -c23, 1.0}};
    double P[3][3], Q[3][3], G[3][3];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            P[i][j] = a23 * M12[i][j] - a12 * M23[i][j];
            Q[i][j] = a13 * M23[i][j] - a23 * M13[i][j];
            G[i][j] = a13 * M12[i][j] - a12 * M13[i][j];
        }
    // det(P + g Q) = sum over the columns taken from Q
    double cub[4] = {0.0, 0.0, 0.0, 0.0};
    for (int mask = 0; mask < 8; ++mask) {
        double Mm[9];
        for (int c = 0; c < 3; ++c)
            for (int r = 0; r < 3; ++r) Mm[r + 3 * c] = ((mask >> c) & 1) ? Q[r][c] : P[r][c];
        cub[((mask & 1) + ((mask >> 1) & 1) + ((mask >> 2) & 1))] += det3(Mm);
    }
    double gs[3];
    const int ng = fp_real_roots(cub, 3, gs);
    double D[3][3], c2best = 0.0;
    bool have = false;
    for (int k = 0; k < ng; ++k) {
        double Dk[3][3];
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) Dk[i][j] = P[i][j] + gs[k] * Q[i][j];
        const double c2 = Dk[0][0] * Dk[1][1] - Dk[0][1] * Dk[1][0] + Dk[0][0] * Dk[2][2] - Dk[0][2] * Dk[2][0] +
                          Dk[1][1] * Dk[2][2] - Dk[1][2] * Dk[2][1];
        if (c2 < c2best) {
            c2best = c2; have = true;
            for (int i = 0; i < 3; ++i)
                for (int j = 0; j < 3; ++j) D[i][j] = Dk[i][j];
        }
    }
    if (!have) return 0;
    const double trD = D[0][0] + D[1][1] + D[2][2];
    const double disc = sqrt(trD * trD - 4.0 * c2best);
    const double sp = trD >= 0.0 ? 0.5 * (trD + disc) : c2best / (0.5 * (trD - disc));     // > 0
    const double sm = c2best / sp;                                                          // < 0
    double ep[3], em[3];
    {
        double T[3][3];
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) T[i][j] = D[i][j] - (i == j ? sp : 0.0);
        fp_sym_null(T, ep);
        for (int i = 0; i < 3; ++i) T[i][i] = D[i][i] - sm;
        fp_sym_null(T, em);
    }
    const double s = sqrt(-sm / sp);
    int count = 0;
    for (int plane = 0; plane < 2; ++plane) {
        double n[3];
        for (int i = 0; i < 3; ++i) n[i] = ep[i] + (plane == 0 ? -s : s) * em[i];
        const double nn = 1.0 / sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
        n[0] *= nn; n[1] *= nn; n[2] *= nn;
        double u[3], w[3];
        onb3(n, u, w);
        const double qa = fp_quad(G, u, u), qb = 2.0 * fp_quad(G, u, w), qc = fp_quad(G, w, w);
        const double qd = qb * qb - 4.0 * qa * qc;
        if (!(qd >= 0.0)) continue;
        const double qq = -0.5 * (qb + copysign(sqrt(qd), qb));
        for (int r = 0; r < 2; ++r) {
            double lam[3];
            if (fabs(qa) >= fabs(qc)) {                        // alpha / beta: roots of qa t^2 + qb t + qc
                const double tt = r == 0 ? qq / qa : qc / qq;
                for (int i = 0; i < 3; ++i) lam[i] = tt * u[i] + w[i];
            } else {                                           // beta / alpha: roots of qc t^2 + qb t + qa
                const double tt = r == 0 ? qq / qc : qa / qq;
                for (int i = 0; i < 3; ++i) lam[i] = u[i] + tt * w[i];
            }
            const double f12 = fp_quad(M12, lam, lam);
            if (!(f12 > 0.0)) continue;
            const double sc = copysign(sqrt(a12 / f12), lam[0] + lam[1] + lam[2]);
            for (int i = 0; i < 3; ++i) lam[i] *= sc;
            if (!(lam[0] > 0.0 && lam[1] > 0.0 && lam[2] > 0.0)) continue;
            // R = [Y01 Y02 Y01xY02] inv([X01 X02 X01xX02]), t = lambda_0 y_0 - R X_0
            double Yc[3][3], Xm[9], Ym[9], Xi[9];
            for (int i = 0; i < 3; ++i)
                for (int e = 0; e < 3; ++e) Yc[i][e] = lam[i] * y[i][e];
            double yd1[3], yd2[3], yx[3], xx[3];
            for (int e = 0; e < 3; ++e) { yd1[e] = Yc[0][e] - Yc[1][e]; yd2[e] = Yc[0][e] - Yc[2][e]; }
            cross3(yd1, yd2, yx);
            cross3(d[0], d[1], xx);
            for (int e = 0; e < 3; ++e) {
                Ym[e] = yd1[e]; Ym[3 + e] = yd2[e]; Ym[6 + e] = yx[e];
                Xm[e] = d[0][e]; Xm[3 + e] = d[1][e]; Xm[6 + e] = xx[e];
            }
            inv3(Xm, Xi);
            mat3_mul(Ym, Xi, R[count]);
            double RX[3];
            mat3_vec(R[count], X[0], RX);
            for (int e = 0; e < 3; ++e) t[count][e] = Yc[0][e] - RX[e];
            ++count;
        }
    }
    return count;
}

// ---------------------------------------------------------------- the minimal three-view pose
// One problem: the 5 columns p (6 x 5, x1 y1 x2 y2 x3 y3 each) and CalM (9 x 3).  Rt2, Rt3 (3 x 4); E (9 x 10, NaN
// padded) and *nE as five_point_essentials.  Returns the status: 0, ST_NO_POSE_2, ST_NO_POSE_3 or ST_NONFINITE (the
// pose NaN in each of those).
TVF_HD int five_point_pose(const double* p, const double* calm, double* Rt2, double* Rt3, double* Eout, int* nE) {
    double K[3][9], Ki[3][9];
    for (int v = 0; v < 3; ++v) {
        for (int c = 0; c < 3; ++c)
            for (int r = 0; r < 3; ++r) K[v][r + 3 * c] = calm[3 * v + r + 9 * c];
        inv3(K[v], Ki[v]);
    }
    double q[3][5][3];                                       // rays K^-1 [x y 1]' of every view
    for (int v = 0; v < 3; ++v)
        for (int j = 0; j < 5; ++j) {
            const double h[3] = {p[6 * j + 2 * v], p[6 * j + 2 * v + 1], 1.0};
            mat3_vec(Ki[v], h, q[v][j]);
        }
    for (int e = 0; e < 12; ++e) { Rt2[e] = (double)NAN; Rt3[e] = (double)NAN; }
    if (!five_point_essentials(q[0], q[1], Eout, nE)) return ST_NO_POSE_2;
    double P1[12];
    load_K1_as_P1(calm, P1);
    bool any2 = false, found = false;
    double best_err = 0.0;
    for (int k = 0; k < *nE; ++k) {
        // view 2: the first of (R, t), (R, -t), (Rp, -t), (Rp, t) with all five points in front of views 1 and 2
        double R[9], Rp[9], t[3];
        decompose_essential(Eout + 9 * k, R, Rp, t);
        double R2[9], t2[3], Xs[5][3];
        bool ok2 = false;
        for (int cnd = 0; cnd < 4 && !ok2; ++cnd) {
            const double* Rc = cnd < 2 ? R : Rp;
            const double sg = (cnd == 0 || cnd == 3) ? 1.0 : -1.0;
            double P2[12];
            for (int c = 0; c < 3; ++c)
                for (int r = 0; r < 3; ++r)
                    P2[r + 3 * c] = K[1][r] * Rc[3 * c] + K[1][r + 3] * Rc[1 + 3 * c] + K[1][r + 6] * Rc[2 + 3 * c];
            for (int r = 0; r < 3; ++r) P2[9 + r] = sg * (K[1][r] * t[0] + K[1][r + 3] * t[1] + K[1][r + 6] * t[2]);
            bool front = true;
            for (int j = 0; j < 5 && front; ++j) {
                double Xh[4];
                triangulate2(P1, P2, p[6 * j], p[6 * j + 1], p[6 * j + 2], p[6 * j + 3], Xh);
                const double z2 = Rc[2] * Xh[0] + Rc[5] * Xh[1] + Rc[8] * Xh[2] + sg * t[2] * Xh[3];
                // |Xh| = 1: a point at infinity (|X4| <= 1e-12, no parallax) is in front of neither view
                front = (Xh[2] * Xh[3] > 0.0) && (z2 * Xh[3] > 0.0) && fabs(Xh[3]) > 1e-12;
                for (int e = 0; e < 3; ++e) Xs[j][e] = Xh[e] / Xh[3];
            }
            if (front) {
                ok2 = true;
                for (int e = 0; e < 9; ++e) R2[e] = Rc[e];
                for (int e = 0; e < 3; ++e) t2[e] = sg * t[e];
            }
        }
        if (!ok2) continue;
        any2 = true;
        // view 3: P3P on columns 0, 1, 2; every point in front of view 3; error of columns 3, 4
        double y3[3][3];
        for (int j = 0; j < 3; ++j) {
            const double s = 1.0 / sqrt(q[2][j][0] * q[2][j][0] + q[2][j][1] * q[2][j][1] + q[2][j][2] * q[2][j][2]);
            for (int e = 0; e < 3; ++e) y3[j][e] = q[2][j][e] * s;
        }
        double R3s[4][9], t3s[4][3];
        const int n3 = p3p_lambda_twist(Xs, y3, R3s, t3s);
        for (int r = 0; r < n3; ++r) {
            bool front = true;
            double err = 0.0;
            for (int j = 0; j < 5; ++j) {
                double xc[3];
                mat3_vec(R3s[r], Xs[j], xc);
                for (int e = 0; e < 3; ++e) xc[e] += t3s[r][e];
                front = front && xc[2] > 0.0;
                if (j >= 3) {
                    double xp[3];
                    mat3_vec(K[2], xc, xp);
                    const double dx = xp[0] / xp[2] - p[6 * j + 4], dy = xp[1] / xp[2] - p[6 * j + 5];
                    err = fmax(err, sqrt(dx * dx + dy * dy));
                }
            }
            if (!front) continue;
            if (!found || err < best_err) {
                found = true; best_err = err;
                for (int e = 0; e < 9; ++e) { Rt2[e] = R2[e]; Rt3[e] = R3s[r][e]; }
                for (int e = 0; e < 3; ++e) { Rt2[9 + e] = t2[e]; Rt3[9 + e] = t3s[r][e]; }
            }
        }
    }
    if (!any2) return ST_NO_POSE_2;
    if (!found) return ST_NO_POSE_3;
    bool fin = true;
    for (int e = 0; e < 12; ++e) fin = fin && isfinite(Rt2[e]) && isfinite(Rt3[e]);
    if (!fin) {
        for (int e = 0; e < 12; ++e) { Rt2[e] = (double)NAN; Rt3[e] = (double)NAN; }
        return ST_NONFINITE;
    }
    return 0;
}

}  // namespace tvf
