// Host build of the covariance functions of csrc/tvf_ba.cuh for tests/test_ba_covariance_cpu.py (TEST-ONLY; the
// same source ba_covariance_kernel inlines), composed in the kernel's order for one problem.  Matrices column-major.
#include "tvf_ba.cuh"

using namespace tvf;

extern "C" {

// state Rt2, Rt3 (3 x 4, |t2| = 1 already), X 3 x n, corresp 6 x n -> cov_cam 12 x 12, cov_pts 9 x n, sigma2, and the
// 11 x 11 chart covariance C (null allowed) with the tangent basis u1, u2.  Returns the status word (0, or
// ST_COV_SINGULAR).
int hc_ba_cov(const double* calm, const double* Rt2, const double* Rt3, const double* X, const double* corresp, int n,
              double* cov_cam, double* cov_pts, double* sigma2, double* C11, double* u1, double* u2) {
    BaCams c; ba_load_cams(calm, Rt2, Rt3, c);
    double sums[BA_NSUM] = {0.0};
    double cost = 0.0;
    bool ok = true;
    for (int i = 0; i < n; ++i) {
        BaPoint p; BaElim el;
        ba_point_jac(c, X + 3 * i, corresp + 6 * i, p);
        ok = ba_point_eliminate(p, 0.0, el) && ba_cov_point_ok(el) && ok;
        ba_point_accumulate(p, el, sums);
        for (int k = 0; k < 6; ++k) cost += p.r[k] * p.r[k];
    }
    for (int k = 0; k < 3; ++k) { u1[k] = c.u1[k]; u2[k] = c.u2[k]; }
    if (!ok || !ba_cov_factor(sums)) return ST_COV_SINGULAR;
    double Xc[BA_NC * BA_NC], C[BA_NC * BA_NC];
    for (int j = 0; j < BA_NC; ++j) ba_cov_column(sums, j, Xc + BA_NC * j);
    for (int j = 0; j < BA_NC; ++j)
        for (int i = 0; i < BA_NC; ++i) C[i + BA_NC * j] = 0.5 * (Xc[i + BA_NC * j] + Xc[j + BA_NC * i]);
    if (C11) for (int e = 0; e < BA_NC * BA_NC; ++e) C11[e] = C[e];
    for (int i = 0; i < 12; ++i)
        for (int j = i; j < 12; ++j) {
            const double v = ba_cov_expand(C, c.u1, c.u2, i, j);
            cov_cam[i + 12 * j] = v; cov_cam[j + 12 * i] = v;
        }
    for (int i = 0; i < n; ++i) {
        BaPoint p; BaElim el;
        ba_point_jac(c, X + 3 * i, corresp + 6 * i, p);
        ba_point_eliminate(p, 0.0, el);
        ba_cov_point(el, C, cov_pts + 9 * i);
    }
    *sigma2 = cost / (3.0 * n - 11.0);
    return 0;
}

}  // extern "C"
