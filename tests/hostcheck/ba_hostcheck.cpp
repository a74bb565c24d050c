// Host build of csrc/tvf_ba.cuh for tests/test_bundle_adjust_cpu.py (TEST-ONLY; the same source the kernel inlines).
// Matrices column-major as in the library; Jacobians are returned row-major (6 x 3 and 6 x 11).
#include "tvf_ba.cuh"

using namespace tvf;

extern "C" {

void hc_ba_basis(const double* calm, const double* Rt2, const double* Rt3, double* u1, double* u2) {
    BaCams c; ba_load_cams(calm, Rt2, Rt3, c);
    for (int k = 0; k < 3; ++k) { u1[k] = c.u1[k]; u2[k] = c.u2[k]; }
}

void hc_ba_jac(const double* calm, const double* Rt2, const double* Rt3, const double* X, const double* x6, double* r,
               double* Jp, double* Jc) {
    BaCams c; ba_load_cams(calm, Rt2, Rt3, c);
    BaPoint p; ba_point_jac(c, X, x6, p);
    for (int k = 0; k < 6; ++k) {
        r[k] = p.r[k];
        for (int j = 0; j < 3; ++j) Jp[3 * k + j] = p.Jp[k][j];
        for (int j = 0; j < BA_NC; ++j) Jc[BA_NC * k + j] = ba_jc(p, k, j);
    }
}

double hc_ba_cost(const double* calm, const double* Rt2, const double* Rt3, const double* X, const double* x6) {
    BaCams c; ba_load_cams(calm, Rt2, Rt3, c);
    return ba_point_cost(c, X, x6);
}

// the BA_NSUM sums of all n points (X 3 x n, corresp 6 x n) at damping mu; then the camera step and the point steps
// (dX 3 x n) of the damped system.  Returns 1 if every point block and the reduced system were positive definite.
int hc_ba_system(const double* calm, const double* Rt2, const double* Rt3, const double* X, const double* corresp, int n,
                 double mu, double* sums, double* dc, double* dX) {
    BaCams c; ba_load_cams(calm, Rt2, Rt3, c);
    for (int e = 0; e < BA_NSUM; ++e) sums[e] = 0.0;
    bool ok = true;
    for (int i = 0; i < n; ++i) {
        BaPoint p; BaElim el;
        ba_point_jac(c, X + 3 * i, corresp + 6 * i, p);
        ok = ba_point_eliminate(p, mu, el) && ok;
        ba_point_accumulate(p, el, sums);
    }
    double work[BA_NSUM];
    for (int e = 0; e < BA_NSUM; ++e) work[e] = sums[e];
    if (!ok || !ba_solve_reduced(work, mu, dc)) return 0;
    for (int i = 0; i < n; ++i) {
        BaPoint p; BaElim el;
        ba_point_jac(c, X + 3 * i, corresp + 6 * i, p);
        ba_point_eliminate(p, mu, el);
        ba_point_step(el, dc, dX + 3 * i);
    }
    return 1;
}

void hc_ba_rotate(const double* w, double* R) { ba_rotate(w, R); }

void hc_ba_update(const double* calm, double* Rt2, double* Rt3, const double* dc) {
    BaCams c; ba_load_cams(calm, Rt2, Rt3, c);
    ba_update_cams(dc, c);
    for (int q = 0; q < 9; ++q) { Rt2[q] = c.R2[q]; Rt3[q] = c.R3[q]; }
    for (int q = 0; q < 3; ++q) { Rt2[9 + q] = c.t2[q]; Rt3[9 + q] = c.t3[q]; }
}

}  // extern "C"
