// Host build of csrc/tvf_ba.cuh's robust-loss functions for tests/test_ba_robust_cpu.py (TEST-ONLY; the same source the
// kernel inlines).  Matrices column-major as in the library.
#include "tvf_ba.cuh"

using namespace tvf;

extern "C" {

double hc_ba_loss_cost(int loss, double s, double c2) { return ba_loss_cost(loss, s, c2); }
double hc_ba_loss_weight(int loss, double s, double c2) { return ba_loss_weight(loss, s, c2); }

void hc_ba_basis(const double* calm, const double* Rt2, const double* Rt3, double* u1, double* u2) {
    BaCams c; ba_load_cams(calm, Rt2, Rt3, c);
    for (int k = 0; k < 3; ++k) { u1[k] = c.u1[k]; u2[k] = c.u2[k]; }
}

// sum over the n points (X 3 x n, corresp 6 x n) of c^2 rho(s_i / c^2), as the kernel sums a problem's cost
double hc_ba_robust_cost(const double* calm, const double* Rt2, const double* Rt3, const double* X, const double* corresp,
                         int n, int loss, double c2) {
    BaCams c; ba_load_cams(calm, Rt2, Rt3, c);
    double f = 0.0;
    for (int i = 0; i < n; ++i) f += ba_loss_cost(loss, ba_point_cost(c, X + 3 * i, corresp + 6 * i), c2);
    return f;
}

// the kernel's weighted linearisation at damping mu: every point weighed (w n), eliminated and accumulated into the
// BA_NSUM sums; then the camera step and the point steps (dX 3 x n).  Returns 1 if every block was positive definite.
int hc_ba_robust_system(const double* calm, const double* Rt2, const double* Rt3, const double* X, const double* corresp,
                        int n, int loss, double c2, double mu, double* w, double* sums, double* gp, double* dc, double* dX) {
    BaCams c; ba_load_cams(calm, Rt2, Rt3, c);
    for (int e = 0; e < BA_NSUM; ++e) sums[e] = 0.0;
    bool ok = true;
    for (int i = 0; i < n; ++i) {
        BaPoint p; BaElim el;
        ba_point_jac(c, X + 3 * i, corresp + 6 * i, p);
        w[i] = ba_point_weigh(p, loss, c2);
        ok = ba_point_eliminate(p, mu, el) && ok;
        ba_point_accumulate(p, el, sums);
        for (int k = 0; k < 3; ++k) gp[3 * i + k] = el.g[k];
    }
    double work[BA_NSUM];
    for (int e = 0; e < BA_NSUM; ++e) work[e] = sums[e];
    if (!ok || !ba_solve_reduced(work, mu, dc)) return 0;
    for (int i = 0; i < n; ++i) {
        BaPoint p; BaElim el;
        ba_point_jac(c, X + 3 * i, corresp + 6 * i, p);
        ba_point_weigh(p, loss, c2);
        ba_point_eliminate(p, mu, el);
        ba_point_step(el, dc, dX + 3 * i);
    }
    return 1;
}

void hc_ba_update(const double* calm, double* Rt2, double* Rt3, const double* dc) {
    BaCams c; ba_load_cams(calm, Rt2, Rt3, c);
    ba_update_cams(dc, c);
    for (int q = 0; q < 9; ++q) { Rt2[q] = c.R2[q]; Rt3[q] = c.R3[q]; }
    for (int q = 0; q < 3; ++q) { Rt2[9 + q] = c.t2[q]; Rt3[9 + q] = c.t3[q]; }
}

}  // extern "C"
