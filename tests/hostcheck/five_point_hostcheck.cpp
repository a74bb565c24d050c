// Host build of csrc/tvf_fivept.cuh for tests/test_five_point_cpu.py (TEST-ONLY; the same source five_point_pose_kernel
// inlines): the Sturm root finder, the essential matrices, the P3P and the whole minimal pose.
#include "tvf_fivept.cuh"

using namespace tvf;

extern "C" {

// the distinct real roots of p (degree d, p[i] of x^i), ascending -> roots; returns their count
int hc_fp_real_roots(const double* p, int d, double* roots) { return fp_real_roots(p, d, roots); }

// the essential matrices of the rays q1, q2 (5 x 3, one ray per row) -> E (9 x 10), *nE; returns 0 on a zero pivot
int hc_five_point_essentials(const double* q1, const double* q2, double* E, int* nE) {
    return five_point_essentials(reinterpret_cast<const double(*)[3]>(q1), reinterpret_cast<const double(*)[3]>(q2), E,
                                 nE) ? 1 : 0;
}

// P3P of the points X and the unit rays y (3 x 3, one per row) -> R (9 x 4), t (3 x 4); returns the count
int hc_p3p(const double* X, const double* y, double* R, double* t) {
    return p3p_lambda_twist(reinterpret_cast<const double(*)[3]>(X), reinterpret_cast<const double(*)[3]>(y),
                            reinterpret_cast<double(*)[9]>(R), reinterpret_cast<double(*)[3]>(t));
}

// the minimal pose of count problems: p (6 x 5 each), calm (9 x 3 each) -> Rt2, Rt3 (3 x 4), E (9 x 10), nE, status
void hc_five_point_pose(const double* p, const double* calm, int count, double* Rt2, double* Rt3, double* E, int* nE,
                        int* status) {
    for (int b = 0; b < count; ++b)
        status[b] = five_point_pose(p + 30 * b, calm + 27 * b, Rt2 + 12 * b, Rt3 + 12 * b, E + 90 * b, nE + b);
}

}  // extern "C"
