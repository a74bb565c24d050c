// tvf_ransac.cuh -- per-thread pieces of the RANSAC pose estimator (tvf_ransac_pose): the counter-based sampler and
// the three-view inlier test.  Host/device functions, so the kernels in tvf_ransac_kernels.cu and the CPU check in
// tests/hostcheck/ransac_hostcheck.cpp share one source.
#pragma once
#include <stdint.h>

#include "tvf_pose.cuh"

namespace tvf {

constexpr int ST_RANSAC_FAILED = 128;    // every hypothesis of the problem was flagged: no pose

// splitmix64's output function
TVF_HD uint64_t ransac_mix64(uint64_t z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// draw j (< 256) of hypothesis h (< 2^24) of the problem with key `seed`
TVF_HD uint64_t ransac_draw(uint64_t seed, uint32_t h, int j) {
    return ransac_mix64(seed ^ ransac_mix64(((uint64_t)h << 8) | (uint64_t)j));
}

// uniform integer in [0, m) from the high 32 bits of r
TVF_HD int ransac_uniform(uint64_t r, uint32_t m) { return (int)(((r >> 32) * (uint64_t)m) >> 32); }

// The s distinct indices in [0, n) of hypothesis h, in draw order (Floyd's algorithm): for j = 0..s-1, with
// m = n - s + j + 1 and u = uniform(m), take u, or m - 1 if u was already taken.
TVF_HD void ransac_sample(uint64_t seed, uint32_t h, int n, int s, int* idx) {
    for (int j = 0; j < s; ++j) {
        const uint32_t m = (uint32_t)(n - s + j + 1);
        int u = ransac_uniform(ransac_draw(seed, h, j), m);
        bool taken = false;
        for (int k = 0; k < j; ++k) taken = taken || (idx[k] == u);
        idx[j] = taken ? (int)m - 1 : u;
    }
}

// the three cameras K1[I|0], K2[R2|t2], K3[R3|t3] (3 x 4 column-major each) of CalM (9 x 3) and a pose
TVF_HD void ransac_cameras(const double* calm, const double* Rt2, const double* Rt3, double* P1, double* P2, double* P3) {
    load_K1_as_P1(calm, P1);
#pragma unroll
    for (int v = 0; v < 2; ++v) {
        const double* Rt = v == 0 ? Rt2 : Rt3;
        double* P = v == 0 ? P2 : P3;
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int r = 0; r < 3; ++r)
                P[r + 3 * c] = calm[3 * (v + 1) + r] * Rt[3 * c] + calm[3 * (v + 1) + r + 9] * Rt[1 + 3 * c] +
                               calm[3 * (v + 1) + r + 18] * Rt[2 + 3 * c];
    }
}

// The inlier test of one point p6 = (x1 y1 x2 y2 x3 y3): triangulate it with the three cameras (triangulation3D.m),
// dehomogenise X(1:3)/X(4), re-project (project3Dpoints.m) and compare with the observation, as experiments_real.m:94-98
// does.  Inlier iff all six residuals are finite and <= th in absolute value; a NaN residual makes the point an outlier
// (the reference counts it as an inlier, since NaN > th is false).  maxres (may be null): the largest |residual|, NaN
// if one is NaN.
TVF_HD bool ransac_inlier(const double* P1, const double* P2, const double* P3, const double* p6, double th,
                          double* maxres = nullptr) {
    double X[4];
    triangulate3(P1, P2, P3, p6, X);
    const double Xe[4] = {X[0] / X[3], X[1] / X[3], X[2] / X[3], 1.0};
    bool ok = true, nan = false;
    double mx = 0.0;
#pragma unroll
    for (int v = 0; v < 3; ++v) {
        double x[3];
        cam_apply(v == 0 ? P1 : (v == 1 ? P2 : P3), Xe, x);
        const double rx = fabs(x[0] / x[2] - p6[2 * v]), ry = fabs(x[1] / x[2] - p6[2 * v + 1]);
        ok = ok && (rx <= th) && (ry <= th);                 // false for NaN, and for +inf (th is finite)
        nan = nan || (rx != rx) || (ry != ry);
        mx = fmax(mx, fmax(rx, ry));
    }
    if (maxres) *maxres = nan ? (double)NAN : mx;
    return ok;
}

}  // namespace tvf
