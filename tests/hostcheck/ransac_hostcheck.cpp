// Host build of csrc/tvf_ransac.cuh for tests/test_ransac_cpu.py (TEST-ONLY; the same source the RANSAC kernels
// inline): the sampler and the inlier test.
#include "tvf_ransac.cuh"

using namespace tvf;

extern "C" {

// count draws: indices of hypothesis hs[i] of key seeds[i] with ns[i] matches and ss[i] (<= 8) per sample -> out[8 i ..]
void hc_ransac_samples(const uint64_t* seeds, const uint32_t* hs, const int* ns, const int* ss, int count, int* out) {
    for (int i = 0; i < count; ++i) ransac_sample(seeds[i], hs[i], ns[i], ss[i], out + 8 * i);
}

// mix64 and uniform, for the NumPy twin's pieces
uint64_t hc_ransac_mix64(uint64_t z) { return ransac_mix64(z); }

// the inlier test of the n matches corresp (6 x n) under calm (9 x 3) and Rt2, Rt3 (3 x 4), all column-major:
// flags (n) and the largest |residual| of each match (n, NaN if one is not finite)
void hc_ransac_inliers(const double* calm, const double* Rt2, const double* Rt3, const double* corresp, int n, double th,
                       int* flags, double* maxres) {
    double P1[12], P2[12], P3[12];
    ransac_cameras(calm, Rt2, Rt3, P1, P2, P3);
    for (int i = 0; i < n; ++i) flags[i] = ransac_inlier(P1, P2, P3, corresp + 6 * i, th, maxres + i) ? 1 : 0;
}

}  // extern "C"
