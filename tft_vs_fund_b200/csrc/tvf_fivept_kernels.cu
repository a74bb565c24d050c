// tvf_fivept_kernels.cu -- the calibrated five-point minimal pose (tvf_five_point_pose, RANSAC method 9's hypotheses):
// one thread per minimal problem, the whole of tvf_fivept.cuh in registers and local memory.
#include "tvf_kernels.h"
#include "tvf_fivept.cuh"

namespace tvf {

namespace {

// problem q: columns in + 30 q (6 x 5), calm + 27 q (calm_batched) or calm; every output may be null
__global__ void __launch_bounds__(128) five_point_pose_kernel(const double* __restrict__ in, const double* __restrict__ calm,
                                                              int calm_batched, long long B, double* Rt2, double* Rt3,
                                                              double* E, int* nE, int* status) {
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < B; q += (long long)gridDim.x * blockDim.x) {
        double p[30], K[27], r2[12], r3[12], e[9 * FP_MAX_E];
        for (int i = 0; i < 30; ++i) p[i] = in[q * 30 + i];
        for (int i = 0; i < 27; ++i) K[i] = calm[(calm_batched ? q * 27 : 0) + i];
        int n = 0;
        const int st = five_point_pose(p, K, r2, r3, e, &n);
        if (Rt2) for (int i = 0; i < 12; ++i) Rt2[q * 12 + i] = r2[i];
        if (Rt3) for (int i = 0; i < 12; ++i) Rt3[q * 12 + i] = r3[i];
        if (E) for (int i = 0; i < 9 * FP_MAX_E; ++i) E[q * 9 * FP_MAX_E + i] = e[i];
        if (nE) nE[q] = n;
        if (status) status[q] = st;
    }
}

}  // namespace

void launch_five_point_pose(const double* in, const double* calm, int calm_batched, long long B, double* Rt2, double* Rt3,
                            double* E, int* nE, int* status, cudaStream_t stream) {
    if (B <= 0) return;
    long long g = (B + 127) / 128;
    if (g > (1LL << 20)) g = 1LL << 20;
    five_point_pose_kernel<<<(unsigned)g, 128, 0, stream>>>(in, calm, calm_batched, B, Rt2, Rt3, E, nE, status);
}

}  // namespace tvf
