// tvf_ba_cov_kernels.cu -- first-order covariance of the three-view bundle adjustment at a given state
// (tvf_ba_covariance).  One warp per problem, lanes own points (point i belongs to lane i mod 32), the mapping of
// bundle_adjust_kernel.  Per-point algebra: tvf_ba.cuh (the adjustment's Jacobian and elimination at mu = 0).
//
//   pass 1   every lane linearises its points at the gauge-normalised state, eliminates each point block V_i (relative
//            pivot floor BA_COV_PIVOT) and adds its sums (tvf_ba.cuh::ba_point_accumulate) to a lane-private row of
//            shared memory, in point order; the rows are then added lane 0..31 in that order (entry e by lane e mod 32),
//            as in bundle_adjust_kernel -- the reduced matrix S is the adjustment's at mu = 0, bit for bit;
//   factor   lane 0 factors S = U'U;
//   invert   lane j < 11 solves column j of S^-1; the chart covariance C is symmetrised as (x_ij + x_ji) / 2 and
//            expanded to the 12 x 12 cov_cam, upper triangle formed and mirrored;
//   pass 2   every lane re-forms its points' elimination (same inputs, same bits) and writes their 3 x 3 marginals.
// Every sum has a fixed order and every decision is warp-uniform, so a problem's result depends on its data alone.
#include "tvf_kernels.h"
#include "tvf_warp.cuh"
#include "tvf_pose.cuh"
#include "tvf_ba.cuh"

namespace tvf {

constexpr int BC_WARPS = 2;
constexpr int BC_SLAB = 32 * BA_NSUM;                  // lane-private partial sums (odd stride: conflict-free)
constexpr int BC_CAMS = (sizeof(BaCams) + 7) / 8;      // doubles per BaCams
constexpr int BC_PER_WARP = BC_SLAB + BA_NSUM + 1 + BA_NC * BA_NC + BC_CAMS;

__device__ __forceinline__ bool cov_finite(double x) { return fabs(x) <= 1.79769313486231570e308; }

__device__ __forceinline__ void cov_load_x6(const double* corresp, long long prob, int n, int i, double* x6) {
    const double2* q = reinterpret_cast<const double2*>(corresp + (prob * n + i) * 6);
    const double2 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
    x6[0] = a.x; x6[1] = a.y; x6[2] = b.x; x6[3] = b.y; x6[4] = c.x; x6[5] = c.y;
}

__global__ void __launch_bounds__(BC_WARPS * 32)
ba_covariance_kernel(const BaCovArgs a) {
    extern __shared__ __align__(16) double bc_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* slab = bc_smem + (size_t)warp * BC_PER_WARP;
    double* red = slab + BC_SLAB;                      // BA_NSUM sums, then the factor flag
    double* Cs = red + BA_NSUM + 1;                    // 11 x 11 chart covariance, column-major
    BaCams& cam = *reinterpret_cast<BaCams*>(Cs + BA_NC * BA_NC);
    double* acc = slab + lane * BA_NSUM;
    const int n = a.n;
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);

    for (long long prob = (long long)blockIdx.x * BC_WARPS + warp; prob < a.B; prob += (long long)gridDim.x * BC_WARPS) {
        const double* cm = a.calm + (a.calm_batched ? prob * 27 : 0);
        const double* rt2 = a.Rt2 + prob * 12;
        const double* rt3 = a.Rt3 + prob * 12;
        const double* Xp = a.X + prob * 3 * n;
        __syncwarp();
        if (lane == 0) ba_load_cams(cm, rt2, rt3, cam);
        bool bad_l = (lane < 27 && !cov_finite(cm[lane])) || (lane < 12 && !(cov_finite(rt2[lane]) && cov_finite(rt3[lane])));
        __syncwarp();
        const double t2n = sqrt(cam.t2[0] * cam.t2[0] + cam.t2[1] * cam.t2[1] + cam.t2[2] * cam.t2[2]);
        const double gs = 1.0 / t2n;
        __syncwarp();
        if (lane == 0) {                               // gauge |t2| = 1, exactly as bundle_adjust_kernel
#pragma unroll
            for (int k = 0; k < 3; ++k) { cam.t2[k] *= gs; cam.t3[k] *= gs; }
            onb3(cam.t2, cam.u1, cam.u2);
        }
        __syncwarp();

        // ---- pass 1: linearise + eliminate + accumulate at mu = 0 --------------------------------------------------
#pragma unroll 1
        for (int e = 0; e < BA_NSUM; ++e) acc[e] = 0.0;
        double cost_l = 0.0;
        bool pd_l = true;
        for (int i = lane; i < n; i += 32) {
            double x6[6], X[3];
            cov_load_x6(a.corresp, prob, n, i, x6);
#pragma unroll
            for (int k = 0; k < 3; ++k) X[k] = Xp[3 * i + k] * gs;
#pragma unroll
            for (int k = 0; k < 6; ++k) bad_l = bad_l || !cov_finite(x6[k]);
            bad_l = bad_l || !(cov_finite(X[0]) && cov_finite(X[1]) && cov_finite(X[2]));
            BaPoint p; BaElim el;
            ba_point_jac(cam, X, x6, p);
            pd_l = ba_point_eliminate(p, 0.0, el) && ba_cov_point_ok(el) && pd_l;
            ba_point_accumulate(p, el, acc);
#pragma unroll
            for (int k = 0; k < 6; ++k) cost_l += p.r[k] * p.r[k];
        }
        const double cost = warp_sum(cost_l);
        const bool bad = __any_sync(FULL, bad_l) || !(t2n > 0.0) || !cov_finite(gs) || !cov_finite(cost);
        int st = bad ? ST_NONFINITE : (__any_sync(FULL, !pd_l) ? ST_COV_SINGULAR : 0);
        if (st == 0) {
            __syncwarp();
            for (int e = lane; e < 66; e += 32) {
                double s = 0.0;
#pragma unroll 8
                for (int l = 0; l < 32; ++l) s += slab[l * BA_NSUM + e];
                red[e] = s;
            }
            __syncwarp();
            if (lane == 0) red[BA_NSUM] = ba_cov_factor(red) ? 1.0 : 0.0;
            __syncwarp();
            if (red[BA_NSUM] == 0.0) st = ST_COV_SINGULAR;
        }
        double* cc = a.cov_cam ? a.cov_cam + prob * 144 : nullptr;
        double* cp = a.cov_pts ? a.cov_pts + prob * 9 * n : nullptr;
        if (st != 0) {                                 // every output of the problem is NaN
            if (cc) for (int e = lane; e < 144; e += 32) cc[e] = qnan;
            if (cp) for (int e = lane; e < 9 * n; e += 32) cp[e] = qnan;
            if (lane == 0) {
                if (a.sigma2) a.sigma2[prob] = qnan;
                if (a.status) a.status[prob] = st;
            }
            continue;
        }

        // ---- invert: column j of S^-1 by lane j, then C = (X + X') / 2 ---------------------------------------------
        double x[BA_NC];
        if (lane < BA_NC) {
            ba_cov_column(red, lane, x);
#pragma unroll
            for (int k = 0; k < BA_NC; ++k) slab[k + BA_NC * lane] = x[k];   // pass 1's slab is free again
        }
        __syncwarp();
        for (int e = lane; e < BA_NC * BA_NC; e += 32) {
            const int i = e % BA_NC, j = e / BA_NC;
            Cs[e] = 0.5 * (slab[i + BA_NC * j] + slab[j + BA_NC * i]);
        }
        __syncwarp();
        if (cc) {
            for (int e = lane; e < 78; e += 32) {      // upper triangle of the 12 x 12, row-major, then mirrored
                int i = 0, rem = e;
                while (rem >= 12 - i) { rem -= 12 - i; ++i; }
                const int j = i + rem;
                const double v = ba_cov_expand(Cs, cam.u1, cam.u2, i, j);
                cc[i + 12 * j] = v; cc[j + 12 * i] = v;
            }
        }

        // ---- pass 2: point marginals ---------------------------------------------------------------------------
        if (cp) {
            for (int i = lane; i < n; i += 32) {
                double x6[6], X[3], cov[9];
                cov_load_x6(a.corresp, prob, n, i, x6);
#pragma unroll
                for (int k = 0; k < 3; ++k) X[k] = Xp[3 * i + k] * gs;
                BaPoint p; BaElim el;
                ba_point_jac(cam, X, x6, p);
                ba_point_eliminate(p, 0.0, el);
                ba_cov_point(el, Cs, cov);
#pragma unroll
                for (int k = 0; k < 9; ++k) cp[9 * i + k] = cov[k];
            }
        }
        if (lane == 0) {
            if (a.sigma2) a.sigma2[prob] = cost / (3.0 * n - 11.0);
            if (a.status) a.status[prob] = 0;
        }
    }
}

int launch_ba_covariance(const BaCovArgs& a, cudaStream_t stream) {
    if (a.B <= 0) return 1;
    const size_t smem = (size_t)BC_WARPS * BC_PER_WARP * sizeof(double);
    // the opt-in is a per-device property of the function: set on every launch, as for bundle_adjust_kernel
    if (cudaFuncSetAttribute(ba_covariance_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    long long blocks = (a.B + BC_WARPS - 1) / BC_WARPS;
    if (blocks > 0x7fffffffLL) blocks = 0x7fffffffLL;
    ba_covariance_kernel<<<(unsigned)blocks, BC_WARPS * 32, smem, stream>>>(a);
    return cudaPeekAtLastError() == cudaSuccess ? 1 : 0;
}

}  // namespace tvf
