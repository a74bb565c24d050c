// tvf_ba_kernels.cu -- batched three-view bundle adjustment (tvf_bundle_adjust): Levenberg-Marquardt on the pixel
// reprojection error with the points eliminated by the Schur complement.  One warp per problem, lanes own points
// (point i belongs to lane i mod 32), the same mapping as optimf_gh_kernel.  Per-point algebra: tvf_ba.cuh.
//
// One iteration:
//   pass A   every lane linearises its points at the current iterate (6 x 3 point and 6 x 11 camera Jacobian),
//            eliminates each point at the current damping and adds its 99 sums (tvf_ba.cuh::ba_point_accumulate)
//            to a lane-private row of shared memory, in point order; the rows are then added lane 0..31 in that
//            order (entry e by lane e mod 32);
//   solve    lane 0 factors the damped 11 x 11 reduced system (Cholesky) and solves for the camera step;
//   pass B   every lane re-forms its points' elimination (same inputs, same bits), back-substitutes dX and evaluates
//            the candidate's cost; candidate points go to the work space `Xc`.
// A step is accepted only if it lowers the cost; a rejected step raises the damping and repeats pass A at the same
// iterate (the same linearisation).  Every sum has a fixed order and every decision is warp-uniform, so a problem's
// result depends on nothing but its own data -- not on its batch, chunk, shard or position.
#include "tvf_kernels.h"
#include "tvf_warp.cuh"
#include "tvf_pose.cuh"
#include "tvf_ba.cuh"

namespace tvf {

constexpr int BA_WARPS = 2;
constexpr int BA_SLAB = 32 * BA_NSUM;                  // lane-private partial sums (odd stride: conflict-free)
constexpr int BA_CAMS = (sizeof(BaCams) + 7) / 8;      // doubles per BaCams
constexpr int BA_PER_WARP = BA_SLAB + BA_NSUM + 1 + 12 + 2 * BA_CAMS;

__device__ __forceinline__ bool finite_(double x) { return fabs(x) <= 1.79769313486231570e308; }

__device__ __forceinline__ void load_x6(const double* corresp, long long prob, int n, int i, double* x6) {
    const double2* q = reinterpret_cast<const double2*>(corresp + (prob * n + i) * 6);
    const double2 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
    x6[0] = a.x; x6[1] = a.y; x6[2] = b.x; x6[3] = b.y; x6[4] = c.x; x6[5] = c.y;
}

__global__ void __launch_bounds__(BA_WARPS * 32)
bundle_adjust_kernel(const BaArgs a) {
    extern __shared__ __align__(16) double ba_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* slab = ba_smem + (size_t)warp * BA_PER_WARP;
    double* red = slab + BA_SLAB;                      // BA_NSUM (+1)
    double* dcs = red + BA_NSUM + 1;                   // 11 camera step entries + solve flag
    BaCams& cur = *reinterpret_cast<BaCams*>(dcs + 12);
    BaCams& cand = *reinterpret_cast<BaCams*>(dcs + 12 + BA_CAMS);
    double* acc = slab + lane * BA_NSUM;
    const int n = a.n;

    for (long long prob = (long long)blockIdx.x * BA_WARPS + warp; prob < a.B; prob += (long long)gridDim.x * BA_WARPS) {
        const double* cm = a.calm + (a.calm_batched ? prob * 27 : 0);
        const double* rt2 = a.Rt2_0 + prob * 12;
        const double* rt3 = a.Rt3_0 + prob * 12;
        double* Xp = a.X + prob * 3 * n;
        double* Xcp = a.Xc + prob * 3 * n;
        __syncwarp();
        if (lane == 0) ba_load_cams(cm, rt2, rt3, cur);
        bool bad_l = (lane < 27 && !finite_(cm[lane])) || (lane < 12 && !(finite_(rt2[lane]) && finite_(rt3[lane])));
        __syncwarp();

        // ---- start points: Reconst0, or triangulation3D({K1[I|0], K2 R_t_2, K3 R_t_3}, Corresp) -----------------
        double cost_l = 0.0;
        {
            double P1[12], P2[12], P3[12];
            if (a.X0 == nullptr) {
                load_K1_as_P1(cm, P1);
#pragma unroll
                for (int col = 0; col < 4; ++col)
#pragma unroll
                    for (int r = 0; r < 3; ++r) {
                        double s2 = 0.0, s3 = 0.0;
#pragma unroll
                        for (int k = 0; k < 3; ++k) { s2 += cur.K2[r + 3 * k] * rt2[k + 3 * col]; s3 += cur.K3[r + 3 * k] * rt3[k + 3 * col]; }
                        P2[r + 3 * col] = s2; P3[r + 3 * col] = s3;
                    }
            }
            for (int i = lane; i < n; i += 32) {
                double x6[6], X[3];
                load_x6(a.corresp, prob, n, i, x6);
                if (a.X0 != nullptr) {
                    const double* q = a.X0 + (prob * n + i) * 3;
                    X[0] = q[0]; X[1] = q[1]; X[2] = q[2];
                } else {
                    double Xh[4];
                    triangulate3(P1, P2, P3, x6, Xh);
                    X[0] = Xh[0] / Xh[3]; X[1] = Xh[1] / Xh[3]; X[2] = Xh[2] / Xh[3];
                }
#pragma unroll
                for (int k = 0; k < 6; ++k) bad_l = bad_l || !finite_(x6[k]);
                bad_l = bad_l || !(finite_(X[0]) && finite_(X[1]) && finite_(X[2]));
                Xp[3 * i] = X[0]; Xp[3 * i + 1] = X[1]; Xp[3 * i + 2] = X[2];
                cost_l += ba_point_cost(cur, X, x6);
            }
        }
        const double cost0 = warp_sum(cost_l);
        const double t2n = sqrt(cur.t2[0] * cur.t2[0] + cur.t2[1] * cur.t2[1] + cur.t2[2] * cur.t2[2]);
        const bool bad = __any_sync(FULL, bad_l) || !(t2n > 0.0) || !finite_(cost0);
        if (bad) {                                     // inputs copied through (the start points are already in X)
            if (lane < 12) { a.Rt2[prob * 12 + lane] = rt2[lane]; a.Rt3[prob * 12 + lane] = rt3[lane]; }
            if (lane == 0) {
                if (a.repr_err) a.repr_err[prob] = sqrt(cost0 / (3.0 * n));
                if (a.iter) a.iter[prob] = 0;
                if (a.status) a.status[prob] = ST_NONFINITE;
            }
            continue;
        }

        // ---- gauge |t2| = 1: t2, t3 and the points scaled by 1/|t2| ----------------------------------------------
        const double gs = 1.0 / t2n;
        __syncwarp();
        if (lane == 0) {
#pragma unroll
            for (int k = 0; k < 3; ++k) { cur.t2[k] *= gs; cur.t3[k] *= gs; }
            onb3(cur.t2, cur.u1, cur.u2);
        }
        __syncwarp();
        cost_l = 0.0;
        for (int i = lane; i < n; i += 32) {
            double x6[6], X[3];
            load_x6(a.corresp, prob, n, i, x6);
#pragma unroll
            for (int k = 0; k < 3; ++k) { X[k] = Xp[3 * i + k] * gs; Xp[3 * i + k] = X[k]; }
            cost_l += ba_point_cost(cur, X, x6);
        }
        double F = 0.5 * warp_sum(cost_l);            // (1/2) sum of squared residuals

        // ---- Levenberg-Marquardt ---------------------------------------------------------------------------------
        double mu = BA_MU0, nu = 2.0, gmax0 = -1.0;
        int lin = 1, solves = 0, st = 0;
        while (true) {
            // pass A: linearise + eliminate + accumulate
#pragma unroll 1
            for (int e = 0; e < BA_NSUM; ++e) acc[e] = 0.0;
            bool pd_l = true;
            double gp_l = 0.0;
            for (int i = lane; i < n; i += 32) {
                double x6[6];
                load_x6(a.corresp, prob, n, i, x6);
                const double X[3] = {Xp[3 * i], Xp[3 * i + 1], Xp[3 * i + 2]};
                BaPoint p; BaElim el;
                ba_point_jac(cur, X, x6, p);
                pd_l = ba_point_eliminate(p, mu, el) && pd_l;
                ba_point_accumulate(p, el, acc);
                gp_l = fmax(gp_l, fmax(fabs(el.g[0]), fmax(fabs(el.g[1]), fabs(el.g[2]))));
            }
            __syncwarp();
            for (int e = lane; e < BA_NSUM; e += 32) {
                double s = 0.0;
#pragma unroll 8
                for (int l = 0; l < 32; ++l) s += slab[l * BA_NSUM + e];
                red[e] = s;
            }
            __syncwarp();
            double gmax = warp_max(gp_l);
#pragma unroll
            for (int k = 0; k < BA_NC; ++k) gmax = fmax(gmax, fabs(red[BA_GC + k]));
            if (gmax0 < 0.0) gmax0 = gmax;
            if (!(gmax > BA_GTOL * gmax0)) break;                                  // small gradient (or zero)
            const bool pd = !__any_sync(FULL, !pd_l);
            __syncwarp();
            if (lane == 0) dcs[11] = (pd && ba_solve_reduced(red, mu, dcs)) ? 1.0 : 0.0;
            __syncwarp();
            ++solves;
            const bool solved = dcs[11] != 0.0;
            if (solved) {
                double dc[BA_NC];
#pragma unroll
                for (int k = 0; k < BA_NC; ++k) dc[k] = dcs[k];
                if (lane == 0) { cand = cur; ba_update_cams(dc, cand); }
                __syncwarp();
                // pass B: back-substitution and the candidate's cost
                double cn_l = 0.0, pr_l = 0.0, s2_l = 0.0, x2_l = 0.0;
                for (int i = lane; i < n; i += 32) {
                    double x6[6];
                    load_x6(a.corresp, prob, n, i, x6);
                    const double X[3] = {Xp[3 * i], Xp[3 * i + 1], Xp[3 * i + 2]};
                    BaPoint p; BaElim el;
                    ba_point_jac(cur, X, x6, p);
                    ba_point_eliminate(p, mu, el);
                    double dX[3], Xn[3];
                    ba_point_step(el, dc, dX);
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        Xn[k] = X[k] + dX[k];
                        Xcp[3 * i + k] = Xn[k];
                        pr_l += mu * el.d[k] * dX[k] * dX[k] - el.g[k] * dX[k];
                        s2_l += dX[k] * dX[k];
                        x2_l += X[k] * X[k];
                    }
                    cn_l += ba_point_cost(cand, Xn, x6);
                }
                const double Fn = 0.5 * warp_sum(cn_l);
                double pred = warp_sum(pr_l), step2 = warp_sum(s2_l), xn2 = warp_sum(x2_l);
#pragma unroll
                for (int k = 0; k < BA_NC; ++k) {
                    pred += mu * red[BA_DIAG + k] * dc[k] * dc[k] - red[BA_GC + k] * dc[k];
                    step2 += dc[k] * dc[k];
                }
                pred *= 0.5;                           // model decrease (1/2) d'(mu D d - g)
                xn2 += cur.t3[0] * cur.t3[0] + cur.t3[1] * cur.t3[1] + cur.t3[2] * cur.t3[2] + 1.0;
                const bool small_step = !(step2 > BA_XTOL * BA_XTOL * xn2);
                if (Fn < F) {                          // accept
                    const double rho = (F - Fn) / pred;
                    const bool small_change = !(F - Fn > BA_FTOL * F);
                    for (int i = lane; i < n; i += 32)
#pragma unroll
                        for (int k = 0; k < 3; ++k) Xp[3 * i + k] = Xcp[3 * i + k];
                    __syncwarp();
                    if (lane == 0) cur = cand;
                    __syncwarp();
                    F = Fn;
                    const double q = 2.0 * rho - 1.0;
                    mu *= fmax(1.0 / 3.0, 1.0 - q * q * q);       // Nielsen
                    nu = 2.0;
                    if (small_step || small_change) break;
                    if (lin >= BA_IT_MAX) { st = ST_BA_NOCONV; break; }
                    ++lin;
                    continue;
                }
                if (small_step) break;
            }
            mu *= nu; nu *= 2.0;                       // rejected (or not solvable): more damping, same linearisation
            if (solves >= BA_SOLVE_MAX) { st = ST_BA_NOCONV; break; }
        }

        __syncwarp();
        if (lane < 12) {
            a.Rt2[prob * 12 + lane] = (lane < 9) ? cur.R2[lane] : cur.t2[lane - 9];
            a.Rt3[prob * 12 + lane] = (lane < 9) ? cur.R3[lane] : cur.t3[lane - 9];
        }
        if (lane == 0) {
            if (a.repr_err) a.repr_err[prob] = sqrt(2.0 * F / (3.0 * n));        // ReprError.m:65
            if (a.iter) a.iter[prob] = lin;
            if (a.status) a.status[prob] = st;
        }
    }
}

int launch_bundle_adjust(const BaArgs& a, cudaStream_t stream) {
    if (a.B <= 0) return 1;
    const size_t smem = (size_t)BA_WARPS * BA_PER_WARP * sizeof(double);
    // the opt-in is a per-device property of the function: set on every launch, as for optimf_gh_kernel
    if (cudaFuncSetAttribute(bundle_adjust_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    long long blocks = (a.B + BA_WARPS - 1) / BA_WARPS;       // one problem per warp: the block scheduler balances
    if (blocks > 0x7fffffffLL) blocks = 0x7fffffffLL;         // problems of different iteration counts
    bundle_adjust_kernel<<<(unsigned)blocks, BA_WARPS * 32, smem, stream>>>(a);
    return cudaPeekAtLastError() == cudaSuccess ? 1 : 0;
}

}  // namespace tvf
