// tvf_ba_kernels.cu -- batched three-view bundle adjustment (tvf_bundle_adjust): Levenberg-Marquardt on the pixel
// reprojection error with the points eliminated by the Schur complement.  One warp per problem, lanes own points
// (point i belongs to lane i mod 32), the same mapping as optimf_gh_kernel.  Per-point algebra: tvf_ba.cuh.
// bundle_adjust_small_kernel runs the same code on groups of 8 lanes, four problems per warp, for n <= 8 (the RANSAC
// hypotheses of tvf_ransac_pose_refined); "warp" and "lane" below then mean the group and the lane within it.
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
constexpr int BA_CAMS = (sizeof(BaCams) + 7) / 8;      // doubles per BaCams
// shared doubles of one group of W lanes (one problem): W lane-private rows of partial sums (odd stride: conflict-free),
// the reduced sums (+1), the camera step with its solve flag, the current and the candidate cameras
template <int W> constexpr int BA_PER_GROUP = W * BA_NSUM + BA_NSUM + 1 + 12 + 2 * BA_CAMS;

__device__ __forceinline__ bool finite_(double x) { return fabs(x) <= 1.79769313486231570e308; }

__device__ __forceinline__ void load_x6(const double* corresp, long long prob, int n, int i, double* x6) {
    const double2* q = reinterpret_cast<const double2*>(corresp + (prob * n + i) * 6);
    const double2 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
    x6[0] = a.x; x6[1] = a.y; x6[2] = b.x; x6[3] = b.y; x6[4] = c.x; x6[5] = c.y;
}

// sum and max over the W lanes of a group (mask m): warp_sum / warp_max's xor butterfly on the offsets W/2 .. 1
template <int W> __device__ __forceinline__ double group_sum(double v, unsigned m) {
#pragma unroll
    for (int o = W / 2; o > 0; o >>= 1) v += __shfl_xor_sync(m, v, o);
    return v;
}

template <int W> __device__ __forceinline__ double group_max(double v, unsigned m) {
#pragma unroll
    for (int o = W / 2; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(m, v, o));
    return v;
}

// a match's share of the objective: its six squared residuals, or c^2 rho(s / c^2) for the robust adjustment
template <bool Robust> __device__ __forceinline__ double match_cost(const BaCams& c, const double* X, const double* x6,
                                                                   const BaRobustArgs& rob) {
    const double s = ba_point_cost(c, X, x6);
    if constexpr (Robust) return ba_loss_cost(rob.loss, s, rob.scale * rob.scale);
    else return s;
}

// the problems of one group of W lanes (mask gm) in a grid-stride loop; lane = the lane within the group.  Ragged: problem
// prob owns matches a.offs[prob] .. a.offs[prob+1]-1 (n varies per problem); the uniform form indexes by prob * a.n.
// Robust: the objective is sum c^2 rho(s_i / c^2) (rob.loss, rob.scale); each linearisation weighs every match's residuals
// and Jacobian rows by sqrt(rho'(s_i / c^2)) at the current iterate (IRLS), in pass A and pass B alike, so both passes
// form the same elimination from the same inputs.  F is (1/2) cost and the weighted g its gradient, so the schedule and
// the stopping rule are the plain adjustment's.
template <int W, bool Ragged, bool Robust = false>
__device__ __forceinline__ void ba_problems(const BaArgs& a, const BaRobustArgs& rob = BaRobustArgs{}) {
    extern __shared__ __align__(16) double ba_smem[];
    constexpr int G = BA_WARPS * 32 / W;               // groups (problems in flight) per block
    const int lane = threadIdx.x & (W - 1), grp = threadIdx.x / W;
    const unsigned gm = (W == 32) ? FULL : ((1u << W) - 1u) << (threadIdx.x & 31 & ~(W - 1));
    double* slab = ba_smem + (size_t)grp * BA_PER_GROUP<W>;
    double* red = slab + W * BA_NSUM;                  // BA_NSUM (+1)
    double* dcs = red + BA_NSUM + 1;                   // 11 camera step entries + solve flag
    BaCams& cur = *reinterpret_cast<BaCams*>(dcs + 12);
    BaCams& cand = *reinterpret_cast<BaCams*>(dcs + 12 + BA_CAMS);
    double* acc = slab + lane * BA_NSUM;
    const int n_all = a.n;

    for (long long prob = (long long)blockIdx.x * G + grp; prob < a.B; prob += (long long)gridDim.x * G) {
        // ragged: the problem's matches as problem 0 of a batch of n = n_b
        const long long off = Ragged ? a.offs[prob] : 0;
        const int n = Ragged ? (int)(a.offs[prob + 1] - off) : n_all;
        const long long pi = Ragged ? 0 : prob;        // the problem index the point loads use
        const double* corresp = a.corresp + off * 6;
        const double* cm = a.calm + (a.calm_batched ? prob * 27 : 0);
        const double* rt2 = a.Rt2_0 + prob * 12;
        const double* rt3 = a.Rt3_0 + prob * 12;
        double* Xp = Ragged ? a.X + off * 3 : a.X + prob * 3 * n;
        double* Xcp = Ragged ? a.Xc + off * 3 : a.Xc + prob * 3 * n;
        if (Ragged && n < 4) {                         // too few: start poses copied through, points and error NaN
            const double qnan = __longlong_as_double(0x7ff8000000000000LL);
            for (int e = lane; e < 12; e += W) { a.Rt2[prob * 12 + e] = rt2[e]; a.Rt3[prob * 12 + e] = rt3[e]; }
            for (int e = lane; e < 3 * n; e += W) Xp[e] = qnan;
            if constexpr (Robust) {
                if (rob.weights) for (int e = lane; e < n; e += W) rob.weights[off + e] = qnan;
                if (lane == 0 && rob.cost) rob.cost[prob] = qnan;
            }
            if (lane == 0) {
                if (a.repr_err) a.repr_err[prob] = qnan;
                if (a.iter) a.iter[prob] = 0;
                if (a.status) a.status[prob] = ST_TOO_FEW_MATCHES;
            }
            continue;
        }
        __syncwarp(gm);
        if (lane == 0) ba_load_cams(cm, rt2, rt3, cur);
        bool bad_l = false;
        for (int e = lane; e < 27; e += W) bad_l = bad_l || !finite_(cm[e]) || (e < 12 && !(finite_(rt2[e]) && finite_(rt3[e])));
        __syncwarp(gm);

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
            for (int i = lane; i < n; i += W) {
                double x6[6], X[3];
                load_x6(corresp, pi, n, i, x6);
                if (a.X0 != nullptr) {
                    const double* q = a.X0 + (Ragged ? off + i : prob * n + i) * 3;
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
        const double cost0 = group_sum<W>(cost_l, gm);
        const double t2n = sqrt(cur.t2[0] * cur.t2[0] + cur.t2[1] * cur.t2[1] + cur.t2[2] * cur.t2[2]);
        const bool bad = __any_sync(gm, bad_l) || !(t2n > 0.0) || !finite_(cost0);
        if (bad) {                                     // inputs copied through (the start points are already in X)
            for (int e = lane; e < 12; e += W) { a.Rt2[prob * 12 + e] = rt2[e]; a.Rt3[prob * 12 + e] = rt3[e]; }
            if constexpr (Robust) {                    // cost and weights NaN
                const double qnan = __longlong_as_double(0x7ff8000000000000LL);
                if (rob.weights) for (int e = lane; e < n; e += W) rob.weights[(Ragged ? off : prob * n) + e] = qnan;
                if (lane == 0 && rob.cost) rob.cost[prob] = qnan;
            }
            if (lane == 0) {
                if (a.repr_err) a.repr_err[prob] = sqrt(cost0 / (3.0 * n));
                if (a.iter) a.iter[prob] = 0;
                if (a.status) a.status[prob] = ST_NONFINITE;
            }
            continue;
        }

        // ---- gauge |t2| = 1: t2, t3 and the points scaled by 1/|t2| ----------------------------------------------
        const double gs = 1.0 / t2n;
        __syncwarp(gm);
        if (lane == 0) {
#pragma unroll
            for (int k = 0; k < 3; ++k) { cur.t2[k] *= gs; cur.t3[k] *= gs; }
            onb3(cur.t2, cur.u1, cur.u2);
        }
        __syncwarp(gm);
        cost_l = 0.0;
        for (int i = lane; i < n; i += W) {
            double x6[6], X[3];
            load_x6(corresp, pi, n, i, x6);
#pragma unroll
            for (int k = 0; k < 3; ++k) { X[k] = Xp[3 * i + k] * gs; Xp[3 * i + k] = X[k]; }
            cost_l += match_cost<Robust>(cur, X, x6, rob);
        }
        double F = 0.5 * group_sum<W>(cost_l, gm);           // (1/2) sum of squared residuals (robust: (1/2) cost)

        // ---- Levenberg-Marquardt ---------------------------------------------------------------------------------
        double mu = BA_MU0, nu = 2.0, gmax0 = -1.0;
        int lin = 1, solves = 0, st = 0;
        while (true) {
            // pass A: linearise + eliminate + accumulate
#pragma unroll 1
            for (int e = 0; e < BA_NSUM; ++e) acc[e] = 0.0;
            bool pd_l = true;
            double gp_l = 0.0;
            for (int i = lane; i < n; i += W) {
                double x6[6];
                load_x6(corresp, pi, n, i, x6);
                const double X[3] = {Xp[3 * i], Xp[3 * i + 1], Xp[3 * i + 2]};
                BaPoint p; BaElim el;
                ba_point_jac(cur, X, x6, p);
                if constexpr (Robust) ba_point_weigh(p, rob.loss, rob.scale * rob.scale);
                pd_l = ba_point_eliminate(p, mu, el) && pd_l;
                ba_point_accumulate(p, el, acc);
                gp_l = fmax(gp_l, fmax(fabs(el.g[0]), fmax(fabs(el.g[1]), fabs(el.g[2]))));
            }
            __syncwarp(gm);
            for (int e = lane; e < BA_NSUM; e += W) {
                double s = 0.0;
#pragma unroll 8
                for (int l = 0; l < W; ++l) s += slab[l * BA_NSUM + e];
                red[e] = s;
            }
            __syncwarp(gm);
            double gmax = group_max<W>(gp_l, gm);
#pragma unroll
            for (int k = 0; k < BA_NC; ++k) gmax = fmax(gmax, fabs(red[BA_GC + k]));
            if (gmax0 < 0.0) gmax0 = gmax;
            if (!(gmax > BA_GTOL * gmax0)) break;                                  // small gradient (or zero)
            const bool pd = !__any_sync(gm, !pd_l);
            __syncwarp(gm);
            if (lane == 0) dcs[11] = (pd && ba_solve_reduced(red, mu, dcs)) ? 1.0 : 0.0;
            __syncwarp(gm);
            ++solves;
            const bool solved = dcs[11] != 0.0;
            if (solved) {
                double dc[BA_NC];
#pragma unroll
                for (int k = 0; k < BA_NC; ++k) dc[k] = dcs[k];
                if (lane == 0) { cand = cur; ba_update_cams(dc, cand); }
                __syncwarp(gm);
                // pass B: back-substitution and the candidate's cost
                double cn_l = 0.0, pr_l = 0.0, s2_l = 0.0, x2_l = 0.0;
                for (int i = lane; i < n; i += W) {
                    double x6[6];
                    load_x6(corresp, pi, n, i, x6);
                    const double X[3] = {Xp[3 * i], Xp[3 * i + 1], Xp[3 * i + 2]};
                    BaPoint p; BaElim el;
                    ba_point_jac(cur, X, x6, p);
                    if constexpr (Robust) ba_point_weigh(p, rob.loss, rob.scale * rob.scale);
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
                    cn_l += match_cost<Robust>(cand, Xn, x6, rob);
                }
                const double Fn = 0.5 * group_sum<W>(cn_l, gm);
                double pred = group_sum<W>(pr_l, gm), step2 = group_sum<W>(s2_l, gm), xn2 = group_sum<W>(x2_l, gm);
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
                    for (int i = lane; i < n; i += W)
#pragma unroll
                        for (int k = 0; k < 3; ++k) Xp[3 * i + k] = Xcp[3 * i + k];
                    __syncwarp(gm);
                    if (lane == 0) cur = cand;
                    __syncwarp(gm);
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

        __syncwarp(gm);
        for (int e = lane; e < 12; e += W) {
            a.Rt2[prob * 12 + e] = (e < 9) ? cur.R2[e] : cur.t2[e - 9];
            a.Rt3[prob * 12 + e] = (e < 9) ? cur.R3[e] : cur.t3[e - 9];
        }
        if constexpr (Robust) {                        // the weights and the plain ReprError at the result
            double s_l = 0.0;
            for (int i = lane; i < n; i += W) {
                double x6[6];
                load_x6(corresp, pi, n, i, x6);
                const double X[3] = {Xp[3 * i], Xp[3 * i + 1], Xp[3 * i + 2]};
                const double s = ba_point_cost(cur, X, x6);
                if (rob.weights) rob.weights[(Ragged ? off : prob * n) + i] = ba_loss_weight(rob.loss, s, rob.scale * rob.scale);
                s_l += s;
            }
            const double s_all = group_sum<W>(s_l, gm);
            if (lane == 0) {
                if (a.repr_err) a.repr_err[prob] = sqrt(s_all / (3.0 * n));
                if (rob.cost) rob.cost[prob] = 2.0 * F;
                if (a.iter) a.iter[prob] = lin;
                if (a.status) a.status[prob] = st;
            }
        } else if (lane == 0) {
            if (a.repr_err) a.repr_err[prob] = sqrt(2.0 * F / (3.0 * n));        // ReprError.m:65
            if (a.iter) a.iter[prob] = lin;
            if (a.status) a.status[prob] = st;
        }
    }
}

__global__ void __launch_bounds__(BA_WARPS * 32) bundle_adjust_kernel(const BaArgs a) { ba_problems<32, false>(a); }
// the ragged batch (a.offs): the same code per problem at n = n_b, so bit-identical to bundle_adjust_kernel on it alone
__global__ void __launch_bounds__(BA_WARPS * 32) bundle_adjust_ragged_kernel(const BaArgs a) { ba_problems<32, true>(a); }

// Packed variant for n <= 8: groups of 8 lanes, four problems per warp.  Bit-identical to bundle_adjust_kernel on the
// same problem, because at n <= 8 lanes 8..31 of bundle_adjust_kernel own no point and contribute exact +0.0:
//   - a lane-private sum (cost, model decrease, step, |X|^2) starts at +0.0 and only adds, so it is never -0.0; the
//     first two xor steps of warp_sum (offsets 16, 8) add +0.0 to it on lanes 0..7 and change nothing, and the
//     remaining offsets 4, 2, 1 are group_sum<8>'s butterfly over the same lanes in the same order;
//   - warp_max of non-negative values: fmax with the +0.0 of the idle lanes changes nothing either;
//   - the slab sum s = 0.0; s += slab[l] (l ascending) never holds -0.0, so adding the 24 trailing +0.0 rows of the
//     idle lanes leaves it as group 8's sum over l = 0..7;
//   - every vote (__any_sync) of the idle lanes is false, and every other step is done by lane 0 or per point.
__global__ void __launch_bounds__(BA_WARPS * 32) bundle_adjust_small_kernel(const BaArgs a) { ba_problems<BA_SMALL_N, false>(a); }

// the robust-loss adjustment (tvf_bundle_adjust_robust), uniform and ragged; the loss id is warp-uniform
__global__ void __launch_bounds__(BA_WARPS * 32) bundle_adjust_robust_kernel(const BaArgs a, const BaRobustArgs rob) {
    ba_problems<32, false, true>(a, rob);
}
__global__ void __launch_bounds__(BA_WARPS * 32) bundle_adjust_robust_ragged_kernel(const BaArgs a, const BaRobustArgs rob) {
    ba_problems<32, true, true>(a, rob);
}

template <int W, class Kernel, class... Extra>
int launch_groups(Kernel kernel, const BaArgs& a, cudaStream_t stream, const Extra&... extra) {
    if (a.B <= 0) return 1;
    constexpr int G = BA_WARPS * 32 / W;
    const size_t smem = (size_t)G * BA_PER_GROUP<W> * sizeof(double);
    // the opt-in is a per-device property of the function: set on every launch, as for optimf_gh_kernel
    if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    long long blocks = (a.B + G - 1) / G;              // one problem per group: the block scheduler balances
    if (blocks > 0x7fffffffLL) blocks = 0x7fffffffLL;  // problems of different iteration counts
    kernel<<<(unsigned)blocks, BA_WARPS * 32, smem, stream>>>(a, extra...);
    return cudaPeekAtLastError() == cudaSuccess ? 1 : 0;
}

int launch_bundle_adjust(const BaArgs& a, cudaStream_t stream) {
    return launch_groups<32>(a.offs ? bundle_adjust_ragged_kernel : bundle_adjust_kernel, a, stream);
}

int launch_bundle_adjust_small(const BaArgs& a, cudaStream_t stream) {
    if (a.n > BA_SMALL_N) return 0;
    return launch_groups<BA_SMALL_N>(bundle_adjust_small_kernel, a, stream);
}

int launch_bundle_adjust_robust(const BaArgs& a, const BaRobustArgs& r, cudaStream_t stream) {
    return launch_groups<32>(a.offs ? bundle_adjust_robust_ragged_kernel : bundle_adjust_robust_kernel, a, stream, r);
}

}  // namespace tvf
