// tvf_core_kernels.cu -- the two model estimators.
//
// linearTFT (TFT_methods/linearTFT.m:36-91, called from LinearTFTPoseEstimation.m:45-53):
//   tft_stage1_kernel   warp per problem   Normalize2Ddata x3 -> 96 Kronecker moments -> 27x27 Gram
//                                          -> null vector t1 (linearTFT.m:45-67)
//   tft_epipoles_kernel thread per problem epipoles of t1: eight 3x3 SVDs (linearTFT.m:71-79)
//   tft_stage2_kernel   warp per problem   15-dim constrained re-solve in range(E), P2/P3, undo the
//                                          normalisation (linearTFT.m:82-91, LinearTFTPoseEstimation.m:53)
// linearF (F_methods/linearF.m:32-62, called from LinearFPoseEstimation.m:46-56):
//   f_stage1_kernel     warp per problem   (re-)normalisation, 36 moments, 9x9 Gram -> null vector
//   f_finish_kernel     thread per problem undo inner normalisation, rank-2 projection, undo outer one
//
// The design matrix never exists: G = A'A = sum_i (p1 p1') (x) (S3 S3') (x) (S2 S2') is assembled from
// 96 per-problem moments (SURVEY.md A.2), and the second null-vector problem needs no second pass over
// the points because (A*Up)'(A*Up) = Up' G Up.  The scalar 3x3 SVD work sits in thread-per-problem
// kernels so that it runs at 32 problems per warp instead of one.
#include "tvf_kernels.h"
#include "tvf_warp.cuh"
#include "tvf_pose.cuh"
#include "tvf_async.cuh"

namespace tvf {

// Launch-shape knobs of the estimator kernels.  The defaults are the measured optimum on B200 (tools/build_variants.py
// builds the alternatives, profiles/r01_variants.md has the sweep): 4 warps per CTA, 5 CTAs per SM (96 registers), warps
// of a CTA kept in step.
#ifndef TVF_CORE_WARPS
#define TVF_CORE_WARPS 4
#endif
#ifndef TVF_CORE_MINB
#define TVF_CORE_MINB 5
#endif
// MUFU-seeded square root / reciprocal (full precision, not correctly rounded) in the normalisation statistics of the
// estimator kernels; the stand-alone Normalize2Ddata kernel keeps the IEEE operations
#ifndef TVF_FAST_STATS
#define TVF_FAST_STATS 1
#endif
#ifndef TVF_STEP_SYNC
#define TVF_STEP_SYNC 1
#endif
// per-kernel overrides: the stage-2 two-problem kernel runs faster WITHOUT the barrier (26.6 against 27.4 ms per 10 M, its
// warps' iteration counts differ), the two-problem stage-1 solver faster WITH it (40.8 against 44.3)
#ifndef TVF_S2_SYNC
#define TVF_S2_SYNC 0
#endif
#ifndef TVF_S1D_SYNC
#define TVF_S1D_SYNC 1
#endif
#if TVF_S2_SYNC
#define S2_SYNC() __syncthreads()
#else
#define S2_SYNC() ((void)0)
#endif
#if TVF_S1D_SYNC
#define S1D_SYNC() __syncthreads()
#else
#define S1D_SYNC() ((void)0)
#endif
#if TVF_STEP_SYNC
#define STEP_SYNC() __syncthreads()
#else
#define STEP_SYNC() ((void)0)
#endif
constexpr int CORE_WARPS = TVF_CORE_WARPS;
constexpr int CORE_MINB = TVF_CORE_MINB;      // resident CTAs per SM the estimator kernels are compiled for
constexpr int FEAT_STRIDE = 15;   // 14 features + 1 pad: conflict-free 64-bit lane-strided stores

// per-problem work-space record handed from stage to stage (doubles)
constexpr int CW_MOM = 0, CW_STATS = 96, CW_T1 = 106, CW_EPI = 134;      // CORE_WS_TFT = 140
constexpr int FW_F = 0, FW_STATS = 18;                                   // CORE_WS_F = 36

__device__ __constant__ unsigned char c_sym6[9] = {0, 1, 2, 1, 3, 4, 2, 4, 5};
__device__ __constant__ signed char c_m4[9] = {0, -1, 1, -1, 0, 2, 1, 2, 3};

// v[i] for a runtime i without forcing the array into local memory
__device__ __forceinline__ double sel3(const double* v, int i) { return (i == 0) ? v[0] : ((i == 1) ? v[1] : v[2]); }

// PACKED: 0 = three separate point arrays, 1 = 6 x n correspondences in global memory, 2 = the same layout staged in
// shared memory (in.p1 = the stage, prob = index inside it)
template <int PACKED>
__device__ __forceinline__ void load_point(const CoreInput& in, long long prob, int i, double* p) {
    if (PACKED == 2) {
        const unsigned addr = smem_u32(in.p1) + (unsigned)(((int)prob * in.n + i) * 48);
        asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(p[0]), "=d"(p[1]) : "r"(addr));
        asm volatile("ld.shared.v2.f64 {%0, %1}, [%2+16];" : "=d"(p[2]), "=d"(p[3]) : "r"(addr));
        asm volatile("ld.shared.v2.f64 {%0, %1}, [%2+32];" : "=d"(p[4]), "=d"(p[5]) : "r"(addr));
    } else if (PACKED) {
        const double2* q = reinterpret_cast<const double2*>(in.p1 + (prob * in.n + i) * 6);
        const double2 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
        p[0] = a.x; p[1] = a.y; p[2] = b.x; p[3] = b.y; p[4] = c.x; p[5] = c.y;
    } else {
        const long long o = (prob * in.n + i) * in.rows;
        const double* ps[3] = {in.p1, in.p2, in.p3};
#pragma unroll
        for (int v = 0; v < 3; ++v) {
            if (ps[v] == nullptr) { p[2 * v] = 0.0; p[2 * v + 1] = 0.0; continue; }
            double x = ps[v][o], y = ps[v][o + 1];
            if (in.rows == 3) { const double w = ps[v][o + 2]; x /= w; y /= w; }   // linearTFT.m:39-43
            p[2 * v] = x; p[2 * v + 1] = y;
        }
    }
}

// Normalize2Ddata.m:34-37 for the three views at once, on points already mapped by
// x -> s0*x + t0 (identity when there is no outer map).  new = s*x + t.
template <bool PACKED>
__device__ __forceinline__ void view_stats(const CoreInput& in, long long prob, int lane,
                                           const double* s0, const double* t0, double* s, double* t) {
    const int n = in.n;
    double sum[6] = {0, 0, 0, 0, 0, 0};
    for (int i = lane; i < n; i += 32) {
        double p[6];
        load_point<PACKED>(in, prob, i, p);
#pragma unroll
        for (int q = 0; q < 6; ++q) sum[q] += s0[q >> 1] * p[q] + t0[q];
    }
    const double invn = 1.0 / (double)n;
    double c[6];
#pragma unroll
    for (int q = 0; q < 6; ++q) c[q] = warp_sum(sum[q]) * invn;
    double d[3] = {0, 0, 0};
    for (int i = lane; i < n; i += 32) {
        double p[6];
        load_point<PACKED>(in, prob, i, p);
#pragma unroll
        for (int v = 0; v < 3; ++v) {
            const double dx = (s0[v] * p[2 * v] + t0[2 * v]) - c[2 * v];
            const double dy = (s0[v] * p[2 * v + 1] + t0[2 * v + 1]) - c[2 * v + 1];
#if TVF_FAST_STATS
            d[v] += sqrt_(dx * dx + dy * dy);
#else
            d[v] += sqrt(dx * dx + dy * dy);
#endif
        }
    }
#pragma unroll
    for (int v = 0; v < 3; ++v) {
        const double norm0 = warp_sum(d[v]) * invn;
#if TVF_FAST_STATS
        s[v] = 1.4142135623730951 * rcp_(norm0);
#else
        s[v] = 1.4142135623730951 / norm0;
#endif
        t[2 * v] = -s[v] * c[2 * v];
        t[2 * v + 1] = -s[v] * c[2 * v + 1];
    }
}

constexpr int REFINE_N_MAX = 12;      // systems with fewer points get refinement steps (needs n <= 32: one point per lane)

// (A'A) x for the trilinearity design matrix of linearTFT.m:45-62, from the rows themselves: lane = point
// computes its 4 residuals y = A_i x and its contribution A_i' y; a transposed butterfly leaves component r
// of the total on lane r.  xs: 27 doubles in shared memory.  (s,t): normalisation of the three views.
template <bool PACKED>
__device__ __forceinline__ double tft_apply_AtA(const CoreInput& in, long long prob, int lane, const double* s,
                                                const double* t, const double* xs) {
    double c[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) c[k] = 0.0;
    if (lane < in.n) {
        double p[6];
        load_point<PACKED>(in, prob, lane, p);
        const double x1 = s[0] * p[0] + t[0], y1 = s[0] * p[1] + t[1];
        const double x2 = s[1] * p[2] + t[2], y2 = s[1] * p[3] + t[3];
        const double x3 = s[2] * p[4] + t[4], y3 = s[2] * p[5] + t[5];
        // rows are p1' (x) b' (x) a' with a in {(1,0,-x2),(0,1,-y2)}, b in {(1,0,-x3),(0,1,-y3)}
        double v[2][2][3];      // [a][b][i]
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            double u0[3], u1[3];    // contraction with a, per k
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const double X0 = xs[3 * k + 9 * i], X1 = xs[1 + 3 * k + 9 * i], X2 = xs[2 + 3 * k + 9 * i];
                u0[k] = X0 - x2 * X2; u1[k] = X1 - y2 * X2;
            }
            v[0][0][i] = u0[0] - x3 * u0[2]; v[0][1][i] = u0[1] - y3 * u0[2];
            v[1][0][i] = u1[0] - x3 * u1[2]; v[1][1][i] = u1[1] - y3 * u1[2];
        }
        const double y00 = x1 * v[0][0][0] + y1 * v[0][0][1] + v[0][0][2];
        const double y01 = x1 * v[0][1][0] + y1 * v[0][1][1] + v[0][1][2];
        const double y10 = x1 * v[1][0][0] + y1 * v[1][0][1] + v[1][0][2];
        const double y11 = x1 * v[1][1][0] + y1 * v[1][1][1] + v[1][1][2];
        // z[k][j] = sum_ab y_ab b_b[k] a_a[j]
        double z[3][3];
        z[0][0] = y00; z[0][1] = y10; z[0][2] = -x2 * y00 - y2 * y10;
        z[1][0] = y01; z[1][1] = y11; z[1][2] = -x2 * y01 - y2 * y11;
#pragma unroll
        for (int j = 0; j < 3; ++j) z[2][j] = -x3 * z[0][j] - y3 * z[1][j];
        const double p1[3] = {x1, y1, 1.0};
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int k = 0; k < 3; ++k)
#pragma unroll
                for (int j = 0; j < 3; ++j) c[j + 3 * k + 9 * i] = p1[i] * z[k][j];
    }
    return warp_reduce_transposed32(c, lane);
}

// (A'A) f for the eight-point design matrix of linearF.m:49-53 (rows [x1x2,x1y2,x1,y1x2,y1y2,y1,x2,y2,1]).
// (sa,ta*) / (sb,tb*): composed normalisation of the two views; va,vb: which views.
template <bool PACKED>
__device__ __forceinline__ double f_apply_AtA(const CoreInput& in, long long prob, int lane, int vb, double sa, double tax,
                                              double tay, double sb, double tbx, double tby, const double* fs) {
    double c[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) c[k] = 0.0;
    if (lane < in.n) {
        double p[6];
        load_point<PACKED>(in, prob, lane, p);
        const double xb = (vb == 1) ? p[2] : p[4], yb = (vb == 1) ? p[3] : p[5];
        const double a[3] = {sa * p[0] + tax, sa * p[1] + tay, 1.0};
        const double b[3] = {sb * xb + tbx, sb * yb + tby, 1.0};
        double y = 0.0;
#pragma unroll
        for (int q = 0; q < 3; ++q)
#pragma unroll
            for (int r = 0; r < 3; ++r) y = fma(a[q] * b[r], fs[3 * q + r], y);
#pragma unroll
        for (int q = 0; q < 3; ++q)
#pragma unroll
            for (int r = 0; r < 3; ++r) c[3 * q + r] = y * a[q] * b[r];
    }
    return warp_reduce_transposed32(c, lane);
}

// G(r,c) -> moment index (96 = structural zero), one table per CTA
__device__ __forceinline__ void build_gidx(unsigned char* gidx) {
    for (int e = threadIdx.x; e < 32 * 27; e += blockDim.x) {
        const int r = e / 27, c = e % 27;
        int idx = 96;                        // structural zeros of the Gram (and rows >= 27) read a slot that holds 0.0
        if (r < 27) {
            const int j = r % 3, k = (r / 3) % 3, i = r / 9;
            const int j2 = c % 3, k2 = (c / 3) % 3, i2 = c / 9;
            const int g = c_m4[j * 3 + j2], b = c_m4[k * 3 + k2];
            if (g >= 0 && b >= 0) idx = c_sym6[i * 3 + i2] * 16 + b * 4 + g;
        }
        gidx[e] = (unsigned char)idx;
    }
}

// trace of the 27 x 27 Gram from its moments: the diagonal entry of row (i,k,j) is moment sym6(i,i)*16 + m4(k,k)*4 +
// m4(j,j) with sym6(i,i) in {0,3,5} and m4(k,k) in {0,0,3}: 12 moments, which occur nowhere else in the Gram
__device__ __forceinline__ bool is_diag_moment(int idx) {
    const int a = idx >> 4, bg = idx & 15;
    return (a == 0 || a == 3 || a == 5) && (bg == 0 || bg == 3 || bg == 12 || bg == 15);
}
__device__ __forceinline__ double diag_moment_weight(int idx) {       // how many diagonal entries equal this moment
    const int bg = idx & 15;
    return (bg == 0) ? 4.0 : ((bg == 15) ? 1.0 : 2.0);
}
__device__ __forceinline__ double gram_trace_from_moments(const double* mom) {
    double tr = 0.0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const int o = (a == 0) ? 0 : ((a == 1) ? 48 : 80);
        tr += 4.0 * mom[o] + 2.0 * (mom[o + 3] + mom[o + 12]) + mom[o + 15];
    }
    return tr;
}

// =========================================================================== TFT stage 1
struct __align__(16) Stage1Scratch {
    double sbuf[64];                 // solver row/vector buffers
    double feat[32 * FEAT_STRIDE];   // per-point features
    double mom[98];                  // 96 moments + zero sentinel
};

// null vector of the 27x27 Gram assembled from the 96 moments in sc.mom (linearTFT.m:64-67)
template <class Resid>
__device__ __forceinline__ void solve_from_moments(Stage1Scratch& sc, const unsigned char* gidx, double* rec, int lane,
                                                   int* status, long long prob, Resid resid, int nrefine) {
    double g[27];
#pragma unroll
    for (int c = 0; c < 27; ++c) g[c] = sc.mom[gidx[lane * 27 + c]];
    bool conv;
    const double tl = smallest_eigvec_spd<27>(g, lane, sc.sbuf, &conv, resid, nrefine);
    if (lane < 27) rec[CW_T1 + lane] = tl;
    if (status != nullptr && lane == 0) status[prob] = conv ? 0 : ST_EIG_NOCONV;
}

template <bool PACKED, bool REFINE>
__global__ void __launch_bounds__(CORE_WARPS * 32, REFINE ? 3 : CORE_MINB)
tft_stage1_kernel(CoreInput in, double* __restrict__ ws, int* __restrict__ status) {
    __shared__ Stage1Scratch scratch[CORE_WARPS];
    __shared__ unsigned char gidx[32 * 27];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    build_gidx(gidx);
    __syncthreads();
    Stage1Scratch& sc = scratch[warp];
    const int beta = (lane >> 2) & 3, gamma = lane & 3, alpha0 = lane >> 4;

    for (long long base = (long long)blockIdx.x * CORE_WARPS; base < in.B; base += (long long)gridDim.x * CORE_WARPS) {
        STEP_SYNC();                 // keeps the CTA's warps in step: they share instruction-cache lines
        const long long prob = base + warp;
        if (prob >= in.B) continue;
        double* rec = ws + prob * CORE_WS_TFT;
        // ---- normalisation (LinearTFTPoseEstimation.m:45-47) -----------------------------
        double s[3] = {1.0, 1.0, 1.0}, t[6] = {0, 0, 0, 0, 0, 0};
        if (in.normalize) {
            const double s0[3] = {1.0, 1.0, 1.0}, t0[6] = {0, 0, 0, 0, 0, 0};
            view_stats<PACKED>(in, prob, lane, s0, t0, s, t);
        }
        // ---- 96 moments: lane l accumulates moments l, l+32, l+64 -----------------------
        double acc0 = 0.0, acc1 = 0.0, acc2 = 0.0;
        for (int pbase = 0; pbase < in.n; pbase += 32) {
            const int cnt = min(32, in.n - pbase);
            __syncwarp();
            if (lane < cnt) {
                double p[6];
                load_point<PACKED>(in, prob, pbase + lane, p);
                const double x1 = s[0] * p[0] + t[0], y1 = s[0] * p[1] + t[1];
                const double x2 = s[1] * p[2] + t[2], y2 = s[1] * p[3] + t[3];
                const double x3 = s[2] * p[4] + t[4], y3 = s[2] * p[5] + t[5];
                double* f = sc.feat + lane * FEAT_STRIDE;
                f[0] = x1 * x1; f[1] = x1 * y1; f[2] = x1; f[3] = y1 * y1; f[4] = y1; f[5] = 1.0;
                f[6] = 1.0; f[7] = -x3; f[8] = -y3; f[9] = x3 * x3 + y3 * y3;
                f[10] = 1.0; f[11] = -x2; f[12] = -y2; f[13] = x2 * x2 + y2 * y2;
            }
            __syncwarp();
            for (int p = 0; p < cnt; ++p) {
                const double* f = sc.feat + p * FEAT_STRIDE;
                const double bc = f[6 + beta] * f[10 + gamma];
                acc0 = fma(f[alpha0], bc, acc0);
                acc1 = fma(f[alpha0 + 2], bc, acc1);
                acc2 = fma(f[alpha0 + 4], bc, acc2);
            }
        }
        __syncwarp();
        sc.mom[lane] = acc0; sc.mom[lane + 32] = acc1; sc.mom[lane + 64] = acc2;
        if (lane == 0) { sc.mom[96] = 0.0; sc.mom[97] = 0.0; }
        rec[CW_MOM + lane] = acc0; rec[CW_MOM + 32 + lane] = acc1; rec[CW_MOM + 64 + lane] = acc2;
        if (lane < 3) rec[CW_STATS + lane] = sel3(s, lane);
        if (lane < 6) rec[CW_STATS + 3 + lane] = (lane < 3) ? sel3(t, lane) : sel3(t + 3, lane - 3);
        __syncwarp();
        if constexpr (REFINE) {
            solve_from_moments(sc, gidx, rec, lane, status, prob,
                               [&](const double* xs) { return tft_apply_AtA<PACKED>(in, prob, lane, s, t, xs); }, 2);
        } else {
            solve_from_moments(sc, gidx, rec, lane, status, prob, NoRefine(), 0);
        }
    }
}

// =========================================================================== TFT stage 1, two problems per warp
// n >= REFINE_N_MAX.  Half h of a warp owns problem 2*pair + h from the first load to the last store: the normalisation
// statistics (points r, r + 16, ... of the problem on lane r; 4-step half-warp reductions), the 96 moments (lane r owns
// the view-3 x view-2 product (beta, gamma) = (r >> 2, r & 3) and accumulates it against all six view-1 features: one
// product, six DFMAs and five shared loads per point for BOTH problems), the unit-trace scaling and diagonal shift
// applied to the moment table (the 12 moments that make up the diagonal of the Gram occur nowhere else in it, so the
// shift is added to them), the gather of rows r and r + 14, and the two-rows-per-lane solver above.
#ifndef TVF_STAGE1_DUAL
#define TVF_STAGE1_DUAL 1
#endif
// solver of the split stage 1 (and of the large-n path): 1 = one problem per warp, one matrix row per lane (96
// registers, 20 warps per SM), 2 = two problems per warp, two rows per lane (168 registers, 12 warps per SM: 22 % fewer
// instructions but measured 18 % SLOWER -- the per-sweep reciprocal / publish / read-back chain is exposed with so few warps)
#ifndef TVF_S1_SOLVER
#define TVF_S1_SOLVER 2
#endif
// 8-byte asynchronous global -> shared copy (LDGSTS) and the wait for all of this thread's copies
__device__ __forceinline__ void cp_async8(double* smem_dst, const double* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

#ifndef TVF_S1D_PREFETCH
#define TVF_S1D_PREFETCH 1
#endif
#ifndef TVF_S1D_MINB
#define TVF_S1D_MINB 3
#endif
constexpr int S1D_FEAT = 18;         // feature row stride (doubles): rows stay 16-byte aligned, lane-strided stores 2-way

struct __align__(16) Stage1DualScratch {
    double sbuf[128];                // solver row/vector buffers: [parity][half][32]
    double feat[2][16 * S1D_FEAT];   // per half: features of 16 points
    double mom[2][100];              // per half: 96 scaled + shifted moments, zero sentinel at 96
};

// scaled + shifted moment table in sc.mom[h] -> rows r and r + 14 -> null vector -> rec
__device__ __forceinline__ void solve_pair_scaled(Stage1DualScratch& sc, const unsigned char* gidx, int lane, bool live,
                                                  double* rec, int* status, long long prob) {
    const int h = lane >> 4, r = lane & 15;
    const double* mom = sc.mom[h];
    const int row0 = (r < 14) ? r : 31, row1 = (r < 13) ? r + 14 : 31;          // rows >= 27 gather the zero sentinel
    double g0[27], g1[27];
#pragma unroll
    for (int c = 0; c < 27; ++c) { g0[c] = mom[gidx[row0 * 27 + c]]; g1[c] = mom[gidx[row1 * 27 + c]]; }
    double x0, x1;
    bool conv;
    smallest_eigvec_spd_half2<27>(g0, g1, lane, sc.sbuf, &x0, &x1, &conv);
    if (live) {
        if (r < 14) rec[CW_T1 + r] = x0;
        if (r < 13) rec[CW_T1 + 14 + r] = x1;
        if (status != nullptr && r == 0) status[prob] = conv ? 0 : ST_EIG_NOCONV;
    }
}

// moments in sc.mom[h] (raw) -> scaled to unit trace, shifted; then rows r and r + 14 -> null vector -> rec
// (raw: where the unscaled moments of this half lie -- sc.mom[h] itself, or the prefetch buffer of the solve-only kernel)
__device__ __forceinline__ void solve_pair_from_moments(Stage1DualScratch& sc, const unsigned char* gidx, int lane, bool live,
                                                        double* rec, int* status, long long prob, const double* raw) {
    const int h = lane >> 4, r = lane & 15;
    double* mom = sc.mom[h];
    const double tr = gram_trace_from_moments(raw);
    const double scl = 1.0 / tr;
    const double delta = 1.0e-13 / 27.0;
    __syncwarp();
#pragma unroll
    for (int q = 0; q < 6; ++q) {
        const int idx = q * 16 + r;
        mom[idx] = fma(raw[idx], scl, is_diag_moment(idx) ? delta : 0.0);
    }
    __syncwarp();
    solve_pair_scaled(sc, gidx, lane, live, rec, status, prob);
}

// Normalisation statistics and the 96 moments of one problem on one half-warp (r = lane & 15).  feat: this half's
// 16 x S1D_FEAT staging buffer.  acc[q] receives moment q*16 + r; (s, t): new = s*x + t per view.
template <int PACKED>
__device__ __forceinline__ void half_stats_moments(const CoreInput& in, long long prob, int r, double* feat, double (&acc)[6],
                                                   double (&s)[3], double (&t)[6]) {
    const int n = in.n;
    const int beta = r >> 2, gamma = r & 3;
    const double invn = 1.0 / (double)n;
    s[0] = s[1] = s[2] = 1.0;
#pragma unroll
    for (int q = 0; q < 6; ++q) { t[q] = 0.0; acc[q] = 0.0; }
    // ---- normalisation (LinearTFTPoseEstimation.m:45-47 -> Normalize2Ddata.m:34-37), three views at once -------
    if (in.normalize) {
        double sum[6] = {0, 0, 0, 0, 0, 0};
        for (int i = r; i < n; i += 16) {
            double p[6];
            load_point<PACKED>(in, prob, i, p);
#pragma unroll
            for (int q = 0; q < 6; ++q) sum[q] += p[q];
        }
        double c[6];
#pragma unroll
        for (int q = 0; q < 6; ++q) c[q] = half_sum(sum[q]) * invn;
        double d[3] = {0, 0, 0};
        for (int i = r; i < n; i += 16) {
            double p[6];
            load_point<PACKED>(in, prob, i, p);
#pragma unroll
            for (int v = 0; v < 3; ++v) {
                const double dx = p[2 * v] - c[2 * v], dy = p[2 * v + 1] - c[2 * v + 1];
#if TVF_FAST_STATS
                d[v] += sqrt_(dx * dx + dy * dy);
#else
                d[v] += sqrt(dx * dx + dy * dy);
#endif
            }
        }
#pragma unroll
        for (int v = 0; v < 3; ++v) {
            const double norm0 = half_sum(d[v]) * invn;
#if TVF_FAST_STATS
            s[v] = 1.4142135623730951 * rcp_(norm0);
#else
            s[v] = 1.4142135623730951 / norm0;
#endif
            t[2 * v] = -s[v] * c[2 * v];
            t[2 * v + 1] = -s[v] * c[2 * v + 1];
        }
    }
    // ---- 96 moments: lane r owns (beta, gamma) and all six alpha ----------------------------------------------
    for (int pbase = 0; pbase < n; pbase += 16) {
        const int cnt = min(16, n - pbase);
        __syncwarp();
        if (r < cnt) {
            double p[6];
            load_point<PACKED>(in, prob, pbase + r, p);
            const double x1 = s[0] * p[0] + t[0], y1 = s[0] * p[1] + t[1];
            const double x2 = s[1] * p[2] + t[2], y2 = s[1] * p[3] + t[3];
            const double x3 = s[2] * p[4] + t[4], y3 = s[2] * p[5] + t[5];
            double2* f2 = reinterpret_cast<double2*>(feat + r * S1D_FEAT);
            f2[0] = make_double2(x1 * x1, x1 * y1); f2[1] = make_double2(x1, y1 * y1); f2[2] = make_double2(y1, 1.0);
            f2[3] = make_double2(1.0, -x3); f2[4] = make_double2(-y3, x3 * x3 + y3 * y3);
            f2[5] = make_double2(1.0, -x2); f2[6] = make_double2(-y2, x2 * x2 + y2 * y2);
        }
        __syncwarp();
        for (int p = 0; p < cnt; ++p) {
            const double* f = feat + p * S1D_FEAT;
            const double2* f2 = reinterpret_cast<const double2*>(f);
            const double bc = f[6 + beta] * f[10 + gamma];
            const double2 a01 = f2[0], a23 = f2[1], a45 = f2[2];
            acc[0] = fma(a01.x, bc, acc[0]); acc[1] = fma(a01.y, bc, acc[1]); acc[2] = fma(a23.x, bc, acc[2]);
            acc[3] = fma(a23.y, bc, acc[3]); acc[4] = fma(a45.x, bc, acc[4]); acc[5] = fma(a45.y, bc, acc[5]);
        }
    }
    __syncwarp();
}

__device__ __forceinline__ void store_moments_stats(double* rec, int r, const double (&acc)[6], const double (&s)[3], const double (&t)[6]) {
#pragma unroll
    for (int q = 0; q < 6; ++q) rec[CW_MOM + q * 16 + r] = acc[q];
    if (r < 3) rec[CW_STATS + r] = sel3(s, r);
    if (r < 6) rec[CW_STATS + 3 + r] = (r < 3) ? sel3(t, r) : sel3(t + 3, r - 3);
}

template <bool PACKED>
__global__ void __launch_bounds__(CORE_WARPS * 32, TVF_S1D_MINB)
tft_stage1_dual_kernel(CoreInput in, double* __restrict__ ws, int* __restrict__ status) {
    __shared__ Stage1DualScratch scratch[CORE_WARPS];
    __shared__ unsigned char gidx[32 * 27];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    build_gidx(gidx);
    __syncthreads();
    Stage1DualScratch& sc = scratch[warp];
    const int h = lane >> 4, r = lane & 15;
    const long long npairs = (in.B + 1) / 2;

    for (long long base = (long long)blockIdx.x * CORE_WARPS; base < npairs; base += (long long)gridDim.x * CORE_WARPS) {
        STEP_SYNC();
        const long long pair = base + warp;
        if (pair >= npairs) continue;
        const bool live = 2 * pair + h < in.B;
        const long long prob = live ? 2 * pair + h : in.B - 1;          // odd batch: the idle half repeats the last problem
        double* rec = ws + prob * CORE_WS_TFT;
        double acc[6], s[3], t[6];
        half_stats_moments<PACKED>(in, prob, r, sc.feat[h], acc, s, t);
#pragma unroll
        for (int q = 0; q < 6; ++q) sc.mom[h][q * 16 + r] = acc[q];
        if (r < 4) sc.mom[h][96 + r] = 0.0;
        if (live) store_moments_stats(rec, r, acc, s, t);
        __syncwarp();
        solve_pair_from_moments(sc, gidx, lane, live, rec, status, prob, sc.mom[h]);
    }
}

// The first half on its own, compiled for many resident warps (it needs few registers and is latency bound: global
// loads, shuffle reductions, square-root chains): statistics + moments -> work-space record.  The solve then runs as
// tft_stage1_solve_dual_kernel.  (TVF_STAGE1_SPLIT; the fused kernel above holds 54 matrix doubles per lane, which
// caps it at 12 warps per SM for its whole run.)
#ifndef TVF_STAGE1_SPLIT
#define TVF_STAGE1_SPLIT 1
#endif
#ifndef TVF_S1M_MINB
#define TVF_S1M_MINB 10
#endif
struct __align__(16) MomentsScratch {
    double feat[2][16 * S1D_FEAT];
};

template <bool PACKED>
__global__ void __launch_bounds__(CORE_WARPS * 32, TVF_S1M_MINB)
tft_moments_kernel(CoreInput in, double* __restrict__ ws) {
    __shared__ MomentsScratch scratch[CORE_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int h = lane >> 4, r = lane & 15;
    const long long npairs = (in.B + 1) / 2;
    for (long long pair = (long long)blockIdx.x * CORE_WARPS + warp; pair < npairs; pair += (long long)gridDim.x * CORE_WARPS) {
        const bool live = 2 * pair + h < in.B;
        const long long prob = live ? 2 * pair + h : in.B - 1;
        double acc[6], s[3], t[6];
        half_stats_moments<PACKED>(in, prob, r, scratch[warp].feat[h], acc, s, t);
        if (live) store_moments_stats(ws + prob * CORE_WS_TFT, r, acc, s, t);
    }
}

// The same with the correspondences of the CTA's next eight problems (one contiguous 8 * n * 48-byte range) brought into a
// two-stage shared-memory buffer by a bulk asynchronous copy (TMA engine) while the current eight are processed: the three
// passes over the points (sums, distances, moments) read shared memory, and no warp waits for DRAM (the plain kernel
// spent most of its stall samples in `long_scoreboard`).  Packed input, n <= MOM_TMA_MAX_N.
#ifndef TVF_S1M_TMA
#define TVF_S1M_TMA 1
#endif
#ifndef TVF_S1M_TMA_MINB
#define TVF_S1M_TMA_MINB 6
#endif
constexpr int MOM_TMA_MAX_N = 64;
__global__ void __launch_bounds__(CORE_WARPS * 32, TVF_S1M_TMA_MINB)
tft_moments_tma_kernel(CoreInput in, double* __restrict__ ws) {
    __shared__ MomentsScratch scratch[CORE_WARPS];
    __shared__ unsigned long long bar[2];
    extern __shared__ __align__(16) unsigned char mom_dsm[];
    constexpr int PPG = 2 * CORE_WARPS;                    // problems per CTA iteration
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int h = lane >> 4, r = lane & 15;
    const unsigned prob_bytes = (unsigned)in.n * 48u, stage_bytes = PPG * prob_bytes;
    const long long ngroups = (in.B + PPG - 1) / PPG;
    auto issue = [&](long long g, int stage) {             // thread 0 only
        const long long left = in.B - g * PPG;
        const unsigned bytes = (unsigned)(left < PPG ? left : PPG) * prob_bytes;
        mbar_expect_tx(&bar[stage], bytes);
        bulk_g2s(mom_dsm + (size_t)stage * stage_bytes, in.p1 + g * PPG * in.n * 6, bytes, &bar[stage]);
    };
    if (threadIdx.x == 0) {
        mbar_init(&bar[0], 1); mbar_init(&bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0 && blockIdx.x < ngroups) issue(blockIdx.x, 0);
    int iter = 0;
    for (long long g = blockIdx.x; g < ngroups; g += gridDim.x, ++iter) {
        __syncthreads();                                   // every warp is done with the stage that is refilled now
        if (threadIdx.x == 0 && g + gridDim.x < ngroups) issue(g + gridDim.x, (iter + 1) & 1);
        mbar_wait(&bar[iter & 1], (unsigned)(iter >> 1) & 1u);
        CoreInput ins = in;
        ins.p1 = reinterpret_cast<const double*>(mom_dsm + (size_t)(iter & 1) * stage_bytes);
        const int lp = 2 * warp + h;
        const long long prob = g * PPG + lp;
        const bool live = prob < in.B;
        double acc[6], s[3], t[6];
        half_stats_moments<2>(ins, live ? lp : 0, r, scratch[warp].feat[h], acc, s, t);
        if (live) store_moments_stats(ws + prob * CORE_WS_TFT, r, acc, s, t);
    }
}

// warps per CTA of the two-problem solve kernel (the CTA barrier per pair keeps them on the same instruction-cache lines)
#ifndef TVF_S1D_WARPS
#define TVF_S1D_WARPS TVF_CORE_WARPS
#endif
constexpr int S1D_WARPS = TVF_S1D_WARPS;
// Large-n path, two problems per warp: the moments were produced by tft_moments_large_kernel.
__global__ void __launch_bounds__(S1D_WARPS * 32, TVF_S1D_MINB)
tft_stage1_solve_dual_kernel(long long B, double* __restrict__ ws, int* __restrict__ status) {
    __shared__ Stage1DualScratch scratch[S1D_WARPS];
    __shared__ unsigned char gidx[32 * 27];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    build_gidx(gidx);
    __syncthreads();
    Stage1DualScratch& sc = scratch[warp];
    const int h = lane >> 4, r = lane & 15;
    const long long npairs = (B + 1) / 2;
#if TVF_S1D_PREFETCH
    // The raw moments of the NEXT pair travel global -> shared (cp.async, no registers: the solver leaves none) while this
    // pair is solved; they land in the feature staging buffer, which the solve-only kernel does not use otherwise.
    double* raw = sc.feat[h];
    const long long stride = (long long)gridDim.x * S1D_WARPS;
    {
        const long long pair = (long long)blockIdx.x * S1D_WARPS + warp;
        if (pair < npairs) {
            const double* src = ws + min(2 * pair + h, B - 1) * CORE_WS_TFT + CW_MOM;
#pragma unroll
            for (int q = 0; q < 6; ++q) cp_async8(raw + q * 16 + r, src + q * 16 + r);
        }
        if (r < 4) sc.mom[h][96 + r] = 0.0;
    }
#endif
    for (long long base = (long long)blockIdx.x * S1D_WARPS; base < npairs; base += (long long)gridDim.x * S1D_WARPS) {
        S1D_SYNC();
        const long long pair = base + warp;
        if (pair >= npairs) continue;
        const bool live = 2 * pair + h < B;
        const long long prob = live ? 2 * pair + h : B - 1;
        double* rec = ws + prob * CORE_WS_TFT;
#if TVF_S1D_PREFETCH
        cp_async_wait_all();
        __syncwarp();
        // scaled table -> sc.mom (two barriers inside); afterwards nobody reads `raw` any more, so the next pair's copy may
        // start: each lane overwrites only the entries it read itself
        const double tr = gram_trace_from_moments(raw);
        const double scl = 1.0 / tr;
        const double delta = 1.0e-13 / 27.0;
        double m6[6];
#pragma unroll
        for (int q = 0; q < 6; ++q) m6[q] = raw[q * 16 + r];
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 6; ++q) sc.mom[h][q * 16 + r] = fma(m6[q], scl, is_diag_moment(q * 16 + r) ? delta : 0.0);
        if (pair + stride < npairs) {
            const double* src = ws + min(2 * (pair + stride) + h, B - 1) * CORE_WS_TFT + CW_MOM;
#pragma unroll
            for (int q = 0; q < 6; ++q) cp_async8(raw + q * 16 + r, src + q * 16 + r);
        }
        __syncwarp();
        solve_pair_scaled(sc, gidx, lane, live, rec, status, prob);
#else
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 6; ++q) sc.mom[h][q * 16 + r] = rec[CW_MOM + q * 16 + r];
        if (r < 4) sc.mom[h][96 + r] = 0.0;
        __syncwarp();
        solve_pair_from_moments(sc, gidx, lane, live, rec, status, prob, sc.mom[h]);
#endif
    }
}

// The second half of stage 1 on its own, one problem per warp (27 x 27 Gram from the 96 moments -> null vector).  The
// moments come from tft_moments_kernel (split stage 1) or from tft_moments_large_kernel (large n).  The unit-trace
// scaling and the diagonal shift are applied to the moment table (see solve_pair_from_moments).
#ifndef TVF_S1S_MINB
#define TVF_S1S_MINB 4
#endif
__global__ void __launch_bounds__(CORE_WARPS * 32, TVF_S1S_MINB)
tft_stage1_solve_kernel(long long B, double* __restrict__ ws, int* __restrict__ status) {
    __shared__ Stage1Scratch scratch[CORE_WARPS];
    __shared__ unsigned char gidx[32 * 27];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    build_gidx(gidx);
    __syncthreads();
    Stage1Scratch& sc = scratch[warp];
    const long long stride = (long long)gridDim.x * CORE_WARPS;
    long long prob = (long long)blockIdx.x * CORE_WARPS + warp;
    // the three moments of this lane for the NEXT problem are fetched while the current one is being solved
    double m0 = 0.0, m1 = 0.0, m2 = 0.0;
    if (prob < B) { const double* rec = ws + prob * CORE_WS_TFT; m0 = rec[CW_MOM + lane]; m1 = rec[CW_MOM + 32 + lane]; m2 = rec[CW_MOM + 64 + lane]; }
    for (long long base = (long long)blockIdx.x * CORE_WARPS; base < B; base += stride, prob += stride) {
        STEP_SYNC();
        if (prob >= B) continue;
        double* rec = ws + prob * CORE_WS_TFT;
        // trace = sum of the 12 diagonal moments with multiplicities 4, 2, 2, 1 (gram_trace_from_moments), as one reduction
        double part = 0.0;
        part += is_diag_moment(lane) ? diag_moment_weight(lane) * m0 : 0.0;
        part += is_diag_moment(lane + 32) ? diag_moment_weight(lane + 32) * m1 : 0.0;
        part += is_diag_moment(lane + 64) ? diag_moment_weight(lane + 64) * m2 : 0.0;
        const double scl = 1.0 / warp_sum(part);
        const double delta = 1.0e-13 / 27.0;
        __syncwarp();
        sc.mom[lane] = fma(m0, scl, is_diag_moment(lane) ? delta : 0.0);
        sc.mom[lane + 32] = fma(m1, scl, is_diag_moment(lane + 32) ? delta : 0.0);
        sc.mom[lane + 64] = fma(m2, scl, is_diag_moment(lane + 64) ? delta : 0.0);
        if (lane == 0) { sc.mom[96] = 0.0; sc.mom[97] = 0.0; }
        __syncwarp();
        if (prob + stride < B) {
            const double* nrec = ws + (prob + stride) * CORE_WS_TFT;
            m0 = nrec[CW_MOM + lane]; m1 = nrec[CW_MOM + 32 + lane]; m2 = nrec[CW_MOM + 64 + lane];
        }
        double g[27];
#pragma unroll
        for (int c = 0; c < 27; ++c) g[c] = sc.mom[gidx[lane * 27 + c]];
        bool conv;
        const double tl = smallest_eigvec_spd<27, NoRefine, true>(g, lane, sc.sbuf, &conv);
        if (lane < 27) rec[CW_T1 + lane] = tl;
        if (status != nullptr && lane == 0) status[prob] = conv ? 0 : ST_EIG_NOCONV;
    }
}

// Solve-only kernel with the row-and-column split layout (smallest_eigvec_spd_cs): TVF_S1_SOLVER = 3.
#ifndef TVF_S1C_MINB
#define TVF_S1C_MINB 4
#endif
__global__ void __launch_bounds__(CORE_WARPS * 32, TVF_S1C_MINB)
tft_stage1_solve_cs_kernel(long long B, double* __restrict__ ws, int* __restrict__ status) {
    __shared__ Stage1Scratch scratch[CORE_WARPS];
    __shared__ unsigned char gidx[32 * 27];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    build_gidx(gidx);
    __syncthreads();
    Stage1Scratch& sc = scratch[warp];
    const int h = lane >> 4, r = lane & 15;
    const int row0 = (r < 14) ? r : 31, row1 = (r < 13) ? r + 14 : 31;          // rows >= 27 gather the zero sentinel
    for (long long base = (long long)blockIdx.x * CORE_WARPS; base < B; base += (long long)gridDim.x * CORE_WARPS) {
        STEP_SYNC();
        const long long prob = base + warp;
        if (prob >= B) continue;
        double* rec = ws + prob * CORE_WS_TFT;
        const double m0 = rec[CW_MOM + lane], m1 = rec[CW_MOM + 32 + lane], m2 = rec[CW_MOM + 64 + lane];
        double part = 0.0;
        part += is_diag_moment(lane) ? diag_moment_weight(lane) * m0 : 0.0;
        part += is_diag_moment(lane + 32) ? diag_moment_weight(lane + 32) * m1 : 0.0;
        part += is_diag_moment(lane + 64) ? diag_moment_weight(lane + 64) * m2 : 0.0;
        const double scl = 1.0 / warp_sum(part);
        const double delta = 1.0e-13 / 27.0;
        __syncwarp();
        sc.mom[lane] = fma(m0, scl, is_diag_moment(lane) ? delta : 0.0);
        sc.mom[lane + 32] = fma(m1, scl, is_diag_moment(lane + 32) ? delta : 0.0);
        sc.mom[lane + 64] = fma(m2, scl, is_diag_moment(lane + 64) ? delta : 0.0);
        if (lane == 0) { sc.mom[96] = 0.0; sc.mom[97] = 0.0; }
        __syncwarp();
        double g0[14], g1[14];
#pragma unroll
        for (int c = 0; c < 14; ++c) {
            const int col = 14 * h + c;                     // column 27 (h = 1, c = 13) is padding
            const bool pad = (h == 1) && (c == 13);
            g0[c] = pad ? 0.0 : sc.mom[gidx[row0 * 27 + (pad ? 0 : col)]];
            g1[c] = pad ? 0.0 : sc.mom[gidx[row1 * 27 + (pad ? 0 : col)]];
        }
        double x0, x1;
        bool conv;
        smallest_eigvec_spd_cs<27>(g0, g1, lane, sc.sbuf, &x0, &x1, &conv);
        if (h == 0) {
            if (r < 14) rec[CW_T1 + r] = x0;
            if (r < 13) rec[CW_T1 + 14 + r] = x1;
        }
        if (status != nullptr && lane == 0) status[prob] = conv ? 0 : ST_EIG_NOCONV;
    }
}

// =========================================================================== TFT epipoles
#ifndef TVF_EPI_MINB
#define TVF_EPI_MINB 4
#endif
__global__ void __launch_bounds__(128, TVF_EPI_MINB)
tft_epipoles_kernel(double* __restrict__ ws, long long B) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double* rec = ws + b * CORE_WS_TFT;
    double T[27];
#pragma unroll
    for (int i = 0; i < 27; ++i) T[i] = rec[CW_T1 + i];
    double e21[3], e31[3];
    tft_epipoles(T, e21, e31);                                             // linearTFT.m:71-79
#pragma unroll
    for (int i = 0; i < 3; ++i) { rec[CW_EPI + i] = e21[i]; rec[CW_EPI + 3 + i] = e31[i]; }
}

// =========================================================================== TFT stage 2
// The projected Gram H = Up' G Up of linearTFT.m:84, straight from the 96 moments (DESIGN.md §3.4).  Column (i,a) of Up is
// e_i (x) vec(p_a q_a') with p_a in (e21, e21, e21, u1, u2) and q_a in (e31, v1, v2, e31, e31), the basis of range(E) per
// slice.  G = sum (p1 p1') (x) M(x3,y3) (x) M(x2,y2) and M = sum_g m4_g N_g with four constant N_g, so
//   H[(i,a),(i',b)] = sum_{beta,gamma} mom[16 sym6(i,i') + 4 beta + gamma] c_beta(q_a,q_b) c_gamma(p_a,p_b)
// with the quadratic forms c(p,q) = (p0 q0 + p1 q1, p0 q2 + p2 q0, p1 q2 + p2 q1, p2 q2) of the N_g.  The entry is symmetric in
// a <-> b and in i <-> i': 6 x 15 distinct values.  Lane r < 15 of the 16 calling lanes takes the pair {a,b} number r, forms
// its 6 values (96 + 24 multiply-adds: first over gamma, then over beta) and stores each at its (up to) 4 places in hs, the
// full 15 x 15 matrix with row stride H15_LD.  pb / qb: (e21, u1, u2) / (e31, v1, v2), 9 doubles each.
constexpr int H15_LD = 18;       // rows 16-byte aligned, and the row reads of 8 lanes hit 8 different bank quads
__device__ __forceinline__ void cforms(const double* p, const double* q, double* c) {
    c[0] = fma(p[0], q[0], p[1] * q[1]);
    c[1] = fma(p[0], q[2], p[2] * q[0]);
    c[2] = fma(p[1], q[2], p[2] * q[1]);
    c[3] = p[2] * q[2];
}
__device__ __forceinline__ void form_h15(const double* mom, const double* pb, const double* qb, int r, double* hs) {
    if (r >= 15) return;
    // pair r -> (a, b), a <= b: (0,0) (0,1) .. (0,4) (1,1) .. (1,4) (2,2) .. (2,4) (3,3) (3,4) (4,4)
    const int a = (int)((0x433222111100000ull >> (4 * r)) & 15), b = (int)((0x443432432143210ull >> (4 * r)) & 15);
    double cp[4], cq[4];
    cforms(pb + 3 * (a < 3 ? 0 : a - 2), pb + 3 * (b < 3 ? 0 : b - 2), cp);
    cforms(qb + 3 * (a < 3 ? a : 0), qb + 3 * (b < 3 ? b : 0), cq);
    double* hab = hs + H15_LD * a + b;      // (row a, column b) of a 5 x 5 block
    double* hba = hs + H15_LD * b + a;
#pragma unroll
    for (int al = 0; al < 6; ++al) {
        const int i = (al < 3) ? 0 : ((al < 5) ? 1 : 2), i2 = (al < 3) ? al : ((al < 5) ? al - 2 : 2);   // sym6(i,i2) = al
        const double* m = mom + 16 * al;
        double hv = 0.0;
#pragma unroll
        for (int be = 0; be < 4; ++be) {
            const double y = fma(m[4 * be], cp[0], fma(m[4 * be + 1], cp[1], fma(m[4 * be + 2], cp[2], m[4 * be + 3] * cp[3])));
            hv = fma(cq[be], y, hv);
        }
        const int o = 5 * H15_LD * i + 5 * i2, ot = 5 * H15_LD * i2 + 5 * i;
        hab[o] = hv; hba[o] = hv;
        if (i != i2) { hab[ot] = hv; hba[ot] = hv; }
    }
}
// row r of H (zeros for r >= 15, as the eigenvector solvers want them)
__device__ __forceinline__ void load_h15_row(const double* hs, int r, double (&g)[15]) {
    const double* row = hs + H15_LD * (r < 15 ? r : 0);
    const double2* row2 = reinterpret_cast<const double2*>(row);
#pragma unroll
    for (int m2 = 0; m2 < 7; ++m2) { const double2 v = row2[m2]; g[2 * m2] = v.x; g[2 * m2 + 1] = v.y; }
    g[14] = row[14];
    if (r >= 15) {
#pragma unroll
        for (int c = 0; c < 15; ++c) g[c] = 0.0;
    }
}

struct __align__(16) Stage2Scratch {
    double sbuf[64];
    double H[15 * H15_LD];           // Up' G Up
    double ax[64];                   // refinement: the 27-vector Up tp at [0, 27), A'A times it at [32, 59)
    double mom[96];
    double bas[18];                  // e21, u1, u2, e31, v1, v2
    double T[28];
    double tp[16];
    double Nm[28];                   // N1, inv(N2), inv(N3)
};

template <bool PACKED, bool REFINE>
__global__ void __launch_bounds__(CORE_WARPS * 32, REFINE ? 3 : CORE_MINB)
tft_stage2_kernel(CoreInput in, const double* __restrict__ ws, double* __restrict__ Tout,
                  double* __restrict__ P2out, double* __restrict__ P3out, int* __restrict__ status) {
    const int normalize = in.normalize;
    const long long B = in.B;
    __shared__ Stage2Scratch scratch[CORE_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    Stage2Scratch& sc = scratch[warp];
    const int jr = lane % 3, kr = (lane / 3) % 3, ir = (lane < 27) ? lane / 9 : 0;

    for (long long base = (long long)blockIdx.x * CORE_WARPS; base < B; base += (long long)gridDim.x * CORE_WARPS) {
        STEP_SYNC();
        const long long prob = base + warp;
        if (prob >= B) continue;
        const double* rec = ws + prob * CORE_WS_TFT;
        sc.mom[lane] = rec[CW_MOM + lane]; sc.mom[lane + 32] = rec[CW_MOM + 32 + lane]; sc.mom[lane + 64] = rec[CW_MOM + 64 + lane];
        const double e21[3] = {rec[CW_EPI], rec[CW_EPI + 1], rec[CW_EPI + 2]};
        const double e31[3] = {rec[CW_EPI + 3], rec[CW_EPI + 4], rec[CW_EPI + 5]};
        double u1[3], u2[3], v1[3], v2[3];
        onb3(e21, u1, u2);
        onb3(e31, v1, v2);
        // basis of range(E) per slice: B0=e21 e31', B1=e21 v1', B2=e21 v2', B3=u1 e31', B4=u2 e31'
        if (lane == 0) {
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                sc.bas[q] = e21[q]; sc.bas[3 + q] = u1[q]; sc.bas[6 + q] = u2[q];
                sc.bas[9 + q] = e31[q]; sc.bas[12 + q] = v1[q]; sc.bas[15 + q] = v2[q];
            }
        }
        __syncwarp();
        form_h15(sc.mom, sc.bas, sc.bas + 9, lane, sc.H);
        __syncwarp();
        // lane (i,a) owns row 5i+a of H; then its smallest eigenvector (linearTFT.m:84)
        double tl2;
        int st = 0;
        {
            const int ia = (lane < 15) ? lane / 5 : 0, aa = (lane < 15) ? lane % 5 : 0;
            double pa[3], qa[3];
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                pa[q] = (aa < 3) ? e21[q] : ((aa == 3) ? u1[q] : u2[q]);
                qa[q] = (aa == 1) ? v1[q] : ((aa == 2) ? v2[q] : e31[q]);
            }
            double g15[15];
            load_h15_row(sc.H, lane, g15);
            const double pe = sel3(e21, jr), pu1 = sel3(u1, jr), pu2 = sel3(u2, jr);
            const double qe = sel3(e31, kr), qv1 = sel3(v1, kr), qv2 = sel3(v2, kr);
            const double st_s[3] = {rec[CW_STATS], rec[CW_STATS + 1], rec[CW_STATS + 2]};
            const double st_t[6] = {rec[CW_STATS + 3], rec[CW_STATS + 4], rec[CW_STATS + 5], rec[CW_STATS + 6],
                                    rec[CW_STATS + 7], rec[CW_STATS + 8]};
            // Up' A'A Up tp from the design rows (refinement of the projected problem, small n only)
            auto resid15 = [&](const double* xs) {
                double a27 = 0.0;
                if (lane < 27) {
                    const double* tp = xs + 5 * ir;
                    a27 = pe * (qe * tp[0] + qv1 * tp[1] + qv2 * tp[2]) + qe * (pu1 * tp[3] + pu2 * tp[4]);
                }
                __syncwarp();
                if (lane < 27) sc.ax[lane] = a27;
                __syncwarp();
                const double g27 = tft_apply_AtA<PACKED>(in, prob, lane, st_s, st_t, sc.ax);
                __syncwarp();
                if (lane < 27) sc.ax[32 + lane] = g27;
                __syncwarp();
                double r = 0.0;
#pragma unroll
                for (int k = 0; k < 3; ++k)
#pragma unroll
                    for (int j = 0; j < 3; ++j) r = fma(pa[j] * qa[k], sc.ax[32 + 9 * ia + 3 * k + j], r);
                return (lane < 15) ? r : 0.0;
            };
            bool conv2;
            double tpl;
            if constexpr (REFINE) tpl = smallest_eigvec_spd<15>(g15, lane, sc.sbuf, &conv2, resid15, 1);
            else tpl = smallest_eigvec_spd<15>(g15, lane, sc.sbuf, &conv2);
            if (!conv2) st |= ST_EIG_NOCONV;
            __syncwarp();
            if (lane < 15) sc.tp[lane] = tpl;
            __syncwarp();
            double acc = 0.0;                                                   // t = Up*tp  (linearTFT.m:85)
            if (lane < 27) {
                const double* tp = sc.tp + 5 * ir;
                acc = pe * (qe * tp[0] + qv1 * tp[1] + qv2 * tp[2]) + qe * (pu1 * tp[3] + pu2 * tp[4]);
            }
            tl2 = acc * rsqrt_(warp_sum(acc * acc));
        }
        if (lane < 27) sc.T[lane] = tl2;
        __syncwarp();

        // ---- P2, P3 (linearTFT.m:86-90): a = pinv(E) t in closed form --------------------
        if (P2out != nullptr && P3out != nullptr) {
            if (lane < 3) {
                const double* Ti = sc.T + 9 * lane;
                double a[3], b[3];
                mat3_vec(Ti, e31, a);
                mat3_tvec(Ti, e21, b);
                const double tau = e21[0] * a[0] + e21[1] * a[1] + e21[2] * a[2];
#pragma unroll
                for (int q = 0; q < 3; ++q) {
                    P2out[prob * 12 + 3 * lane + q] = a[q] - 0.5 * tau * e21[q];
                    P3out[prob * 12 + 3 * lane + q] = 0.5 * tau * e31[q] - b[q];
                }
            } else if (lane == 3) {
#pragma unroll
                for (int q = 0; q < 3; ++q) { P2out[prob * 12 + 9 + q] = e21[q]; P3out[prob * 12 + 9 + q] = e31[q]; }
            }
        }

        // ---- undo the normalisation (LinearTFTPoseEstimation.m:53 -> transform_TFT.m:43-49) ------
        double tout = tl2;
        if (normalize) {
            const double s0 = rec[CW_STATS], s1 = rec[CW_STATS + 1], s2 = rec[CW_STATS + 2];
            const double N1[9] = {s0, 0, 0, 0, s0, 0, rec[CW_STATS + 3], rec[CW_STATS + 4], 1.0};
            const double N2[9] = {s1, 0, 0, 0, s1, 0, rec[CW_STATS + 5], rec[CW_STATS + 6], 1.0};
            const double N3[9] = {s2, 0, 0, 0, s2, 0, rec[CW_STATS + 7], rec[CW_STATS + 8], 1.0};
            double N2i[9], N3i[9];
            inv3(N2, N2i); inv3(N3, N3i);
            if (lane == 0) {
#pragma unroll
                for (int q = 0; q < 9; ++q) { sc.Nm[q] = N1[q]; sc.Nm[9 + q] = N2i[q]; sc.Nm[18 + q] = N3i[q]; }
            }
            __syncwarp();
            double acc = 0.0;
            if (lane < 27) {
#pragma unroll
                for (int b = 0; b < 3; ++b)
#pragma unroll
                    for (int a = 0; a < 3; ++a) {
                        const double sab = sc.Nm[3 * ir] * sc.T[a + 3 * b] + sc.Nm[1 + 3 * ir] * sc.T[9 + a + 3 * b] +
                                           sc.Nm[2 + 3 * ir] * sc.T[18 + a + 3 * b];
                        acc = fma(sc.Nm[9 + jr + 3 * a] * sc.Nm[18 + kr + 3 * b], sab, acc);
                    }
            }
            tout = acc * rsqrt_(warp_sum(acc * acc));                                         // :49
        }
        if (lane < 27) Tout[prob * 27 + lane] = tout;
        if (status != nullptr && lane == 0 && st != 0) status[prob] |= st;
    }
}

// ---- two problems per warp (n >= REFINE_N_MAX), one per half-warp from the staged record to the last store: half h = problem
// 2 pair + h forms its H (form_h15 on its 16 lanes), solves it (smallest_eigvec_spd_half) and runs the back end with two
// entries of T per lane.
// The pair's two work-space records are adjacent in global memory (2 x 1120 bytes): lane 0 fetches the NEXT pair's with one
// bulk asynchronous copy per warp (own mbarrier) as soon as the current pair's moments have been consumed (the epipoles
// and statistics are copied aside first), so no pair waits for its loads.
#ifndef TVF_S2_TMA
#define TVF_S2_TMA 1
#endif
struct __align__(16) Stage2DualScratch {
    double sbuf[64];
    double H[2][15 * H15_LD];            // Up' G Up of the two problems
#if TVF_S2_TMA
    double rec2[2 * CORE_WS_TFT];        // the two work-space records as they lie in global memory (one bulk copy)
#else
    double mom2[2][96];                  // moments of the two problems
#endif
    double es[2][28];                    // e21, u1, u2 (0..8), e31, v1, v2 (9..17), normalisation statistics (18..26)
    double T[2][28];
    double tp[2][16];
};

#ifndef TVF_STAGE2_DUAL
#define TVF_STAGE2_DUAL 1
#endif

// resident CTAs per SM the kernel is compiled for: 5 (96 registers, 12 bytes spilled) measured 14.7 ms per 10 M against 15.1 at 4
// (128 registers, 4 bytes spilled) and 16.2 at 3 (profiles/r03_stage2_factored_h.md)
#ifndef TVF_S2D_MINB
#define TVF_S2D_MINB 5
#endif
__global__ void __launch_bounds__(CORE_WARPS * 32, TVF_S2D_MINB)
tft_stage2_dual_kernel(int normalize, long long B, const double* __restrict__ ws, double* __restrict__ Tout,
                       double* __restrict__ P2out, double* __restrict__ P3out, int* __restrict__ status) {
    __shared__ Stage2DualScratch scratch[CORE_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    Stage2DualScratch& sc = scratch[warp];
    const int h = lane >> 4, r15 = lane & 15;
    // entries e0 = r15 and e1 = r15 + 16 of T (index j + 3k + 9i); e1 exists for r15 < 11 (the clamped index is never stored)
    const bool has1 = r15 < 11;
    const int e0 = r15, e1 = has1 ? r15 + 16 : 26;
    const long long npairs = (B + 1) / 2;
#if TVF_S2_TMA
    __shared__ unsigned long long wbar[CORE_WARPS];
    const long long pstride = (long long)gridDim.x * CORE_WARPS;
    auto fetch = [&](long long pr) {                        // lane 0 only: records of pair pr -> sc.rec2
        const unsigned bytes = (2 * pr + 1 < B ? 2u : 1u) * (unsigned)(CORE_WS_TFT * 8);
        mbar_expect_tx(&wbar[warp], bytes);
        bulk_g2s(sc.rec2, ws + 2 * pr * CORE_WS_TFT, bytes, &wbar[warp]);
    };
    if (lane == 0) mbar_init(&wbar[warp], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();
    if (lane == 0 && (long long)blockIdx.x * CORE_WARPS + warp < npairs) fetch((long long)blockIdx.x * CORE_WARPS + warp);
    unsigned parity = 0;
#endif

    for (long long base = (long long)blockIdx.x * CORE_WARPS; base < npairs; base += (long long)gridDim.x * CORE_WARPS) {
        S2_SYNC();
        const long long pair = base + warp;
        if (pair >= npairs) continue;
        const long long prob0 = 2 * pair;
        const int nprob = (prob0 + 1 < B) ? 2 : 1;
        const bool live = h < nprob;            // odd batch: the idle half works on problem prob0 and stores nothing
        const int hp = live ? h : 0;
        // lane 16 p + q: epipoles (q < 6) and normalisation statistics (6 <= q < 15) of problem p, set aside
        const int es_slot = (r15 < 3) ? r15 : ((r15 < 6) ? r15 + 6 : r15 + 12);
#if TVF_S2_TMA
        mbar_wait(&wbar[warp], parity);
        parity ^= 1u;
        const double* mom = sc.rec2 + hp * CORE_WS_TFT + CW_MOM;
        {
            const double* recq = sc.rec2 + hp * CORE_WS_TFT;
            if (r15 < 15) sc.es[h][es_slot] = (r15 < 6) ? recq[CW_EPI + r15] : recq[CW_STATS + r15 - 6];
        }
#else
        // every global load of the pair is issued up front (moments, epipoles, normalisation statistics): one exposed memory
        // latency per pair
        const double* mom = sc.mom2[hp];
        {
            double mm[2][3];
#pragma unroll
            for (int p = 0; p < 2; ++p) {
                const double* rec = ws + (prob0 + ((p < nprob) ? p : 0)) * CORE_WS_TFT;
                mm[p][0] = rec[CW_MOM + lane]; mm[p][1] = rec[CW_MOM + 32 + lane]; mm[p][2] = rec[CW_MOM + 64 + lane];
            }
            const double* recq = ws + (prob0 + hp) * CORE_WS_TFT;
            const double ev = (r15 < 6) ? recq[CW_EPI + r15] : ((r15 < 15) ? recq[CW_STATS + r15 - 6] : 0.0);
#pragma unroll
            for (int p = 0; p < 2; ++p) {
                sc.mom2[p][lane] = mm[p][0]; sc.mom2[p][lane + 32] = mm[p][1]; sc.mom2[p][lane + 64] = mm[p][2];
            }
            if (r15 < 15) sc.es[h][es_slot] = ev;
        }
#endif
        __syncwarp();
        {
            // orthonormal completions, once per problem: lane 0 of the half -> u1, u2; lane 1 -> v1, v2
            double* e = sc.es[h] + 9 * (r15 & 1);
            double u1[3], u2[3];
            onb3(e, u1, u2);
            if (r15 < 2) {
#pragma unroll
                for (int q = 0; q < 3; ++q) { e[3 + q] = u1[q]; e[6 + q] = u2[q]; }
            }
            __syncwarp();
        }
        const double* bh = sc.es[h];
        form_h15(mom, bh, bh + 9, r15, sc.H[h]);
        __syncwarp();
#if TVF_S2_TMA
        if (lane == 0 && pair + pstride < npairs) fetch(pair + pstride);       // every lane is done with sc.rec2
#endif
        // ---- the smallest eigenvector of H (linearTFT.m:84), both problems at once
        {
            double g15[15];
            load_h15_row(sc.H[h], r15, g15);
            if (!live) {                                   // odd batch: the idle half solves the identity
#pragma unroll
                for (int c = 0; c < 15; ++c) g15[c] = (c == r15) ? 1.0 : 0.0;
            }
            bool conv2;
            const double tpl = smallest_eigvec_spd_half<15>(g15, lane, sc.sbuf, &conv2);
            __syncwarp();
            if (r15 < 15) sc.tp[h][r15] = tpl;
            if (live && !conv2 && r15 == 0 && status != nullptr) status[prob0 + h] |= ST_EIG_NOCONV;
        }
        __syncwarp();
        // ---- back end, both problems at once: t = Up*tp, P2/P3, undo the normalisation
        const long long prob = prob0 + h;
        const double* tp = sc.tp[h];
        auto up_tp = [&](int e) {                                               // t = Up*tp  (linearTFT.m:85)
            const int j = e % 3, k = (e / 3) % 3, i = e / 9;
            const double pe = bh[j], pu1 = bh[3 + j], pu2 = bh[6 + j], qe = bh[9 + k], qv1 = bh[12 + k], qv2 = bh[15 + k];
            const double* t5 = tp + 5 * i;
            return pe * (qe * t5[0] + qv1 * t5[1] + qv2 * t5[2]) + qe * (pu1 * t5[3] + pu2 * t5[4]);
        };
        double t0 = up_tp(e0), t1 = has1 ? up_tp(e1) : 0.0;
        {
            const double nrm = rsqrt_(half_sum(fma(t0, t0, t1 * t1)));
            t0 *= nrm; t1 *= nrm;
        }
        double* Th = sc.T[h];
        Th[e0] = t0;
        if (has1) Th[e1] = t1;
        __syncwarp();
        if (live && P2out != nullptr && P3out != nullptr) {                      // linearTFT.m:86-90, a = pinv(E) t in closed form
            const double* e21 = bh;
            const double* e31 = bh + 9;
            if (r15 < 3) {
                const double* Ti = Th + 9 * r15;
                double a[3], b[3];
                mat3_vec(Ti, e31, a);
                mat3_tvec(Ti, e21, b);
                const double tau = e21[0] * a[0] + e21[1] * a[1] + e21[2] * a[2];
#pragma unroll
                for (int q = 0; q < 3; ++q) {
                    P2out[prob * 12 + 3 * r15 + q] = a[q] - 0.5 * tau * e21[q];
                    P3out[prob * 12 + 3 * r15 + q] = 0.5 * tau * e31[q] - b[q];
                }
            } else if (r15 == 3) {
#pragma unroll
                for (int q = 0; q < 3; ++q) { P2out[prob * 12 + 9 + q] = e21[q]; P3out[prob * 12 + 9 + q] = e31[q]; }
            }
        }
        if (normalize) {
            // LinearTFTPoseEstimation.m:53 -> transform_TFT.m:43-49 with the three Normalize2Ddata matrices
            // N_v = [s 0 tx; 0 s ty; 0 0 1]: T_new(:,:,i) = inv(N2) * (sum_r N1(r,i) T(:,:,r)) * inv(N3).'.  The matrices
            // are similarities, so the sum over r has at most three terms, inv(N) = [1/s 0 -tx/s; 0 1/s -ty/s; 0 0 1] is
            // known in closed form, and element (j,k) of the product touches rows {j, 2} and columns {k, 2} only.
            const double* st9p = bh + 18;
            const double s1 = st9p[0], i2 = rcp_(st9p[1]), i3 = rcp_(st9p[2]);
            const double t1x = st9p[3], t1y = st9p[4];
            auto unnorm = [&](int e) {
                const int jr = e % 3, kr = (e / 3) % 3, ir = e / 9;
                // row j of inv(N2): (a2, .., b2): out(j,:) = a2 * S(j,:) + b2 * S(2,:)   (j = 2: a2 = 1, b2 = 0)
                const double a2 = (jr == 2) ? 1.0 : i2, b2 = (jr == 0) ? -st9p[5] * i2 : ((jr == 1) ? -st9p[6] * i2 : 0.0);
                const double a3 = (kr == 2) ? 1.0 : i3, b3 = (kr == 0) ? -st9p[7] * i3 : ((kr == 1) ? -st9p[8] * i3 : 0.0);
                // S(j',k') of slice i: i = 0,1: s1 * T_i;  i = 2: t1x T_0 + t1y T_1 + T_2
                auto S = [&](int jj, int kk) -> double {
                    const int x = jj + 3 * kk;
                    if (ir == 2) return fma(t1x, Th[x], fma(t1y, Th[9 + x], Th[18 + x]));
                    return s1 * Th[9 * ir + x];
                };
                const double sjk = S(jr, kr), s2k = S(2, kr), sj2 = S(jr, 2), s22 = S(2, 2);
                // out(j,k) = sum_{j',k'} inv2(j,j') S(j',k') inv3(k,k') over j' in {j,2}, k' in {k,2}
                return a3 * (a2 * sjk + b2 * s2k) + b3 * (a2 * sj2 + b2 * s22);
            };
            t0 = unnorm(e0); t1 = has1 ? unnorm(e1) : 0.0;
            const double nrm = rsqrt_(half_sum(fma(t0, t0, t1 * t1)));                // :49
            t0 *= nrm; t1 *= nrm;
        }
        if (live) {
            Tout[prob * 27 + e0] = t0;
            if (has1) Tout[prob * 27 + e1] = t1;
        }
        __syncwarp();                                                            // sc.es, sc.T are reused by the next pair
    }
}

// =========================================================================== linearF stage 1
struct __align__(16) FScratch {
    double sbuf[64];
    double feat[32 * FEAT_STRIDE];
    double mom[2][40];               // 36 moments of the view pairs (1,2) and (1,3)
};

// mode: in.normalize != 0 -> pose path (two pairs 1-2 and 1-3, outer normalisation); else one pair
template <bool PACKED, bool REFINE>
__global__ void __launch_bounds__(CORE_WARPS * 32, REFINE ? 3 : CORE_MINB)
f_stage1_kernel(CoreInput in, double* __restrict__ ws, int* __restrict__ status) {
    __shared__ FScratch scratch[CORE_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    FScratch& sc = scratch[warp];
    // 36 moments: lane l -> (alpha,beta) = (l/6, l%6); lanes 0..3 also take moment 32+l
    const int m1 = 32 + lane;
    const int a0 = lane / 6, b0 = lane % 6, a1 = (m1 < 36) ? m1 / 6 : 0, b1 = (m1 < 36) ? m1 % 6 : 0;
    const int ar = (lane < 9) ? lane / 3 : 0, br = (lane < 9) ? lane % 3 : 0;

    for (long long base = (long long)blockIdx.x * CORE_WARPS; base < in.B; base += (long long)gridDim.x * CORE_WARPS) {
        STEP_SYNC();
        const long long prob = base + warp;
        if (prob >= in.B) continue;
        double* rec = ws + prob * CORE_WS_F;
        const double one3[3] = {1.0, 1.0, 1.0}, zero6[6] = {0, 0, 0, 0, 0, 0};
        double s0[3] = {1.0, 1.0, 1.0}, t0[6] = {0, 0, 0, 0, 0, 0};
        if (in.normalize) view_stats<PACKED>(in, prob, lane, one3, zero6, s0, t0);   // LinearFPoseEstimation.m:46-48
        double si[3], ti[6];
        view_stats<PACKED>(in, prob, lane, s0, t0, si, ti);                          // linearF.m:45-46
        int st = 0;
        const int npairs = in.normalize ? 2 : 1;
        for (int pr = 0; pr < npairs; ++pr) {
            const int vb = 1 + pr;
            // inner map composed with the outer one: x' = si*(s0*x + t0) + ti
            const double sa = si[0] * s0[0], sb = sel3(si, vb) * sel3(s0, vb);
            const double tax = si[0] * t0[0] + ti[0], tay = si[0] * t0[1] + ti[1];
            const double tbx = sel3(si, vb) * (vb == 1 ? t0[2] : t0[4]) + (vb == 1 ? ti[2] : ti[4]);
            const double tby = sel3(si, vb) * (vb == 1 ? t0[3] : t0[5]) + (vb == 1 ? ti[3] : ti[5]);
            double acc0 = 0.0, acc1 = 0.0;
            for (int pbase = 0; pbase < in.n; pbase += 32) {
                const int cnt = min(32, in.n - pbase);
                __syncwarp();
                if (lane < cnt) {
                    double p[6];
                    load_point<PACKED>(in, prob, pbase + lane, p);
                    const double xb = (vb == 1) ? p[2] : p[4], yb = (vb == 1) ? p[3] : p[5];
                    const double x1 = sa * p[0] + tax, y1 = sa * p[1] + tay;
                    const double x2 = sb * xb + tbx, y2 = sb * yb + tby;
                    double* f = sc.feat + lane * FEAT_STRIDE;
                    f[0] = x1 * x1; f[1] = x1 * y1; f[2] = x1; f[3] = y1 * y1; f[4] = y1; f[5] = 1.0;
                    f[6] = x2 * x2; f[7] = x2 * y2; f[8] = x2; f[9] = y2 * y2; f[10] = y2; f[11] = 1.0;
                }
                __syncwarp();
                for (int p = 0; p < cnt; ++p) {
                    const double* f = sc.feat + p * FEAT_STRIDE;
                    acc0 = fma(f[a0], f[6 + b0], acc0);
                    acc1 = fma(f[a1], f[6 + b1], acc1);
                }
            }
            __syncwarp();
            sc.mom[pr][lane] = acc0;
            if (lane < 4) sc.mom[pr][32 + lane] = acc1;
            __syncwarp();
            if constexpr (REFINE) {
                // G9(r,c), r = 3*a + b for the row [x1x2, x1y2, x1, y1x2, y1y2, y1, x2, y2, 1] (linearF.m:51-52)
                double g[9];
#pragma unroll
                for (int c = 0; c < 9; ++c) {
                    const double v = sc.mom[pr][c_sym6[ar * 3 + c / 3] * 6 + c_sym6[br * 3 + c % 3]];
                    g[c] = (lane < 9) ? v : 0.0;
                }
                bool conv;                                                                 // linearF.m:54-55
                const double fl = smallest_eigvec_spd<9>(g, lane, sc.sbuf, &conv, [&](const double* xs) {
                    return f_apply_AtA<PACKED>(in, prob, lane, vb, sa, tax, tay, sb, tbx, tby, xs); }, 2);
                if (!conv) st |= ST_EIG_NOCONV;
                if (lane < 9) rec[FW_F + 9 * pr + lane] = fl;
            }
        }
        if constexpr (!REFINE) {
            // both 9x9 systems at once, one per half-warp (half 1 solves the identity when there is a single pair)
            const int h = lane >> 4, r = lane & 15;
            const int arh = (r < 9) ? r / 3 : 0, brh = (r < 9) ? r % 3 : 0;
            const bool live = h < npairs && r < 9;
            double g[9];
#pragma unroll
            for (int c = 0; c < 9; ++c) {
                const double v = sc.mom[h < npairs ? h : 0][c_sym6[arh * 3 + c / 3] * 6 + c_sym6[brh * 3 + c % 3]];
                g[c] = live ? v : ((h >= npairs && c == r) ? 1.0 : 0.0);
            }
            bool conv;                                                                     // linearF.m:54-55
            const double fl = smallest_eigvec_spd_half<9>(g, lane, sc.sbuf, &conv);
            if (h < npairs && !conv) st |= ST_EIG_NOCONV;
            st |= __shfl_xor_sync(0xffffffffu, st, 16);                                    // lane 0 reports both halves
            if (live) rec[FW_F + 9 * h + r] = fl;
        }
        if (lane < 3) { rec[FW_STATS + lane] = sel3(s0, lane); rec[FW_STATS + 9 + lane] = sel3(si, lane); }
        if (lane < 6) {
            rec[FW_STATS + 3 + lane] = (lane < 3) ? sel3(t0, lane) : sel3(t0 + 3, lane - 3);
            rec[FW_STATS + 12 + lane] = (lane < 3) ? sel3(ti, lane) : sel3(ti + 3, lane - 3);
        }
        if (status != nullptr && lane == 0) status[prob] = st;
    }
}

// linearF.m:58-62 and LinearFPoseEstimation.m:55-56, one thread per problem
__global__ void __launch_bounds__(128)
f_finish_kernel(const double* __restrict__ ws, int normalize, long long B, double* __restrict__ Fout) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const double* rec = ws + b * CORE_WS_F;
    const double* s0 = rec + FW_STATS; const double* t0 = s0 + 3; const double* si = s0 + 9; const double* ti = s0 + 12;
    const int npairs = normalize ? 2 : 1;
    for (int pr = 0; pr < npairs; ++pr) {
        const int vb = 1 + pr;
        double Fv[9];
#pragma unroll
        for (int q = 0; q < 9; ++q) Fv[q] = rec[FW_F + 9 * pr + q];                       // reshape(V(:,9),3,3)
        const double Na[9] = {si[0], 0, 0, 0, si[0], 0, ti[0], ti[1], 1.0};
        const double Nb[9] = {si[vb], 0, 0, 0, si[vb], 0, ti[2 * vb], ti[2 * vb + 1], 1.0};
        double tmp[9], Fu[9], F[9];
        mat3_mul_tn(Nb, Fv, tmp);
        mat3_mul(tmp, Na, Fu);                                                            // linearF.m:58
        double U[9], sv[3], V[9];
        svd3_full(Fu, U, sv, V);                                                          // :61, D(3,3)=0
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int r = 0; r < 3; ++r) F[r + 3 * c] = sv[0] * U[r] * V[c] + sv[1] * U[3 + r] * V[3 + c];   // :62
        if (normalize) {                                                                  // LinearFPoseEstimation.m:55-56
            const double Ma[9] = {s0[0], 0, 0, 0, s0[0], 0, t0[0], t0[1], 1.0};
            const double Mb[9] = {s0[vb], 0, 0, 0, s0[vb], 0, t0[2 * vb], t0[2 * vb + 1], 1.0};
            mat3_mul_tn(Mb, F, tmp);
            mat3_mul(tmp, Ma, F);
        }
#pragma unroll
        for (int q = 0; q < 9; ++q) Fout[b * (9 * npairs) + 9 * pr + q] = F[q];
    }
}

// ---------------------------------------------------------------------------
static inline unsigned core_grid(long long B, int sm_count) {
    long long blocks = (B + CORE_WARPS - 1) / CORE_WARPS;
    const long long cap = (long long)sm_count * CORE_MINB * 4;
    if (blocks > cap) blocks = cap;
    return (unsigned)(blocks < 1 ? 1 : blocks);
}

static inline unsigned core_grid_minb(long long units, int sm_count, int minb) {
    long long blocks = (units + CORE_WARPS - 1) / CORE_WARPS;
    const long long cap = (long long)sm_count * minb * 4;
    if (blocks > cap) blocks = cap;
    return (unsigned)(blocks < 1 ? 1 : blocks);
}

int launch_tft_stage1(const CoreInput& in, double* ws, int* status, int sm_count, cudaStream_t stream) {
    if (in.B <= 0) return 0;
    const unsigned g = core_grid(in.B, sm_count);
    const bool refine = in.n < REFINE_N_MAX;       // barely determined systems: polish with the un-squared rows
#if TVF_STAGE1_DUAL
    if (!refine) {
#if TVF_STAGE1_SPLIT
        const unsigned gm = core_grid_minb((in.B + 1) / 2, sm_count, TVF_S1M_MINB);
#if TVF_S1M_TMA
        if (in.packed && in.n <= MOM_TMA_MAX_N) {
            const size_t dyn = 2 * (size_t)(2 * CORE_WARPS) * in.n * 48;
            cudaFuncSetAttribute(tft_moments_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);   // per launch: per device
            const unsigned gt = core_grid_minb((in.B + 1) / 2, sm_count, TVF_S1M_TMA_MINB);
            tft_moments_tma_kernel<<<gt, CORE_WARPS * 32, dyn, stream>>>(in, ws);
            return 1;
        }
#endif
        if (in.packed) tft_moments_kernel<true><<<gm, CORE_WARPS * 32, 0, stream>>>(in, ws);
        else tft_moments_kernel<false><<<gm, CORE_WARPS * 32, 0, stream>>>(in, ws);
        return 1;                 // the caller follows up with launch_tft_stage1_solve
#else
        const unsigned gd = core_grid_minb((in.B + 1) / 2, sm_count, TVF_S1D_MINB);
        if (in.packed) tft_stage1_dual_kernel<true><<<gd, CORE_WARPS * 32, 0, stream>>>(in, ws, status);
        else tft_stage1_dual_kernel<false><<<gd, CORE_WARPS * 32, 0, stream>>>(in, ws, status);
        return 0;
#endif
    }
#endif
    if (in.packed && refine) tft_stage1_kernel<true, true><<<g, CORE_WARPS * 32, 0, stream>>>(in, ws, status);
    else if (in.packed) tft_stage1_kernel<true, false><<<g, CORE_WARPS * 32, 0, stream>>>(in, ws, status);
    else if (refine) tft_stage1_kernel<false, true><<<g, CORE_WARPS * 32, 0, stream>>>(in, ws, status);
    else tft_stage1_kernel<false, false><<<g, CORE_WARPS * 32, 0, stream>>>(in, ws, status);
    return 0;
}

void launch_tft_stage1_solve(long long B, double* ws, int* status, int sm_count, cudaStream_t stream) {
    if (B <= 0) return;
#if TVF_S1_SOLVER == 2
    {
        long long blocks = ((B + 1) / 2 + S1D_WARPS - 1) / S1D_WARPS;
        const long long cap = (long long)sm_count * TVF_S1D_MINB * 4;
        if (blocks > cap) blocks = cap;
        tft_stage1_solve_dual_kernel<<<(unsigned)(blocks < 1 ? 1 : blocks), S1D_WARPS * 32, 0, stream>>>(B, ws, status);
    }
#elif TVF_S1_SOLVER == 3
    tft_stage1_solve_cs_kernel<<<core_grid_minb(B, sm_count, TVF_S1C_MINB), CORE_WARPS * 32, 0, stream>>>(B, ws, status);
#else
    tft_stage1_solve_kernel<<<core_grid_minb(B, sm_count, TVF_S1S_MINB), CORE_WARPS * 32, 0, stream>>>(B, ws, status);
#endif
}

void launch_tft_epipoles(double* ws, long long B, cudaStream_t stream) {
    if (B <= 0) return;
    tft_epipoles_kernel<<<(unsigned)((B + 127) / 128), 128, 0, stream>>>(ws, B);
}

void launch_tft_stage2(const CoreInput& in, const double* ws, double* T, double* P2, double* P3, int* status,
                       int sm_count, cudaStream_t stream) {
    if (in.B <= 0) return;
    const unsigned g = core_grid(in.B, sm_count);
    const bool refine = in.n < REFINE_N_MAX;
#if TVF_STAGE2_DUAL
    if (!refine) {          // the un-refined step never touches the points again: two problems per warp
        tft_stage2_dual_kernel<<<core_grid_minb((in.B + 1) / 2, sm_count, TVF_S2D_MINB), CORE_WARPS * 32, 0, stream>>>(in.normalize, in.B, ws, T, P2, P3, status);
        return;
    }
#endif
    if (in.packed && refine) tft_stage2_kernel<true, true><<<g, CORE_WARPS * 32, 0, stream>>>(in, ws, T, P2, P3, status);
    else if (in.packed) tft_stage2_kernel<true, false><<<g, CORE_WARPS * 32, 0, stream>>>(in, ws, T, P2, P3, status);
    else if (refine) tft_stage2_kernel<false, true><<<g, CORE_WARPS * 32, 0, stream>>>(in, ws, T, P2, P3, status);
    else tft_stage2_kernel<false, false><<<g, CORE_WARPS * 32, 0, stream>>>(in, ws, T, P2, P3, status);
}

void launch_f_stage1(const CoreInput& in, double* ws, int* status, int sm_count, cudaStream_t stream) {
    if (in.B <= 0) return;
    const unsigned g = core_grid(in.B, sm_count);
    const bool refine = in.n < REFINE_N_MAX;
    if (in.packed && refine) f_stage1_kernel<true, true><<<g, CORE_WARPS * 32, 0, stream>>>(in, ws, status);
    else if (in.packed) f_stage1_kernel<true, false><<<g, CORE_WARPS * 32, 0, stream>>>(in, ws, status);
    else if (refine) f_stage1_kernel<false, true><<<g, CORE_WARPS * 32, 0, stream>>>(in, ws, status);
    else f_stage1_kernel<false, false><<<g, CORE_WARPS * 32, 0, stream>>>(in, ws, status);
}

void launch_f_finish(const double* ws, int normalize, long long B, double* F, cudaStream_t stream) {
    if (B <= 0) return;
    f_finish_kernel<<<(unsigned)((B + 127) / 128), 128, 0, stream>>>(ws, normalize, B, F);
}

}  // namespace tvf
