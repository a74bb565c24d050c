// tvf_large_kernels.cu -- Gram formation for large-n triplets (BASELINE config 5: 10 000 correspondences
// per scene): the first half of linearTFT's stage 1 (Normalize2Ddata.m:33-39 x3 + the design-matrix Gram
// of linearTFT.m:45-64) as a bandwidth-oriented kernel.
//
// One thread-block CLUSTER of 8 CTAs owns a scene.  Each CTA pulls its contiguous slice of the scene
// (n/8 points x 48 B) from HBM into shared memory with ONE bulk asynchronous copy (TMA, cp.async.bulk ->
// SASS UBLKCP) that signals an mbarrier; three CTAs of different clusters share an SM, so one CTA's copy and
// cluster barriers overlap the arithmetic of the others, and a CTA issues the copy of its next slice the
// moment the last read of the current one has retired.  The scene is read from HBM exactly once.
//
// The reference's normalisation forces three dependent sweeps (mean -> mean distance -> moments of the
// normalised points).  Here there are two, both on the shared-memory copy: (1) coordinate sums -> centroid;
// (2) ONE fused sweep that accumulates the distance sums and the 96 moments of the CENTRED, unscaled points.
// Isotropic scaling multiplies every moment by an exact monomial s1^a s3^b s2^c, applied once per scene, so
// the scale is not needed inside the sweep and the squares x^2 + y^2 serve both the distances and m4.
// Only 6 + 99 partial sums per CTA cross the cluster through distributed shared memory (DSMEM), added in
// rank order (deterministic).
//
// Per point the arithmetic is ~160 FP64 issue slots (6 centring, 11 products, 95 accumulations split over two
// warp groups that each re-derive the shared products, 3 square roots at ~8, 6 for the centroid) against 48
// bytes.  B200 issues 64 FP64 lanes/clk/SM, so the FP64 pipe allows ~1.15e11 points/s = 5.5 TB/s: this
// kernel sits on the FP64/HBM ridge and is reported against both rooflines.  FP64 tensor cores do not help:
// DMMA and DFMA share one pipe on B200 (37.1 vs 36.5 TFLOP/s alone, 36 TFLOP/s combined when mixed --
// tools/microbench_fp64.cu, profiles/r01_microbench_fp64.json), and the Kronecker form needs 96 accumulations
// per point where a dense FP64 MMA on the 4x27 rows would need 5 832 (SURVEY.md App. B.3).
#include <cooperative_groups.h>

#include "tvf_kernels.h"
#include "tvf_warp.cuh"
#include "tvf_async.cuh"

namespace cg = cooperative_groups;

namespace tvf {

// TVF_LG_CLUSTER / TVF_LG_MINB: CTAs per scene / CTAs per SM the register budget is compiled for.  The shipping shape
// (8 x 128 threads, 3 per SM) is the measured optimum: profiles/r02_variants.md section 7 has 5 ... 10 CTAs per scene,
// 128- to 384-thread CTAs, chunked / early refill of the slice and per-warp exchanges, all slower.
#ifndef TVF_LG_CLUSTER
#define TVF_LG_CLUSTER 8
#endif
#ifndef TVF_LG_MINB
#define TVF_LG_MINB 3
#endif
constexpr int LG_CLUSTER = TVF_LG_CLUSTER;
constexpr int LG_THREADS = 128;
constexpr int LG_WARPS = LG_THREADS / 32;
constexpr int CW_MOM_L = 0, CW_STATS_L = 96;

// address of `local_smem_addr` in the shared memory of CTA `rank` of this cluster
__device__ __forceinline__ unsigned mapa_u32(unsigned local_smem_addr, unsigned rank) {
    unsigned r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(rank));
    return r;
}
// asynchronous remote store of one double into a peer CTA's shared memory; when the data has landed, 8 bytes are
// credited to the peer's mbarrier (same completion mechanism as the bulk copies).  No fence, no rendezvous.
__device__ __forceinline__ void st_async_f64(unsigned remote_addr, double v, unsigned remote_bar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.f64 [%0], %1, [%2];" ::"r"(remote_addr), "d"(v),
                 "r"(remote_bar)
                 : "memory");
}

__device__ __forceinline__ double warp_sum_l(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Transposed butterflies over per-lane partial sums v[OFF .. OFF+W): afterwards lane L holds the warp-wide
// total of v[OFF + (L mod W)] (returned).  W = 32: 31 shuffles; W = 16: 16 + 15 shuffles.
template <int OFF, int W, int NV>
__device__ __forceinline__ double warp_reduce_transposed(double (&v)[NV], int lane) {
    static_assert(W == 32 || W == 16, "W");
    if (W == 16) {
#pragma unroll
        for (int i = 0; i < 16; ++i) v[OFF + i] += __shfl_xor_sync(0xffffffffu, v[OFF + i], 16);
    }
#pragma unroll
    for (int half = W / 2; half >= 1; half >>= 1) {
        const bool hi = (lane & half) != 0;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            const double send = hi ? v[OFF + i] : v[OFF + i + half];
            const double keep = hi ? v[OFF + i + half] : v[OFF + i];
            v[OFF + i] = keep + __shfl_xor_sync(0xffffffffu, send, half);
        }
    }
    return v[OFF];
}

// sqrt(x) for x >= 0 without the ~15 FP64 issue slots of the IEEE sequence: MUFU.RSQ64H seed (relative error ~2^-20, it
// only looks at the high word), one Goldschmidt step (-> ~2^-39) and a residual correction (-> below 1 ulp; not
// correctly rounded).  The half reciprocal h is taken from the seed by an exponent decrement on
// the integer pipe and is NOT refined -- it only scales the last correction, whose own size is 2^-39 of the result, so
// its 2^-20 error enters at 2^-59: 5 FP64 issue slots instead of 7 (+1.4 % on the kernel).  x below 1e-300 (incl. 0)
// returns 0.
__device__ __forceinline__ double sqrt_fast(double x) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double h = __hiloint2double(__double2hiint(y) - 0x00100000, __double2loint(y));     // y / 2 (y is normal here)
    double g = x * y;
    const double r = fma(-g, h, 0.5);
    g = fma(g, r, g);
    const double d = fma(-g, g, x);
    g = fma(d, h, g);
    return (__double2hiint(x) > 0x01a00000) ? g : 0.0;      // x > ~1e-300 (x >= 0), without touching the FP64 pipe
}

// shared-memory layout (dynamic): [slice bytes] | Scratch
struct __align__(16) LargeScratch {
    unsigned long long bar_tma;     // bulk copy of the slice
    unsigned long long bar1[2];     // coordinate sums of all 8 ranks have landed in in1[parity]
    unsigned long long bar3;        // this CTA finalises the scene: the 8 x 99 sums have landed in in3
    double wpart1[LG_WARPS][8];     // per-warp partials, pass 1: 6 coordinate sums
    double wpart2[LG_WARPS][56];    // per-warp partials, pass 2: 48 moments + 2 distance sums
#if TVF_LARGE_DMMA
    double wpartD[LG_WARPS][100];   // tensor-core variant: per-warp partials of all 96 moments + 3 distance sums
#endif
    double in1[2][LG_CLUSTER][8];   // [scene parity][source rank][6 coordinate sums]   (written by st.async from every rank)
    double in3[LG_CLUSTER][104];    // [source rank][96 centred raw moments + 3 distance sums]
    double cen[2][8];               // cluster-wide centroids by scene parity
    double scl[4];                  // finalising CTA only: the three scales s_v
};

// The 48 sums one warp group owns: index k = alpha*8 + bl*4 + gamma with
//   alpha: view-1 feature [x^2, xy, x, y^2, y, 1], gamma: view-2 feature [1, x, y, x^2+y^2],
//   bl: view-3 feature, group 0 -> [1, x], group 1 -> [y, x^2+y^2]   (global beta = 2*G + bl),
// all in CENTRED, UNSCALED coordinates and without the minus signs of m4 = [1,-x,-y,r]: isotropic scaling
// and the signs are exact per-moment factors applied once per scene (see the epilogue), so the fused pass
// needs the centroid only and computes the distance sums of Normalize2Ddata.m:35 from the same squares.
template <int G>
__device__ __forceinline__ void moments_pass(const double* __restrict__ pts, int npts, int first, const double (&cen)[6],
                                             double (&acc)[48], double (&ds)[2]) {
    int i = first;
    if (i >= npts) return;
    double2 a, b, c;
    {
        const double2* q = reinterpret_cast<const double2*>(pts + 6 * i);
        a = q[0]; b = q[1]; c = q[2];
    }
    while (true) {
        const int nx = i + 64;
        const bool more = nx < npts;
        double2 na = a, nb = b, nc = c;
        if (more) {                                        // next point's coordinates are in flight during this point's FMAs
            const double2* q = reinterpret_cast<const double2*>(pts + 6 * nx);
            na = q[0]; nb = q[1]; nc = q[2];
        }
        const double x1 = a.x - cen[0], y1 = a.y - cen[1];
        const double x2 = b.x - cen[2], y2 = b.y - cen[3];
        const double x3 = c.x - cen[4], y3 = c.y - cen[5];
        const double xx = x1 * x1, xy = x1 * y1, yy = y1 * y1;
        const double r2 = fma(x2, x2, y2 * y2);
        double u0[4], u1[4];
        if (G == 0) {
            u0[0] = 1.0; u0[1] = x2; u0[2] = y2; u0[3] = r2;
            u1[0] = x3; u1[1] = x3 * x2; u1[2] = x3 * y2; u1[3] = x3 * r2;
            ds[0] += sqrt_fast(xx + yy);
            ds[1] += sqrt_fast(r2);
        } else {
            const double r3 = fma(x3, x3, y3 * y3);
            u0[0] = y3; u0[1] = y3 * x2; u0[2] = y3 * y2; u0[3] = y3 * r2;
            u1[0] = r3; u1[1] = r3 * x2; u1[2] = r3 * y2; u1[3] = r3 * r2;
            ds[0] += sqrt_fast(r3);
        }
        const double a5[5] = {xx, xy, x1, yy, y1};
#pragma unroll
        for (int al = 0; al < 5; ++al) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                if (G == 0 && g == 0) acc[al * 8 + g] += a5[al];
                else acc[al * 8 + g] = fma(a5[al], u0[g], acc[al * 8 + g]);
                acc[al * 8 + 4 + g] = fma(a5[al], u1[g], acc[al * 8 + 4 + g]);
            }
        }
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            if (!(G == 0 && g == 0)) acc[40 + g] += u0[g];     // the sum of ones is the point count
            acc[44 + g] += u1[g];
        }
        if (!more) break;
        a = na; b = nb; c = nc; i = nx;
    }
}

// ---- tensor-core variant of the fused pass (TVF_LARGE_DMMA=1; north star: "tensor cores ... for Gram formation on
// large-n triplets, where that step really is a dense contraction") -------------------------------------------------
// The 96 moments are the 6 x 16 x n contraction M = sum_i A6_i (x) U16_i (A6 = view-1 features, U16 = the 16 view-3 x
// view-2 products).  Padded to 8 x 16 it is two DMMA.8x8x4 accumulator tiles per warp; a k-step consumes 4 points.
// Fragment layout of mma.sync.m8n8k4.f64: lane l supplies A[l>>2][l&3] and B[l&3][l>>2], i.e. for point (l & 3) of
// the k-step the ONE view-1 feature m = l >> 2 and the ONE product n = l >> 2 (+ 8 for the second tile) -- every
// point's coordinates are therefore centred by 8 lanes, and each lane builds its three operands with lane-constant
// selects.  Per 4 points that is ~24 FP64 instructions + 2 DMMA (= 16 DFMA issue slots on the shared FP64 pipe) against
// ~19 for the DFMA form: the tensor-core form spends MORE pipe time, and is kept as measured evidence only.
#ifndef TVF_LARGE_DMMA
#define TVF_LARGE_DMMA 0
#endif
__device__ __forceinline__ void dmma_8x8x4(double (&c)[2], double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}

// warp `warp` of LG_WARPS takes k-steps warp, warp + LG_WARPS, ...; c0/c1: accumulator tiles (products 0..7 / 8..15);
// ds: this lane's share of the three distance sums (lanes with m = 0,1,2 own view 1,2,3)
__device__ __forceinline__ void moments_pass_dmma(const double* __restrict__ pts, int npts, int warp, int lane,
                                                  const double (&cen)[6], double (&c0)[2], double (&c1)[2], double& ds) {
    const int m = lane >> 2, kp = lane & 3;
    const int gam = m & 3, bhi = m >> 2;
    for (int base = warp * 4; base < npts; base += LG_WARPS * 4) {
        const int p = base + kp;
        const bool valid = p < npts;
        const double2* q = reinterpret_cast<const double2*>(pts + 6 * (valid ? p : base));
        const double2 a = q[0], b = q[1], c = q[2];
        const double x1 = a.x - cen[0], y1 = a.y - cen[1];
        const double x2 = b.x - cen[2], y2 = b.y - cen[3];
        const double x3 = c.x - cen[4], y3 = c.y - cen[5];
        const double r2 = fma(x2, x2, y2 * y2), r3 = fma(x3, x3, y3 * y3);
        // A operand: view-1 feature m of [x^2, xy, x, y^2, y, 1, 0, 0]
        const double ua = (m < 3) ? x1 : ((m < 5) ? y1 : ((m == 5) ? 1.0 : 0.0));
        const double ub = (m == 0) ? x1 : ((m == 1 || m == 3) ? y1 : 1.0);
        const double av = valid ? ua * ub : 0.0;
        // B operands: product n = 4*beta + gamma of m4(view 3)[beta] * m4(view 2)[gamma], m4 = [1, x, y, x^2+y^2]
        const double g = (gam == 0) ? 1.0 : ((gam == 1) ? x2 : ((gam == 2) ? y2 : r2));
        const double b0 = bhi ? x3 : 1.0, b1 = bhi ? r3 : y3;
        dmma_8x8x4(c0, av, g * b0);
        dmma_8x8x4(c1, av, g * b1);
        // distance sums of Normalize2Ddata.m:35: lanes m = 0, 1, 2 take views 1, 2, 3 of their point
        const double dd = (m == 0) ? fma(x1, x1, y1 * y1) : ((m == 1) ? r2 : r3);
        const double sq = sqrt_fast(dd);
        ds += (valid && m < 3) ? sq : 0.0;
    }
}

// grid = num_clusters * 8 CTAs; cluster c handles scenes c, c + num_clusters, ...  Three CTAs (of different
// clusters) share an SM, so one CTA's bulk copy and waits overlap the arithmetic of the others; the copy of a
// CTA's next slice is issued as soon as the last read of the current one has retired.
//
// There is NO cluster barrier in the steady state (barrier.cluster costs a GPU-scope MEMBAR plus a full
// rendezvous; ncu attributed 33 % of all warp samples to it).  The two exchanges of a scene are point-to-point:
// each CTA pushes its partial sums into the peers' shared memory with st.async, whose completion is counted in
// bytes on the RECEIVER's mbarrier -- (1) 6 coordinate sums from every rank to every rank (all need the
// centroid), (2) 99 sums from every rank to the scene's finalising rank (rotates with the scene, so no CTA is
// the permanent straggler).  Receive buffers are reused two (in1) / eight (in3) scenes later; a sender can only
// get that far ahead after the receiver has itself sent its next contribution, i.e. after it consumed the buffer.
// Warp roles in the fused pass: group G = warp & 1 (which half of the 96 sums), half H = warp >> 1 (which
// points: i = 32*H + lane, step 64).
__global__ void __cluster_dims__(LG_CLUSTER, 1, 1) __launch_bounds__(LG_THREADS, TVF_LG_MINB)
tft_moments_large_kernel(const double* __restrict__ corresp, int n, long long B, int slice_pts, int normalize,
                         double* __restrict__ ws) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned rank = cluster.block_rank();
    const long long cid = blockIdx.x / LG_CLUSTER, ncl = gridDim.x / LG_CLUSTER;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const size_t slice_bytes = (size_t)slice_pts * 48;
    const double* pts = reinterpret_cast<const double*>(smem_raw);
    LargeScratch& sc = *reinterpret_cast<LargeScratch*>(smem_raw + slice_bytes);

    const int p_lo = min(n, (int)rank * slice_pts), p_hi = min(n, p_lo + slice_pts);
    const int npts = p_hi - p_lo;                       // this CTA's points of every scene
    const unsigned bytes = (unsigned)npts * 48u;
    const double inv_n = 1.0 / (double)n;

    if (tid == 0) {
        mbar_init(&sc.bar_tma, 1); mbar_init(&sc.bar1[0], 1); mbar_init(&sc.bar1[1], 1); mbar_init(&sc.bar3, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    cluster.sync();                                     // every peer's barriers exist before any remote traffic
    if (tid == 0 && bytes > 0 && cid < B) {
        mbar_expect_tx(&sc.bar_tma, bytes);
        bulk_g2s(smem_raw, corresp + (cid * n + p_lo) * 6, bytes, &sc.bar_tma);
    }
    unsigned it = 0;                                    // scenes this cluster has processed
    for (long long scene = cid; scene < B; scene += ncl, ++it) {
        const int par = it & 1;
        if (bytes > 0) mbar_wait(&sc.bar_tma, it & 1u);
        // ---- pass 1: centroids (Normalize2Ddata.m:34) ------------------------------------------------
        double cen[6] = {0, 0, 0, 0, 0, 0};
        if (normalize) {
            double sa[6] = {0, 0, 0, 0, 0, 0}, sb[6] = {0, 0, 0, 0, 0, 0};
            int i = tid;
            for (; i + 3 * LG_THREADS < npts; i += 4 * LG_THREADS) {
                double2 v[12];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const double2* q = reinterpret_cast<const double2*>(pts + 6 * (i + u * LG_THREADS));
                    v[3 * u] = q[0]; v[3 * u + 1] = q[1]; v[3 * u + 2] = q[2];
                }
#pragma unroll
                for (int u = 0; u < 4; u += 2) {
                    sa[0] += v[3 * u].x; sa[1] += v[3 * u].y; sa[2] += v[3 * u + 1].x; sa[3] += v[3 * u + 1].y;
                    sa[4] += v[3 * u + 2].x; sa[5] += v[3 * u + 2].y;
                    sb[0] += v[3 * u + 3].x; sb[1] += v[3 * u + 3].y; sb[2] += v[3 * u + 4].x; sb[3] += v[3 * u + 4].y;
                    sb[4] += v[3 * u + 5].x; sb[5] += v[3 * u + 5].y;
                }
            }
            for (; i < npts; i += LG_THREADS) {
                const double2* q = reinterpret_cast<const double2*>(pts + 6 * i);
                const double2 a = q[0], b = q[1], c = q[2];
                sa[0] += a.x; sa[1] += a.y; sa[2] += b.x; sa[3] += b.y; sa[4] += c.x; sa[5] += c.y;
            }
#pragma unroll
            for (int k = 0; k < 6; ++k) { const double w = warp_sum_l(sa[k] + sb[k]); if (lane == 0) sc.wpart1[warp][k] = w; }
            __syncthreads();
            if (tid < 6 * LG_CLUSTER) {                    // thread (dest rank, component): push this CTA's sum to every rank
                const unsigned dst = tid / 6, k = tid % 6;
                double a = 0.0;
#pragma unroll
                for (int w = 0; w < LG_WARPS; ++w) a += sc.wpart1[w][k];
                st_async_f64(mapa_u32(smem_u32(&sc.in1[par][rank][k]), dst), a, mapa_u32(smem_u32(&sc.bar1[par]), dst));
            }
            if (tid == 0) mbar_expect_tx(&sc.bar1[par], LG_CLUSTER * 6 * 8);
            mbar_wait(&sc.bar1[par], (it >> 1) & 1u);
            if (tid < 6) {
                double a = 0.0;
#pragma unroll
                for (int r = 0; r < LG_CLUSTER; ++r) a += sc.in1[par][r][tid];      // rank order: deterministic
                sc.cen[par][tid] = a * inv_n;
            }
            __syncthreads();
#pragma unroll
            for (int k = 0; k < 6; ++k) cen[k] = sc.cen[par][k];
        }
        // ---- pass 2 (fused): distance sums (:35) + the 96 centred raw moments ----------------------------
#if TVF_LARGE_DMMA
        {
            double c0[2] = {0.0, 0.0}, c1[2] = {0.0, 0.0}, dsl = 0.0;
            moments_pass_dmma(pts, npts, warp, lane, cen, c0, c1, dsl);
            const int m = lane >> 2, kp = lane & 3;
            if (m < 6) {                                   // rows 6, 7 of the accumulator tiles are padding
                sc.wpartD[warp][m * 16 + 2 * kp] = c0[0]; sc.wpartD[warp][m * 16 + 2 * kp + 1] = c0[1];
                sc.wpartD[warp][m * 16 + 8 + 2 * kp] = c1[0]; sc.wpartD[warp][m * 16 + 8 + 2 * kp + 1] = c1[1];
            }
            // lanes with the same m hold the partial distance sum of view m + 1: add over kp (xor 1, 2), then lane m*4 stores
            dsl += __shfl_xor_sync(0xffffffffu, dsl, 1);
            dsl += __shfl_xor_sync(0xffffffffu, dsl, 2);
            if (kp == 0 && m < 3) sc.wpartD[warp][96 + m] = dsl;
        }
#else
        double acc[48], ds[2] = {0.0, 0.0};
#pragma unroll
        for (int k = 0; k < 48; ++k) acc[k] = 0.0;
        const int grp = warp & 1, first = (warp >> 1) * 32 + lane;
        if (grp == 0) moments_pass<0>(pts, npts, first, cen, acc, ds);
        else moments_pass<1>(pts, npts, first, cen, acc, ds);
        const double t32 = warp_reduce_transposed<0, 32>(acc, lane);
        const double t16 = warp_reduce_transposed<32, 16>(acc, lane);
        const double d0 = warp_sum_l(ds[0]), d1 = warp_sum_l(ds[1]);
        sc.wpart2[warp][lane] = t32;
        if (lane < 16) sc.wpart2[warp][32 + lane] = t16;
        if (lane == 0) { sc.wpart2[warp][48] = d0; sc.wpart2[warp][49] = d1; }
#endif
        __syncthreads();                                  // every thread is done with the slice
        {
            const long long next = scene + ncl;
            if (tid == 0 && bytes > 0 && next < B) {
                mbar_expect_tx(&sc.bar_tma, bytes);
                bulk_g2s(smem_raw, corresp + (next * n + p_lo) * 6, bytes, &sc.bar_tma);
            }
        }
        const unsigned fin = it % LG_CLUSTER;              // the rank that finalises this scene
        if (tid < 99) {
            double v;
#if TVF_LARGE_DMMA
            v = 0.0;
#pragma unroll
            for (int w = 0; w < LG_WARPS; ++w) v += sc.wpartD[w][tid];          // index = alpha*16 + beta*4 + gamma | 96 + view
            if (tid == 80) v = (double)npts;
#else
            if (tid < 96) {
                const int al = tid >> 4, be = (tid >> 2) & 3, ga = tid & 3;     // moment index = alpha*16 + beta*4 + gamma
                const int g = be >> 1, k = al * 8 + (be & 1) * 4 + ga;
                v = (tid == 80) ? (double)npts : sc.wpart2[g][k] + sc.wpart2[g + 2][k];
            } else {
                const int w = tid - 96, g = (w == 2) ? 1 : 0, k = (w == 1) ? 49 : 48;
                v = sc.wpart2[g][k] + sc.wpart2[g + 2][k];
            }
#endif
            st_async_f64(mapa_u32(smem_u32(&sc.in3[rank][tid]), fin), v, mapa_u32(smem_u32(&sc.bar3), fin));
        }
        if (rank == fin) {                                 // CTA-uniform branch
            if (tid == 0) mbar_expect_tx(&sc.bar3, LG_CLUSTER * 99 * 8);
            mbar_wait(&sc.bar3, (it / LG_CLUSTER) & 1u);
            double a = 0.0;
            if (tid < 99) {
#pragma unroll
                for (int r = 0; r < LG_CLUSTER; ++r) a += sc.in3[r][tid];           // rank order: deterministic
                if (tid >= 96) sc.scl[tid - 96] = normalize ? 1.4142135623730951 / (a * inv_n) : 1.0;       // :36
            }
            __syncthreads();
            double* rec = ws + scene * CORE_WS_TFT;
            const double s1 = sc.scl[0], s2 = sc.scl[1], s3 = sc.scl[2];
            if (tid < 96) {
                const int al = tid >> 4, be = (tid >> 2) & 3, ga = tid & 3;
                // degree of each feature in its view's coordinates, and the signs of m4 = [1, -x, -y, r]
                const double f1 = (al == 5) ? 1.0 : ((al == 2 || al == 4) ? s1 : s1 * s1);
                const double f3 = (be == 0) ? 1.0 : ((be == 3) ? s3 * s3 : -s3);
                const double f2 = (ga == 0) ? 1.0 : ((ga == 3) ? s2 * s2 : -s2);
                rec[CW_MOM_L + tid] = a * (f1 * (f3 * f2));
            }
            if (tid < 9) {                                 // N = [s 0 -s*cx; 0 s -s*cy; 0 0 1]  (:37)
                const double s = (tid < 3) ? sc.scl[tid] : sc.scl[(tid - 3) >> 1];
                rec[CW_STATS_L + tid] = (tid < 3) ? s : -s * (normalize ? sc.cen[par][tid - 3] : 0.0);
            }
        }
    }
    cluster.sync();      // no CTA retires while a peer may still write into (or wait on data from) its shared memory
}

// returns 0 when the shape is not supported by this kernel (caller falls back to tft_stage1_kernel)
int launch_tft_moments_large(const double* corresp, int n, long long B, int normalize, double* ws, int sm_count,
                             cudaStream_t stream) {
    if (B <= 0) return 1;
    const int slice_pts = (n + LG_CLUSTER - 1) / LG_CLUSTER;
    const size_t smem = (size_t)slice_pts * 48 + sizeof(LargeScratch) + 128;
    if (smem > 200 * 1024) return 0;
    // per-device function attribute: set on every launch (cheap), never cached process-wide
    if (cudaFuncSetAttribute(tft_moments_large_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
#if TVF_LG_CLUSTER > 8
    cudaFuncSetAttribute(tft_moments_large_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
#endif
    // clusters that can be co-resident (8 CTAs of a cluster must share a GPC, so this is not sm_count*3/8 in
    // general); scenes are assigned statically, so launching more than fit would serialise whole clusters.
    // Cached per (device, shared-memory size) and per host thread.
    static thread_local int max_clusters = 0, max_clusters_dev = -1;
    static thread_local size_t max_clusters_smem = 0;
    int cur_dev = 0;
    cudaGetDevice(&cur_dev);
    if (max_clusters == 0 || max_clusters_smem != smem || max_clusters_dev != cur_dev) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(sm_count * TVF_LG_MINB / LG_CLUSTER * LG_CLUSTER)); cfg.blockDim = dim3(LG_THREADS);
        cfg.dynamicSmemBytes = smem;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = LG_CLUSTER; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        int nc = 0;
        if (cudaOccupancyMaxActiveClusters(&nc, tft_moments_large_kernel, &cfg) != cudaSuccess || nc < 1) {
            cudaGetLastError();
            nc = sm_count * 2 / LG_CLUSTER;
        }
        max_clusters = nc; max_clusters_smem = smem; max_clusters_dev = cur_dev;
    }
    long long clusters = max_clusters;
    if (clusters > B) clusters = B;
    if (clusters < 1) clusters = 1;
    tft_moments_large_kernel<<<(unsigned)(clusters * LG_CLUSTER), LG_THREADS, smem, stream>>>(corresp, n, B, slice_pts,
                                                                                            normalize, ws);
    return cudaPeekAtLastError() == cudaSuccess ? 1 : 0;
}

}  // namespace tvf
