// tvf_pose_kernels.cu -- the pose tail shared by both methods
// (R_t_from_TFT.m:40-106, LinearFPoseEstimation.m:59-78, triangulation3D.m,
// ReprError.m) plus the stand-alone batched forms of the small reference
// functions.  Thread mappings:
//   candidates : one thread per problem (3x3 algebra, 18 tiny SVDs)
//   votes / scale / final : one thread per (problem, point); a CTA covers
//       floor(256/n) whole problems (or strides over the points of one problem
//       when n > 256) so every per-problem reduction stays inside the CTA and
//       runs in a fixed order (integer atomics for the votes, a fixed-shape
//       shared-memory tree for the FP64 sums) -> bit-reproducible results.
#include "tvf_kernels.h"
#include "tvf_pose.cuh"
#include "tvf_async.cuh"

namespace tvf {

constexpr int PT_THREADS = 256;

struct PointMap {
    int ppb;    // problems per CTA iteration
    int tpp;    // threads per problem
    int lp;     // local problem of this thread
    int lpt;    // thread's rank inside its problem
    __device__ __forceinline__ PointMap(int n, int threads = PT_THREADS) {
        tpp = (n <= threads) ? n : threads;
        ppb = threads / tpp;
        lp = threadIdx.x / tpp;
        lpt = threadIdx.x - lp * tpp;
    }
};

#ifndef TVF_TAIL_SERIAL_SUM
#define TVF_TAIL_SERIAL_SUM 1
#endif

// Sums of the tpp partials of each problem in TWO arrays at once, result at lpt==0.  Up to 32 points per problem the
// owner thread adds them in index order after ONE barrier (a fixed order, so still bit-reproducible); the log-depth
// tree of seg_reduce costs a CTA barrier per level, which is what the fused tail was waiting on.
__device__ __forceinline__ void seg_reduce2(double* ra, double* rb, const PointMap& m) {
#if TVF_TAIL_SERIAL_SUM
    if (m.tpp <= 32) {
        __syncthreads();
        if (m.lp < m.ppb && m.lpt == 0) {
            double a = ra[threadIdx.x], b = rb[threadIdx.x];
            for (int i = 1; i < m.tpp; ++i) { a += ra[threadIdx.x + i]; b += rb[threadIdx.x + i]; }
            ra[threadIdx.x] = a; rb[threadIdx.x] = b;
        }
        __syncthreads();
        return;
    }
#endif
    int s = 1;
    while (s < m.tpp) s <<= 1;
    for (s >>= 1; s >= 1; s >>= 1) {
        __syncthreads();
        if (m.lp < m.ppb && m.lpt < s && m.lpt + s < m.tpp) {
            ra[threadIdx.x] += ra[threadIdx.x + s];
            rb[threadIdx.x] += rb[threadIdx.x + s];
        }
    }
    __syncthreads();
}

// fixed-shape tree over the tpp partials of each problem; result lands at lpt==0
__device__ __forceinline__ void seg_reduce(double* red, const PointMap& m) {
    int s = 1;
    while (s < m.tpp) s <<= 1;
    for (s >>= 1; s >= 1; s >>= 1) {
        __syncthreads();
        if (m.lp < m.ppb && m.lpt < s && m.lpt + s < m.tpp) red[threadIdx.x] += red[threadIdx.x + s];
    }
    __syncthreads();
}

__device__ __forceinline__ const double* calm_of(const PoseTailArgs& a, long long b) {
    return a.calm + (a.calm_batched ? b * 27 : 0);
}

// ------------------------------------------------------------------ candidates
#ifndef TVF_CAND_STORE128
#define TVF_CAND_STORE128 1
#endif
#ifndef TVF_CAND_THREADS
#define TVF_CAND_THREADS 128
#endif
#ifndef TVF_CAND_PER_SM
#define TVF_CAND_PER_SM 384          // resident threads per SM the candidates kernel is compiled for (register cap 65536 / this):
                                     // 384 (168 registers, 140 bytes spilled) 4.98 ms per 10 M against 5.12 at 512 (128 registers, 1.1 KB
                                     // spilled), 5.63 at 256 (196 registers, no spills), 6.02 at 640
#endif
__global__ void __launch_bounds__(TVF_CAND_THREADS, TVF_CAND_PER_SM / TVF_CAND_THREADS)
candidates_kernel(int mode, const double* __restrict__ model, PoseTailArgs a) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.B) return;
    double calm[27];
    const double* cm = calm_of(a, b);
#pragma unroll
    for (int i = 0; i < 27; ++i) calm[i] = __ldg(cm + i);
    double cand[CAND_SIZE];
    int st;
    if (mode == 0) {
        double T[27];
#pragma unroll
        for (int i = 0; i < 27; ++i) T[i] = model[b * 27 + i];
        st = candidates_from_tft(T, calm, cand);
    } else {
        double F[18];
#pragma unroll
        for (int i = 0; i < 18; ++i) F[i] = model[b * 18 + i];
        st = candidates_from_f(F, F + 9, calm, cand);
    }
#if TVF_CAND_STORE128
    {   // the record is 672 bytes and the arena 256-byte aligned: 42 128-bit stores instead of 84 64-bit ones
        double2* dst = reinterpret_cast<double2*>(a.cand + b * CAND_SIZE);
#pragma unroll
        for (int i = 0; i < CAND_SIZE / 2; ++i) dst[i] = make_double2(cand[2 * i], cand[2 * i + 1]);
    }
#else
#pragma unroll
    for (int i = 0; i < CAND_SIZE; ++i) a.cand[b * CAND_SIZE + i] = cand[i];
#endif
    if (a.status != nullptr && st != 0) a.status[b] |= st;
}

// ------------------------------------------------------------------------ votes
// the ray test in its form for a view-1 camera K1*[I | 0] (three cofactors are single products)
#ifndef TVF_RAY_AFF
#define TVF_RAY_AFF true
#endif
#ifndef TVF_VOTES_MINB
#define TVF_VOTES_MINB 2
#endif
__global__ void __launch_bounds__(PT_THREADS, TVF_VOTES_MINB)
votes_kernel(PoseTailArgs a) {
    __shared__ int sv[PT_THREADS * 10];
    const PointMap m(a.n);
    for (long long b0 = (long long)blockIdx.x * m.ppb; b0 < a.B; b0 += (long long)gridDim.x * m.ppb) {
        for (int e = threadIdx.x; e < m.ppb * 10; e += PT_THREADS) sv[e] = 0;
        __syncthreads();
        const long long b = b0 + m.lp;
        if (m.lp < m.ppb && b < a.B) {
            double P1[12];
            load_K1_as_P1(calm_of(a, b), P1);
            const double* cand = a.cand + b * CAND_SIZE;
            int v2[2] = {0, 0}, v3[2] = {0, 0}, n2 = 0, n3 = 0;
            for (int pt = m.lpt; pt < a.n; pt += m.tpp) {
                const double2* q = reinterpret_cast<const double2*>(a.corresp + (b * a.n + pt) * 6);
                const double2 p1 = __ldg(q), p2 = __ldg(q + 1), p3 = __ldg(q + 2);
                double ra[4], rb[4], m7[7];
                dlt_rows(P1, p1.x, p1.y, ra, rb);
                dlt_row_minors<TVF_RAY_AFF>(ra, rb, m7);               // P1 = K1*[I | 0]
                cheirality_point<TVF_RAY_AFF>(ra, rb, m7, cand, p2.x, p2.y, v2, &n2, nullptr, nullptr);
                cheirality_point<TVF_RAY_AFF>(ra, rb, m7, cand + CAND_PAIR, p3.x, p3.y, v3, &n3, nullptr, nullptr);
            }
            int vote[8], nan2, nan3;
            expand_votes(v2, n2, vote, &nan2);
            expand_votes(v3, n3, vote + 4, &nan3);
            int* dst = sv + m.lp * 10;
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (vote[k] != 0) atomicAdd(dst + k, vote[k]);
            if (nan2) atomicOr(dst + 8, nan2);
            if (nan3) atomicOr(dst + 9, nan3);
        }
        __syncthreads();
        for (int e = threadIdx.x; e < m.ppb * 10; e += PT_THREADS) {
            const long long bb = b0 + e / 10;
            if (bb < a.B) a.votes[bb * 10 + (e % 10)] = sv[e];
        }
        __syncthreads();
    }
}

struct Selected {
    int k2, k3;
    double P1[12], P2[12], Rt2[12], Rt3[12], KR3u3[12];   // KR3u3 = [K3*R3 | K3*t3] (t3 not yet scaled)
};

__device__ __forceinline__ void load_selected(const PoseTailArgs& a, long long b, Selected& s) {
    const int* v = a.votes + b * 10;
    int vote[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) vote[k] = v[k];
    s.k2 = select_candidate(vote, v[8]);
    s.k3 = select_candidate(vote + 4, v[9]);
    load_K1_as_P1(calm_of(a, b), s.P1);
    const double* cand = a.cand + b * CAND_SIZE;
    selected_pose(cand, s.k2 < 0 ? 0 : s.k2, s.Rt2, s.P2);
    selected_pose(cand + CAND_PAIR, s.k3 < 0 ? 0 : s.k3, s.Rt3, s.KR3u3);
}

// ------------------------------------------------------------------------ scale
#ifndef TVF_TAIL3_MINB
#define TVF_TAIL3_MINB 2          // scale / final kernels of the n > 256 tail: 2 CTAs per SM (128 registers) instead of 1 (216)
#endif
__global__ void __launch_bounds__(PT_THREADS)
scale_kernel(PoseTailArgs a) {
    __shared__ double rnum[PT_THREADS], rden[PT_THREADS];
    const PointMap m(a.n);
    for (long long b0 = (long long)blockIdx.x * m.ppb; b0 < a.B; b0 += (long long)gridDim.x * m.ppb) {
        const long long b = b0 + m.lp;
        double num = 0.0, den = 0.0;
        if (m.lp < m.ppb && b < a.B) {
            Selected s;
            load_selected(a, b, s);
            for (int pt = m.lpt; pt < a.n; pt += m.tpp) {
                const double2* q = reinterpret_cast<const double2*>(a.corresp + (b * a.n + pt) * 6);
                const double2 p1 = __ldg(q), p2 = __ldg(q + 1), p3 = __ldg(q + 2);
                const double p6[6] = {p1.x, p1.y, p2.x, p2.y, p3.x, p3.y};
                double cn, cd;
                scale_point(s.P1, s.P2, s.KR3u3, s.KR3u3 + 9, p6, &cn, &cd);
                num += cn; den += cd;
            }
        }
        rnum[threadIdx.x] = num; rden[threadIdx.x] = den;
        seg_reduce(rnum, m);
        seg_reduce(rden, m);
        if (m.lp < m.ppb && b < a.B && m.lpt == 0) {
            a.scale[2 * b] = rnum[threadIdx.x];
            a.scale[2 * b + 1] = rden[threadIdx.x];
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------ final
__global__ void __launch_bounds__(PT_THREADS)
final_kernel(PoseTailArgs a) {
    __shared__ double rsq[PT_THREADS];
    const PointMap m(a.n);
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    for (long long b0 = (long long)blockIdx.x * m.ppb; b0 < a.B; b0 += (long long)gridDim.x * m.ppb) {
        const long long b = b0 + m.lp;
        const bool live = (m.lp < m.ppb && b < a.B);
        double sq = 0.0;
        bool ok = false;
        Selected s;
        if (live) {
            load_selected(a, b, s);
            ok = (s.k2 >= 0 && s.k3 >= 0);
            const double lam = -a.scale[2 * b] / a.scale[2 * b + 1];          // R_t_from_TFT.m:72-74
#pragma unroll
            for (int i = 0; i < 3; ++i) { s.Rt3[9 + i] *= lam; s.KR3u3[9 + i] *= lam; }
            for (int pt = m.lpt; pt < a.n; pt += m.tpp) {
                const double2* q = reinterpret_cast<const double2*>(a.corresp + (b * a.n + pt) * 6);
                const double2 p1 = __ldg(q), p2 = __ldg(q + 1), p3 = __ldg(q + 2);
                const double p6[6] = {p1.x, p1.y, p2.x, p2.y, p3.x, p3.y};
                double X[3];
                sq += final_point(s.P1, s.P2, s.KR3u3, p6, X);
                if (a.reconst != nullptr) {
                    double* dst = a.reconst + (b * a.n + pt) * 3;
                    dst[0] = ok ? X[0] : qnan; dst[1] = ok ? X[1] : qnan; dst[2] = ok ? X[2] : qnan;
                }
            }
        }
        rsq[threadIdx.x] = sq;
        seg_reduce(rsq, m);
        if (live && m.lpt == 0) {
            const double err = sqrt(rsq[threadIdx.x] / (3.0 * (double)a.n));   // ReprError.m:65
            int st = 0;
            if (s.k2 < 0) st |= ST_NO_POSE_2;
            if (s.k3 < 0) st |= ST_NO_POSE_3;
            bool fin = isfinite(err);
#pragma unroll
            for (int i = 0; i < 12; ++i) fin = fin && isfinite(s.Rt2[i]) && isfinite(s.Rt3[i]);
            if (!fin) st |= ST_NONFINITE;
            if (a.Rt2 != nullptr)
#pragma unroll
                for (int i = 0; i < 12; ++i) a.Rt2[b * 12 + i] = ok ? s.Rt2[i] : qnan;
            if (a.Rt3 != nullptr)
#pragma unroll
                for (int i = 0; i < 12; ++i) a.Rt3[b * 12 + i] = ok ? s.Rt3[i] : qnan;
            if (a.repr_err != nullptr) a.repr_err[b] = ok ? err : qnan;
            if (a.status != nullptr && st != 0) a.status[b] |= st;
        }
        __syncthreads();
    }
}

// ---- n > 128: one problem per CTA iteration.  The selected cameras (36 doubles) are computed once per problem by one
// thread and published in shared memory instead of being rebuilt and held in 60 registers by every thread (216 -> 128
// registers for the final pass: two CTAs per SM instead of one).
__global__ void __launch_bounds__(PT_THREADS, 2)
scale_large_kernel(PoseTailArgs a) {
    __shared__ double rnum[PT_THREADS], rden[PT_THREADS];
    __shared__ double sP[36];            // P1 | P2 | [K3*R3 | K3*t3]
    const PointMap m(a.n);               // ppb == 1
    for (long long b = blockIdx.x; b < a.B; b += gridDim.x) {
        if (threadIdx.x == 0) {
            Selected s;
            load_selected(a, b, s);
#pragma unroll
            for (int i = 0; i < 12; ++i) { sP[i] = s.P1[i]; sP[12 + i] = s.P2[i]; sP[24 + i] = s.KR3u3[i]; }
        }
        __syncthreads();
        double num = 0.0, den = 0.0;
        for (int pt = threadIdx.x; pt < a.n; pt += PT_THREADS) {
            const double2* q = reinterpret_cast<const double2*>(a.corresp + (b * a.n + pt) * 6);
            const double2 p1 = __ldg(q), p2 = __ldg(q + 1), p3 = __ldg(q + 2);
            const double p6[6] = {p1.x, p1.y, p2.x, p2.y, p3.x, p3.y};
            double cn, cd;
            scale_point(sP, sP + 12, sP + 24, sP + 33, p6, &cn, &cd);
            num += cn; den += cd;
        }
        rnum[threadIdx.x] = num; rden[threadIdx.x] = den;
        seg_reduce(rnum, m);
        seg_reduce(rden, m);
        if (threadIdx.x == 0) { a.scale[2 * b] = rnum[0]; a.scale[2 * b + 1] = rden[0]; }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(PT_THREADS, 2)
final_large_kernel(PoseTailArgs a) {
    __shared__ double rsq[PT_THREADS];
    __shared__ double sP[36];
    __shared__ int sok;
    const PointMap m(a.n);               // ppb == 1
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    for (long long b = blockIdx.x; b < a.B; b += gridDim.x) {
        if (threadIdx.x == 0) {
            Selected s;
            load_selected(a, b, s);
            const bool ok = (s.k2 >= 0 && s.k3 >= 0);
            const double lam = -a.scale[2 * b] / a.scale[2 * b + 1];          // R_t_from_TFT.m:72-74
#pragma unroll
            for (int i = 0; i < 3; ++i) { s.Rt3[9 + i] *= lam; s.KR3u3[9 + i] *= lam; }
#pragma unroll
            for (int i = 0; i < 12; ++i) { sP[i] = s.P1[i]; sP[12 + i] = s.P2[i]; sP[24 + i] = s.KR3u3[i]; }
            int st = 0;
            if (s.k2 < 0) st |= ST_NO_POSE_2;
            if (s.k3 < 0) st |= ST_NO_POSE_3;
            bool fin = true;
#pragma unroll
            for (int i = 0; i < 12; ++i) fin = fin && isfinite(s.Rt2[i]) && isfinite(s.Rt3[i]);
            if (!fin) st |= ST_NONFINITE;
            if (a.Rt2 != nullptr)
#pragma unroll
                for (int i = 0; i < 12; ++i) a.Rt2[b * 12 + i] = ok ? s.Rt2[i] : qnan;
            if (a.Rt3 != nullptr)
#pragma unroll
                for (int i = 0; i < 12; ++i) a.Rt3[b * 12 + i] = ok ? s.Rt3[i] : qnan;
            if (a.status != nullptr && st != 0) a.status[b] |= st;
            sok = ok ? 1 : 0;
        }
        __syncthreads();
        const bool ok = sok != 0;
        double sq = 0.0;
        for (int pt = threadIdx.x; pt < a.n; pt += PT_THREADS) {
            const double2* q = reinterpret_cast<const double2*>(a.corresp + (b * a.n + pt) * 6);
            const double2 p1 = __ldg(q), p2 = __ldg(q + 1), p3 = __ldg(q + 2);
            const double p6[6] = {p1.x, p1.y, p2.x, p2.y, p3.x, p3.y};
            double X[3];
            sq += final_point(sP, sP + 12, sP + 24, p6, X);
            if (a.reconst != nullptr) {
                double* dst = a.reconst + (b * a.n + pt) * 3;
                dst[0] = ok ? X[0] : qnan; dst[1] = ok ? X[1] : qnan; dst[2] = ok ? X[2] : qnan;
            }
        }
        rsq[threadIdx.x] = sq;
        seg_reduce(rsq, m);
        if (threadIdx.x == 0) {
            const double err = sqrt(rsq[0] / (3.0 * (double)a.n));                // ReprError.m:65
            if (a.repr_err != nullptr) a.repr_err[b] = ok ? err : qnan;
            if (a.status != nullptr && !isfinite(err)) a.status[b] |= ST_NONFINITE;
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------- fused tail (7 <= n <= 256)
// votes + t3 scale + final triangulation/ReprError in one launch: each CTA owns whole problems (one
// thread per point), so every per-problem reduction is CTA-local and the three phases are separated by
// __syncthreads only.  The two-view solutions found during the cheirality test are reused for the scale
// (the selected candidate's DLT is the one R_t_from_TFT.m:69 computes again).  The selected cameras live
// in shared memory (36 doubles per problem), not in registers, between the phases.

#ifndef TVF_TAIL_MINB
#define TVF_TAIL_MINB 2
#endif
// 1 = round-2 form: both pair-2 candidates are triangulated accurately during the votes and the selected solution is
// reused for the scale (3 accurate DLTs per point); 0 = all four votes by the certified ray test, ONE accurate two-view
// DLT of the selected pose in the scale phase
#ifndef TVF_TAIL_REUSE_X
#define TVF_TAIL_REUSE_X 0
#endif
#ifndef TVF_TAIL_TMA
#define TVF_TAIL_TMA 1
#endif
// entry i (0..35) of the three cameras P1 | P2 | P3 of a problem for the selected candidates k2, k3
__device__ __forceinline__ double camera_entry(const double* calm, const double* cand, int k2, int k3, int i) {
    if (i < 12) return (i < 9) ? calm[(i % 3) + 9 * (i / 3)] : 0.0;                  // K1*[I | 0]
    const int pair = (i >= 24) ? 1 : 0, e = i - 12 - 12 * pair, k = pair ? k3 : k2;
    const double* c = cand + pair * CAND_PAIR;
    if (e < 9) return c[((k < 2) ? OFF_KR : OFF_KRP) + e];
    return ((k == 0 || k == 3) ? 1.0 : -1.0) * c[OFF_KT + e - 9];
}
// entry i (0..11) of [R | t] of candidate k of a pair (selected_pose, one element)
__device__ __forceinline__ double pose_entry(const double* c, int k, int i) {
    if (i < 9) return c[((k < 2) ? OFF_R : OFF_RP) + i];
    return ((k == 0 || k == 3) ? 1.0 : -1.0) * c[OFF_T + i - 9];
}
// seg_reduce2 for tpp <= 32 with the two arrays summed by two different threads of the problem (same index order as
// seg_reduce2: bit-identical sums), result at the problem's first thread
__device__ __forceinline__ void seg_reduce2_split(double* ra, double* rb, const PointMap& m) {
    if (m.tpp > 32) { seg_reduce2(ra, rb, m); return; }
    __syncthreads();
    if (m.lp < m.ppb && m.lpt < 2) {
        double* r = (m.lpt ? rb : ra) + (threadIdx.x - m.lpt);
        double acc = r[0];
        for (int i = 1; i < m.tpp; ++i) acc += r[i];
        r[0] = acc;
    }
    __syncthreads();
}
__device__ __forceinline__ void seg_reduce1(double* ra, const PointMap& m) {
    if (m.tpp > 32) { seg_reduce(ra, m); return; }
    __syncthreads();
    if (m.lp < m.ppb && m.lpt == 0) {
        double* r = ra + threadIdx.x;
        double acc = r[0];
        for (int i = 1; i < m.tpp; ++i) acc += r[i];
        r[0] = acc;
    }
}

// Every per-problem scalar step (candidate selection, t3 scale) is recomputed by ALL threads of the problem from shared
// memory instead of by one thread followed by a barrier, and the per-problem vectors (cameras, [R|t] outputs) are
// spread one element per thread: a warp holds one or two "first threads", so the single-thread sections cost every
// warp their full instruction count.  Five CTA barriers per iteration instead of nine.
#ifndef TVF_TAIL_CTA
#define TVF_TAIL_CTA 128
#endif
#ifndef TVF_TAIL_MINB_SMALL
#define TVF_TAIL_MINB_SMALL ((TVF_TAIL_MINB * PT_THREADS) / TVF_TAIL_CTA)
#endif
template <int THREADS>
__global__ void __launch_bounds__(THREADS, THREADS == PT_THREADS ? TVF_TAIL_MINB : TVF_TAIL_MINB_SMALL)
pose_tail_fused_kernel(PoseTailArgs a) {
    constexpr int MAX_PPB = THREADS / TAIL_FUSED_MIN_N;
    constexpr int PT_THREADS = THREADS;         // (shadows the file-wide constant inside this kernel)
    __shared__ int sv[MAX_PPB * 4];             // per local problem: vote(R,t), vote(Rp,t) for pairs 2 and 3
    __shared__ int snan[MAX_PPB];
    __shared__ double sP[MAX_PPB * 36];         // P1 | P2 | P3 = [K3*R3 | K3*t3]  (3x4 column-major each), t3 NOT yet scaled
    __shared__ double red0[THREADS], red1[THREADS], red2[THREADS];
    const PointMap m(a.n, THREADS);
    const int own = threadIdx.x - m.lpt;        // first thread of this thread's problem
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
#if TVF_TAIL_TMA
    // The correspondences and the candidate records of the CTA's NEXT group of problems (two contiguous ranges of global
    // memory: ppb*n*48 and ppb*672 bytes) are brought into the other half of a two-stage shared-memory buffer by two bulk
    // asynchronous copies (TMA engine) that one thread issues at the top of the iteration; every phase reads shared memory.
    extern __shared__ __align__(16) unsigned char tail_dsm[];
    __shared__ unsigned long long tbar[2];
    const unsigned pts_bytes = (unsigned)m.ppb * (unsigned)a.n * 48u, cand_bytes = (unsigned)m.ppb * (unsigned)(CAND_SIZE * 8);
    const unsigned stage_bytes = pts_bytes + cand_bytes;
    const long long bstep = (long long)gridDim.x * m.ppb;
    auto issue = [&](long long b0n, int stage) {          // thread 0 only
        const long long left = a.B - b0n;
        const unsigned np = (unsigned)(left < m.ppb ? left : m.ppb);
        unsigned char* dst = tail_dsm + (size_t)stage * stage_bytes;
        mbar_expect_tx(&tbar[stage], np * (unsigned)a.n * 48u + np * (unsigned)(CAND_SIZE * 8));
        bulk_g2s(dst, a.corresp + b0n * a.n * 6, np * (unsigned)a.n * 48u, &tbar[stage]);
        bulk_g2s(dst + pts_bytes, a.cand + b0n * CAND_SIZE, np * (unsigned)(CAND_SIZE * 8), &tbar[stage]);
    };
    if (threadIdx.x == 0) {
        mbar_init(&tbar[0], 1); mbar_init(&tbar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
#endif
    for (int e = threadIdx.x; e < m.ppb * 4; e += PT_THREADS) sv[e] = 0;
    for (int e = threadIdx.x; e < m.ppb; e += PT_THREADS) snan[e] = 0;
    __syncthreads();
#if TVF_TAIL_TMA
    if (threadIdx.x == 0 && (long long)blockIdx.x * m.ppb < a.B) issue((long long)blockIdx.x * m.ppb, 0);
    int iter = 0;
#endif
    for (long long b0 = (long long)blockIdx.x * m.ppb; b0 < a.B; b0 += (long long)gridDim.x * m.ppb) {
        const long long b = b0 + m.lp;
        const bool live = (m.lp < m.ppb && b < a.B);
#if TVF_TAIL_TMA
        // the other stage was last read before the final barrier of the previous iteration: free to be refilled
        if (threadIdx.x == 0 && b0 + bstep < a.B) issue(b0 + bstep, (iter + 1) & 1);
        const unsigned char* stg = tail_dsm + (size_t)(iter & 1) * stage_bytes;
        mbar_wait(&tbar[iter & 1], (unsigned)(iter >> 1) & 1u);
        ++iter;
        const double* cand = reinterpret_cast<const double*>(stg + pts_bytes) + (live ? m.lp : 0) * CAND_SIZE;
#else
        const double* cand = a.cand + (live ? b : 0) * CAND_SIZE;
#endif
        double* Ps = sP + (live ? m.lp : 0) * 36;
        double p6[6] = {0, 0, 0, 0, 0, 0};
#if TVF_TAIL_REUSE_X
        double Xa[4] = {0, 0, 0, 1}, Xb[4] = {0, 0, 0, 1};
#endif
        // ---- phase 1: cheirality votes (R_t_from_TFT.m:91-104) --------------------------------
        if (live) {
            double P1[12];
            load_K1_as_P1(calm_of(a, b), P1);
#if TVF_TAIL_TMA
            const double2* q = reinterpret_cast<const double2*>(stg) + (m.lp * a.n + m.lpt) * 3;
            const double2 q1 = q[0], q2 = q[1], q3 = q[2];
#else
            const double2* q = reinterpret_cast<const double2*>(a.corresp + (b * a.n + m.lpt) * 6);
            const double2 q1 = __ldg(q), q2 = __ldg(q + 1), q3 = __ldg(q + 2);
#endif
            p6[0] = q1.x; p6[1] = q1.y; p6[2] = q2.x; p6[3] = q2.y; p6[4] = q3.x; p6[5] = q3.y;
            double ra[4], rb[4], m7[7];
            dlt_rows(P1, p6[0], p6[1], ra, rb);
            dlt_row_minors<TVF_RAY_AFF>(ra, rb, m7);                   // P1 = K1*[I | 0]
            int v2[2] = {0, 0}, v3[2] = {0, 0}, n2 = 0, n3 = 0;
#if TVF_TAIL_REUSE_X
            cheirality_point<TVF_RAY_AFF>(ra, rb, m7, cand, p6[2], p6[3], v2, &n2, Xa, Xb);
#else
            cheirality_point<TVF_RAY_AFF>(ra, rb, m7, cand, p6[2], p6[3], v2, &n2, nullptr, nullptr);
#endif
            cheirality_point<TVF_RAY_AFF>(ra, rb, m7, cand + CAND_PAIR, p6[4], p6[5], v3, &n3, nullptr, nullptr);
            int* dst = sv + m.lp * 4;
            if (v2[0]) atomicAdd(dst + 0, v2[0]);
            if (v2[1]) atomicAdd(dst + 1, v2[1]);
            if (v3[0]) atomicAdd(dst + 2, v3[0]);
            if (v3[1]) atomicAdd(dst + 3, v3[1]);
            if (n2 | n3) atomicOr(snan + m.lp, n2 | (n3 << 2));
        }
        __syncthreads();
        // ---- selection by every thread; the cameras one element per thread -----------------------------
        int k2 = 15, k3 = 15;
        if (live) {
            int vote[8], nan2, nan3;
            expand_votes(sv + m.lp * 4, snan[m.lp] & 3, vote, &nan2);
            expand_votes(sv + m.lp * 4 + 2, (snan[m.lp] >> 2) & 3, vote + 4, &nan3);
            const int s2 = select_candidate(vote, nan2), s3 = select_candidate(vote + 4, nan3);
            k2 = (s2 < 0) ? 15 : s2; k3 = (s3 < 0) ? 15 : s3;
            if (m.lpt == 0 && a.votes != nullptr) {
                int* gv = a.votes + b * 10;
#pragma unroll
                for (int k = 0; k < 8; ++k) gv[k] = vote[k];
                gv[8] = nan2; gv[9] = nan3;
            }
            const double* calm = calm_of(a, b);
            for (int i = m.lpt; i < 36; i += m.tpp) Ps[i] = camera_entry(calm, cand, s2 < 0 ? 0 : s2, s3 < 0 ? 0 : s3, i);
        }
        __syncthreads();
        for (int e = threadIdx.x; e < m.ppb * 4; e += PT_THREADS) sv[e] = 0;       // for the next iteration (two barriers ahead)
        for (int e = threadIdx.x; e < m.ppb; e += PT_THREADS) snan[e] = 0;
        // ---- phase 2: t3 scale (R_t_from_TFT.m:68-74) ----------------------------------------------
        double num = 0.0, den = 0.0;
        if (live) {
#if TVF_TAIL_REUSE_X
            // X of the selected pair-2 candidate: (R,t)->Xa, (R,-t)->(Xa, -w), (Rp,-t)->(Xb, -w), (Rp,t)->Xb
            const bool useA = (k2 == 0 || k2 == 1 || k2 == 15);
            const double w = ((k2 == 1 || k2 == 2) ? -1.0 : 1.0) * (useA ? Xa[3] : Xb[3]);
            const double iw = 1.0 / w;
            const double Xc[3] = {(useA ? Xa[0] : Xb[0]) * iw, (useA ? Xa[1] : Xb[1]) * iw, (useA ? Xa[2] : Xb[2]) * iw};
            double X3[3], c1[3], c2[3];
            mat3_vec(Ps + 24, Xc, X3);
            const double p3[3] = {p6[4], p6[5], 1.0};
            cross3(p3, X3, c1);
            cross3(p3, Ps + 33, c2);
            num = c1[0] * c2[0] + c1[1] * c2[1] + c1[2] * c2[2];
            den = c2[0] * c2[0] + c2[1] * c2[1] + c2[2] * c2[2];
#else
            // the ONE accurate two-view DLT of the point: cameras 1 and 2 of the selected pose (R_t_from_TFT.m:69)
            scale_point(Ps, Ps + 12, Ps + 24, Ps + 33, p6, &num, &den);
#endif
        }
        red0[threadIdx.x] = num; red1[threadIdx.x] = den;
        seg_reduce2_split(red0, red1, m);
        const bool ok = (k2 != 15) && (k3 != 15);
        double sq = 0.0;
        if (live) {
            const double snum = red0[own], sden = red1[own];
            const double lam = -snum / sden;
            // [R2|t2], [R3|lam*t3] (:74), one element per thread; pose flags by the first thread
            bool fin = true;
            const int kk2 = (k2 == 15) ? 0 : k2, kk3 = (k3 == 15) ? 0 : k3;
            for (int i = m.lpt; i < 12; i += m.tpp) {
                const double r2 = pose_entry(cand, kk2, i);
                double r3 = pose_entry(cand + CAND_PAIR, kk3, i);
                if (i >= 9) r3 *= lam;
                fin = fin && isfinite(r2) && isfinite(r3);
                if (a.Rt2 != nullptr) a.Rt2[b * 12 + i] = ok ? r2 : qnan;
                if (a.Rt3 != nullptr) a.Rt3[b * 12 + i] = ok ? r3 : qnan;
            }
            int st = fin ? 0 : ST_NONFINITE;
            if (m.lpt == 0) {
                if (a.scale != nullptr) { a.scale[2 * b] = snum; a.scale[2 * b + 1] = sden; }
                if (k2 == 15) st |= ST_NO_POSE_2;
                if (k3 == 15) st |= ST_NO_POSE_3;
            }
            if (a.status != nullptr && st != 0) atomicOr(a.status + b, st);
            // ---- phase 3: final triangulation + ReprError, P3 = K3*[R3 | lam*t3] -------------------------
            const double t3s[3] = {Ps[33] * lam, Ps[34] * lam, Ps[35] * lam};
            double X[3];
            sq = final_point_kt(Ps, Ps + 12, Ps + 24, t3s, p6, X);
            if (a.reconst != nullptr) {
                double* dst = a.reconst + (b * a.n + m.lpt) * 3;
                dst[0] = ok ? X[0] : qnan; dst[1] = ok ? X[1] : qnan; dst[2] = ok ? X[2] : qnan;
            }
        }
        red2[threadIdx.x] = sq;
        seg_reduce1(red2, m);
        if (live && m.lpt == 0) {
            const double err = sqrt(red2[threadIdx.x] / (3.0 * (double)a.n));       // ReprError.m:65
            if (a.repr_err != nullptr) a.repr_err[b] = ok ? err : qnan;
            if (a.status != nullptr && !isfinite(err)) atomicOr(a.status + b, ST_NONFINITE);
        }
    }
}

// -------------------------------------------------- T = TFT_from_P(K1[I|0], K2 Rt2, K3 Rt3)
__global__ void __launch_bounds__(128)
tft_from_pose_kernel(const double* __restrict__ calm, int calm_batched, const double* __restrict__ Rt2,
                     const double* __restrict__ Rt3, long long B, double* __restrict__ T) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const double* cm = calm + (calm_batched ? b * 27 : 0);
    double K[3][9];
#pragma unroll
    for (int v = 0; v < 3; ++v)
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int r = 0; r < 3; ++r) K[v][r + 3 * c] = __ldg(cm + 3 * v + r + 9 * c);
    double P1[12], P2[12], P3[12], R[12];
#pragma unroll
    for (int i = 0; i < 9; ++i) P1[i] = K[0][i];
    P1[9] = 0.0; P1[10] = 0.0; P1[11] = 0.0;
#pragma unroll
    for (int i = 0; i < 12; ++i) R[i] = Rt2[b * 12 + i];
    mat3_mul(K[1], R, P2); mat3_vec(K[1], R + 9, P2 + 9);
#pragma unroll
    for (int i = 0; i < 12; ++i) R[i] = Rt3[b * 12 + i];
    mat3_mul(K[2], R, P3); mat3_vec(K[2], R + 9, P3 + 9);
    double t[27];
    tft_from_p(P1, P2, P3, t);
#pragma unroll
    for (int i = 0; i < 27; ++i) T[b * 27 + i] = t[i];
}

// ------------------------------------------------------- stand-alone batched functions
__global__ void normalize2d_kernel(const double* __restrict__ pts, int n, long long B, double* __restrict__ out,
                                   double* __restrict__ Nmat) {
    // one warp per problem (Normalize2Ddata.m:33-39)
    const int lane = threadIdx.x & 31;
    const long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= B) return;
    const double* p = pts + b * 2 * n;
    double sx = 0.0, sy = 0.0;
    for (int i = lane; i < n; i += 32) { sx += p[2 * i]; sy += p[2 * i + 1]; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { sx += __shfl_xor_sync(0xffffffffu, sx, o); sy += __shfl_xor_sync(0xffffffffu, sy, o); }
    const double cx = sx / n, cy = sy / n;
    double d = 0.0;
    for (int i = lane; i < n; i += 32) { const double dx = p[2 * i] - cx, dy = p[2 * i + 1] - cy; d += sqrt(dx * dx + dy * dy); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
    const double s = 1.4142135623730951 / (d / n);
    const double tx = -s * cx, ty = -s * cy;
    if (out != nullptr)
        for (int i = lane; i < n; i += 32) { out[b * 2 * n + 2 * i] = s * p[2 * i] + tx; out[b * 2 * n + 2 * i + 1] = s * p[2 * i + 1] + ty; }
    if (Nmat != nullptr && lane == 0) {
        double* N = Nmat + b * 9;
        N[0] = s; N[1] = 0; N[2] = 0; N[3] = 0; N[4] = s; N[5] = 0; N[6] = tx; N[7] = ty; N[8] = 1.0;
    }
}

__global__ void transform_tft_kernel(const double* __restrict__ T, const double* __restrict__ M1,
                                     const double* __restrict__ M2, const double* __restrict__ M3, int mats_batched,
                                     int inverse, long long B, double* __restrict__ Tout) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const long long mo = mats_batched ? b * 9 : 0;
    double t[27], m1[9], m2[9], m3[9], o[27];
#pragma unroll
    for (int i = 0; i < 27; ++i) t[i] = T[b * 27 + i];
#pragma unroll
    for (int i = 0; i < 9; ++i) { m1[i] = M1[mo + i]; m2[i] = M2[mo + i]; m3[i] = M3[mo + i]; }
    transform_tft(t, m1, m2, m3, inverse, o);
#pragma unroll
    for (int i = 0; i < 27; ++i) Tout[b * 27 + i] = o[i];
}

__global__ void tft_from_p_kernel(const double* __restrict__ P1, const double* __restrict__ P2,
                                  const double* __restrict__ P3, long long B, double* __restrict__ T) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double a[12], c[12], d[12], t[27];
#pragma unroll
    for (int i = 0; i < 12; ++i) { a[i] = P1[b * 12 + i]; c[i] = P2[b * 12 + i]; d[i] = P3[b * 12 + i]; }
    tft_from_p(a, c, d, t);
#pragma unroll
    for (int i = 0; i < 27; ++i) T[b * 27 + i] = t[i];
}

// image point (x,y) of view v for (problem b, point pt); rows = 2 or 3 per view
__device__ __forceinline__ void load_xy(const double* pts, int M, int rows, int n, long long b, int pt, int v,
                                        double* x, double* y) {
    const double* p = pts + ((b * n + pt) * M + v) * rows;
    double px = p[0], py = p[1];
    if (rows == 3) { const double w = p[2]; px /= w; py /= w; }     // triangulation3D.m:43-45
    *x = px; *y = py;
}

template <int M>
__device__ __forceinline__ void triangulate_m(const double* P, const double* pts, int rows, int n, long long b, int pt,
                                              double* X) {
    double a[2 * M][4];
#pragma unroll
    for (int v = 0; v < M; ++v) {
        double x, y;
        load_xy(pts, M, rows, n, b, pt, v, &x, &y);
        dlt_rows(P + 12 * v, x, y, a[2 * v], a[2 * v + 1]);
    }
    dlt_null<2 * M>(a, X);
}

__global__ void triangulate_kernel(const double* __restrict__ P, int M, int cams_batched, const double* __restrict__ pts,
                                   int rows, int n, long long B, double* __restrict__ X) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B * n) return;
    const long long b = e / n;
    const int pt = (int)(e - b * n);
    const double* Pb = P + (cams_batched ? b * 12 * M : 0);
    double x[4];
    if (M == 2) triangulate_m<2>(Pb, pts, rows, n, b, pt, x);
    else triangulate_m<3>(Pb, pts, rows, n, b, pt, x);
#pragma unroll
    for (int i = 0; i < 4; ++i) X[e * 4 + i] = x[i];
}

__global__ void __launch_bounds__(PT_THREADS)
repr_error_kernel(const double* __restrict__ P, int M, int cams_batched, const double* __restrict__ corresp, int rows,
                  int n, long long B, const double* __restrict__ pts3d, int pts_rows, double* __restrict__ err) {
    __shared__ double rsq[PT_THREADS];
    const PointMap m(n);
    for (long long b0 = (long long)blockIdx.x * m.ppb; b0 < B; b0 += (long long)gridDim.x * m.ppb) {
        const long long b = b0 + m.lp;
        const bool live = (m.lp < m.ppb && b < B);
        double sq = 0.0;
        if (live) {
            const double* Pb = P + (cams_batched ? b * 12 * M : 0);
            for (int pt = m.lpt; pt < n; pt += m.tpp) {
                double X[4];
                if (pts3d == nullptr) {                                           // ReprError.m:43-44
                    if (M == 2) triangulate_m<2>(Pb, corresp, rows, n, b, pt, X);
                    else triangulate_m<3>(Pb, corresp, rows, n, b, pt, X);
                } else {
                    const double* q = pts3d + (b * n + pt) * pts_rows;
                    X[0] = q[0]; X[1] = q[1]; X[2] = q[2]; X[3] = (pts_rows == 4) ? q[3] : 1.0;   // :45-48
                }
                for (int v = 0; v < M; ++v) {
                    double x, y, pr[3];
                    load_xy(corresp, M, rows, n, b, pt, v, &x, &y);
                    cam_apply(Pb + 12 * v, X, pr);
                    const double dx = pr[0] / pr[2] - x, dy = pr[1] / pr[2] - y;
                    sq += dx * dx + dy * dy;
                }
            }
        }
        rsq[threadIdx.x] = sq;
        seg_reduce(rsq, m);
        if (live && m.lpt == 0) err[b] = sqrt(rsq[threadIdx.x] / ((double)M * (double)n));
        __syncthreads();
    }
}

// Corresp = project3Dpoints(Points3D, Pcam)   (auxiliar_functions/project3Dpoints.m:28-35)
__global__ void project3d_kernel(const double* __restrict__ pts3d, const double* __restrict__ P, int M, int cams_batched,
                                 int n, long long B, double* __restrict__ out) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B * n) return;
    const long long b = e / n;
    const double* Pb = P + (cams_batched ? b * 12 * M : 0);
    const double X[4] = {pts3d[e * 3], pts3d[e * 3 + 1], pts3d[e * 3 + 2], 1.0};
    for (int v = 0; v < M; ++v) {
        double x[3];
        cam_apply(Pb + 12 * v, X, x);
        out[(e * M + v) * 2] = x[0] / x[2];
        out[(e * M + v) * 2 + 1] = x[1] / x[2];
    }
}

__global__ void ang_error_kernel(const double* __restrict__ Rt_true, int true_batched, const double* __restrict__ Rt_est,
                                 long long B, double* __restrict__ rot, double* __restrict__ tr) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double a[12], e[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) { a[i] = Rt_true[(true_batched ? b * 12 : 0) + i]; e[i] = Rt_est[b * 12 + i]; }
    double r, t;
    ang_error(a, e, &r, &t);
    rot[b] = r; tr[b] = t;
}

// ------------------------------------------------------- sweep evaluation (experiments.m:112-124)
// Per-trial ReprError / AngError accumulated per noise level.  Thread g owns level g % L and a fixed,
// strided subset of that level's trials, so its four partial sums are updated by one thread in a fixed
// order (chunk after chunk); sweep_eval_finish adds the per-thread partials in index order.  Bit-stable.
// NC = 6 (the after-adjustment columns of tvf_sweep_run_levels_ba): a trial is also skipped when its second status word
// (the adjustment's) is flagged, and its `iter` is summed into a sixth column.  NC = 5 never reads status2 / iter.
template <int NC>
__global__ void __launch_bounds__(256)
sweep_eval_accumulate_kernel(const double* __restrict__ Rt2, const double* __restrict__ Rt3, const double* __restrict__ repr,
                             const int* __restrict__ status, const int* __restrict__ status2, const int* __restrict__ iter,
                             long long first_trial, long long B, int L, int Q, const double* __restrict__ Rt0,
                             double* __restrict__ partial) {
    static_assert(NC == 5 || NC == 6, "sweep_eval: 5 or 6 columns");
    constexpr int SKIP = ST_NO_POSE_2 | ST_NO_POSE_3 | ST_NONFINITE;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= L * Q) return;
    const int level = g % L, q = g / L;
    const int r = (int)(((level - first_trial % L) % L + L) % L);
    double gt2[12], gt3[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) { gt2[i] = Rt0[i]; gt3[i] = Rt0[12 + i]; }
    double s_rep = 0.0, s_rot = 0.0, s_t = 0.0, cnt = 0.0, bad = 0.0, s_it = 0.0;
    for (long long b = r + (long long)L * q; b < B; b += (long long)L * Q) {
        if (status != nullptr && (status[b] & SKIP)) { bad += 1.0; continue; }
        if constexpr (NC == 6) {
            if (status2[b] & SKIP) { bad += 1.0; continue; }
        }
        double e2[12], e3[12];
#pragma unroll
        for (int i = 0; i < 12; ++i) { e2[i] = Rt2[b * 12 + i]; e3[i] = Rt3[b * 12 + i]; }
        double r2, t2, r3, t3;
        ang_error(gt2, e2, &r2, &t2);                                   // experiments.m:117-118
        ang_error(gt3, e3, &r3, &t3);
        s_rep += repr[b]; s_rot += (r2 + r3) * 0.5; s_t += (t2 + t3) * 0.5; cnt += 1.0;   // :112-120
        if constexpr (NC == 6) s_it += (double)iter[b];
    }
    double* p = partial + (size_t)g * NC;
    p[0] += s_rep; p[1] += s_rot; p[2] += s_t; p[3] += cnt; p[4] += bad;
    if constexpr (NC == 6) p[5] += s_it;
}

template <int NC>
__global__ void sweep_eval_finish_kernel(const double* __restrict__ partial, int L, int Q, double* __restrict__ table) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= L * NC) return;
    const int level = e / NC, c = e % NC;
    double a = 0.0;
    for (int q = 0; q < Q; ++q) a += partial[((size_t)q * L + level) * NC + c];
    table[e] = a;
}

void launch_sweep_eval_accumulate(const double* Rt2, const double* Rt3, const double* repr, const int* status,
                                  long long first_trial, long long B, int L, int Q, const double* d_Rt0, double* d_partial,
                                  cudaStream_t s, const int* status2, const int* iter) {
    if (B <= 0) return;
    if (status2 != nullptr)
        sweep_eval_accumulate_kernel<6><<<(L * Q + 255) / 256, 256, 0, s>>>(Rt2, Rt3, repr, status, status2, iter, first_trial,
                                                                             B, L, Q, d_Rt0, d_partial);
    else
        sweep_eval_accumulate_kernel<5><<<(L * Q + 255) / 256, 256, 0, s>>>(Rt2, Rt3, repr, status, nullptr, nullptr, first_trial,
                                                                             B, L, Q, d_Rt0, d_partial);
}

void launch_sweep_eval_finish(const double* d_partial, int L, int Q, double* d_table, cudaStream_t s, int ncol) {
    if (ncol == 6) sweep_eval_finish_kernel<6><<<(L * 6 + 63) / 64, 64, 0, s>>>(d_partial, L, Q, d_table);
    else sweep_eval_finish_kernel<5><<<(L * 5 + 63) / 64, 64, 0, s>>>(d_partial, L, Q, d_table);
}

// ------------------------------------------------------------------- launchers
static inline unsigned grid_for(long long work, int per_block, long long cap) {
    long long g = (work + per_block - 1) / per_block;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (unsigned)g;
}

void launch_candidates(int mode, const double* model, const PoseTailArgs& a, cudaStream_t stream) {
    if (a.B <= 0) return;
    candidates_kernel<<<grid_for(a.B, TVF_CAND_THREADS, 1LL << 30), TVF_CAND_THREADS, 0, stream>>>(mode, model, a);
}

static inline unsigned tail_grid(const PoseTailArgs& a, int sm_count) {
    const int tpp = (a.n <= PT_THREADS) ? a.n : PT_THREADS;
    const int ppb = PT_THREADS / tpp;
    return grid_for(a.B, ppb, (long long)sm_count * 32);
}

// CTA size of the fused tail: 128 threads (four resident CTAs per SM: the five barriers of an iteration wait for four warps
// instead of eight) unless 256 threads pack whole problems noticeably better (n = 48: 5 x 48 of 256 against 2 x 48 of 128)
#ifndef TVF_TAIL_SMALL_CTA
#define TVF_TAIL_SMALL_CTA 1
#endif
static inline int fused_tail_threads(int n) {
#if TVF_TAIL_SMALL_CTA
    if (n <= TVF_TAIL_CTA) {
        const int live_s = (TVF_TAIL_CTA / n) * n * (256 / TVF_TAIL_CTA), live256 = (256 / n) * n;      // live threads per 256
        if (live_s * 16 >= live256 * 15) return TVF_TAIL_CTA;
    }
#endif
    return 256;
}

template <int THREADS>
static void launch_fused_t(const PoseTailArgs& a, int sm_count, cudaStream_t stream) {
    const int tpp = (a.n <= THREADS) ? a.n : THREADS;
    const int ppb = THREADS / tpp;
    const unsigned grid = grid_for(a.B, ppb, (long long)sm_count * 16 * (THREADS == PT_THREADS ? TVF_TAIL_MINB : TVF_TAIL_MINB_SMALL));
#if TVF_TAIL_TMA
    const size_t dyn = 2 * (size_t)ppb * ((size_t)a.n * 48 + CAND_SIZE * 8);      // two stages of points + candidate records
    // (set on every launch: the attribute is per device and per context, a process-wide flag would miss the second GPU)
    cudaFuncSetAttribute(pose_tail_fused_kernel<THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
    pose_tail_fused_kernel<THREADS><<<grid, THREADS, dyn, stream>>>(a);
#else
    pose_tail_fused_kernel<THREADS><<<grid, THREADS, 0, stream>>>(a);
#endif
}

void launch_pose_tail_fused(const PoseTailArgs& a, int sm_count, cudaStream_t stream) {
    if (a.B <= 0) return;
    if (fused_tail_threads(a.n) == TVF_TAIL_CTA) launch_fused_t<TVF_TAIL_CTA>(a, sm_count, stream);
    else launch_fused_t<256>(a, sm_count, stream);
}

void launch_votes(const PoseTailArgs& a, int sm_count, cudaStream_t stream) {
    if (a.B <= 0) return;
    votes_kernel<<<tail_grid(a, sm_count), PT_THREADS, 0, stream>>>(a);
}

void launch_scale(const PoseTailArgs& a, int sm_count, cudaStream_t stream) {
    if (a.B <= 0) return;
    if (a.n > PT_THREADS / 2) scale_large_kernel<<<tail_grid(a, sm_count), PT_THREADS, 0, stream>>>(a);
    else scale_kernel<<<tail_grid(a, sm_count), PT_THREADS, 0, stream>>>(a);
}

void launch_final(const PoseTailArgs& a, int sm_count, cudaStream_t stream) {
    if (a.B <= 0) return;
    if (a.n > PT_THREADS / 2) final_large_kernel<<<tail_grid(a, sm_count), PT_THREADS, 0, stream>>>(a);
    else final_kernel<<<tail_grid(a, sm_count), PT_THREADS, 0, stream>>>(a);
}

void launch_tft_from_pose(const double* calm, int calm_batched, const double* Rt2, const double* Rt3, long long B,
                          double* T, cudaStream_t stream) {
    if (B <= 0) return;
    tft_from_pose_kernel<<<grid_for(B, 128, 1LL << 30), 128, 0, stream>>>(calm, calm_batched, Rt2, Rt3, B, T);
}

void launch_normalize2d(const double* pts, int n, long long B, double* out, double* Nmat, cudaStream_t s) {
    if (B <= 0) return;
    normalize2d_kernel<<<grid_for(B * 32, 256, 1LL << 30), 256, 0, s>>>(pts, n, B, out, Nmat);
}

void launch_transform_tft(const double* T, const double* M1, const double* M2, const double* M3, int mats_batched,
                          int inverse, long long B, double* Tout, cudaStream_t s) {
    if (B <= 0) return;
    transform_tft_kernel<<<grid_for(B, 128, 1LL << 30), 128, 0, s>>>(T, M1, M2, M3, mats_batched, inverse, B, Tout);
}

void launch_tft_from_p(const double* P1, const double* P2, const double* P3, long long B, double* T, cudaStream_t s) {
    if (B <= 0) return;
    tft_from_p_kernel<<<grid_for(B, 128, 1LL << 30), 128, 0, s>>>(P1, P2, P3, B, T);
}

void launch_triangulate(const double* P, int M, int cams_batched, const double* pts, int rows, int n, long long B,
                        double* X, cudaStream_t s) {
    if (B <= 0 || n <= 0) return;
    triangulate_kernel<<<grid_for(B * n, 128, 1LL << 30), 128, 0, s>>>(P, M, cams_batched, pts, rows, n, B, X);
}

void launch_repr_error(const double* P, int M, int cams_batched, const double* corresp, int rows, int n, long long B,
                       const double* pts3d, int pts_rows, double* err, cudaStream_t s) {
    if (B <= 0) return;
    const int tpp = (n <= PT_THREADS) ? n : PT_THREADS;
    const int ppb = PT_THREADS / tpp;
    repr_error_kernel<<<grid_for(B, ppb, 148LL * 32), PT_THREADS, 0, s>>>(P, M, cams_batched, corresp, rows, n, B, pts3d,
                                                                          pts_rows, err);
}

void launch_project3d(const double* pts3d, const double* P, int M, int cams_batched, int n, long long B, double* out,
                      cudaStream_t s) {
    if (B <= 0 || n <= 0) return;
    project3d_kernel<<<grid_for(B * n, 128, 1LL << 30), 128, 0, s>>>(pts3d, P, M, cams_batched, n, B, out);
}

void launch_ang_error(const double* Rt_true, int true_batched, const double* Rt_est, long long B, double* rot,
                      double* tr, cudaStream_t s) {
    if (B <= 0) return;
    ang_error_kernel<<<grid_for(B, 128, 1LL << 30), 128, 0, s>>>(Rt_true, true_batched, Rt_est, B, rot, tr);
}

}  // namespace tvf
