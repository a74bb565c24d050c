// tvf_ransac_kernels.cu -- the RANSAC pose estimator's own kernels (tvf_ransac_pose, tvf_consensus): sampling, the
// three-view consensus (the hot path), selection, the refit's compaction and the result rule.  The hypotheses and the
// refit themselves are the pose path's kernels (run_pose_chunk in tvf_api.cu).
#include "tvf_kernels.h"
#include "tvf_ransac.cuh"

namespace tvf {

namespace {

unsigned blocks_for(long long work, int threads, long long cap) {
    long long b = (work + threads - 1) / threads;
    if (b > cap) b = cap;
    return (unsigned)(b < 1 ? 1 : b);
}

// one thread per hypothesis q = b H + h
__global__ void ransac_sample_kernel(RansacArgs a, int H, int s) {
    const long long Q = a.B * H;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < Q; q += (long long)gridDim.x * blockDim.x) {
        const long long b = q / H;
        int idx[8];
        ransac_sample(a.seeds[b], (uint32_t)(q - b * H), a.n, s, idx);
        double* out = a.gin + q * 6 * s;
        for (int j = 0; j < s; ++j) {
            const double2* p = reinterpret_cast<const double2*>(a.corresp + (b * a.n + idx[j]) * 6);
            double2* o = reinterpret_cast<double2*>(out + 6 * j);
            o[0] = p[0]; o[1] = p[1]; o[2] = p[2];
        }
        if (a.calm_batched)
            for (int e = 0; e < 27; ++e) a.gcalm[q * 27 + e] = a.calm[b * 27 + e];
    }
}

// One thread per (pose, point) pair, pose-major, grid-stride with whole warps, so a warp holds one or a few poses.
// Each warp adds its inlier count per pose with one atomic (integers: the sum does not depend on the order).
__global__ void __launch_bounds__(256) ransac_consensus_kernel(const double* __restrict__ corresp, const double* __restrict__ calm,
                                                               int calm_batched, int n, long long Q, int H,
                                                               const double* __restrict__ Rt2, const double* __restrict__ Rt3,
                                                               const int* __restrict__ hstatus, double th, int* count,
                                                               unsigned char* mask) {
    const long long total = Q * n;
    const int lane = threadIdx.x & 31;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long e0 = (long long)blockIdx.x * blockDim.x + threadIdx.x - lane; e0 < total; e0 += stride) {
        const long long e = e0 + lane;
        const bool live = e < total;
        const long long q = live ? e / n : -1;
        const int i = live ? (int)(e - q * n) : 0;
        bool inl = false, flagged = false;
        if (live) {
            flagged = hstatus != nullptr && hstatus[q] != 0;
            if (!flagged) {
                const long long b = q / H;
                double P1[12], P2[12], P3[12], p6[6];
                ransac_cameras(calm + (calm_batched ? b * 27 : 0), Rt2 + q * 12, Rt3 + q * 12, P1, P2, P3);
                const double2* p = reinterpret_cast<const double2*>(corresp + (b * n + i) * 6);
                const double2 u = p[0], v = p[1], w = p[2];
                p6[0] = u.x; p6[1] = u.y; p6[2] = v.x; p6[3] = v.y; p6[4] = w.x; p6[5] = w.y;
                inl = ransac_inlier(P1, P2, P3, p6, th);
            }
            if (mask) mask[e] = inl ? 1 : 0;
        }
        const unsigned peers = __match_any_sync(0xffffffffu, q);
        const unsigned votes = __ballot_sync(0xffffffffu, inl);
        const int c = __popc(peers & votes);
        if (live && lane == __ffs(peers) - 1 && c) atomicAdd(count + q, c);
        if (live && flagged && i == 0) atomicAdd(count + q, -1);
    }
}

// one warp per problem: the largest count, ties to the smallest h
__global__ void ransac_select_kernel(RansacArgs a, int H) {
    const int lane = threadIdx.x & 31;
    const long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= a.B) return;
    int best = -2, bh = 0x7fffffff;
    for (int h = lane; h < H; h += 32) {
        const int c = a.hcount[b * H + h];
        if (c > best) { best = c; bh = h; }                // h ascends per lane: the first of equal counts stays
    }
    for (int off = 16; off > 0; off >>= 1) {
        const int c = __shfl_xor_sync(0xffffffffu, best, off), hh = __shfl_xor_sync(0xffffffffu, bh, off);
        if (c > best || (c == best && hh < bh)) { best = c; bh = hh; }
    }
    const bool failed = best < 0;
    if (lane == 0) a.best_h[b] = failed ? -1 : bh;
    if (lane < 12) {
        const long long q = b * H + bh;
        a.bestRt2[b * 12 + lane] = failed ? (double)NAN : a.hRt2[q * 12 + lane];
        a.bestRt3[b * 12 + lane] = failed ? (double)NAN : a.hRt3[q * 12 + lane];
    }
}

// one warp per listed problem: its consensus columns in index order (ballot prefix sums)
__global__ void ransac_gather_kernel(RansacArgs a, const int* __restrict__ plist, int m, int k) {
    const int lane = threadIdx.x & 31;
    const long long j = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (j >= m) return;
    const long long b = plist[j];
    const unsigned char* mk = a.mask_best + b * a.n;
    double* out = a.rin + j * 6 * k;
    int base = 0;
    for (int i0 = 0; i0 < a.n; i0 += 32) {
        const int i = i0 + lane;
        const bool in = i < a.n && mk[i] != 0;
        const unsigned bal = __ballot_sync(0xffffffffu, in);
        if (in) {
            const int pos = base + __popc(bal & ((1u << lane) - 1u));
            const double* p = a.corresp + (b * a.n + i) * 6;
            for (int r = 0; r < 6; ++r) out[pos * 6 + r] = p[r];
        }
        base += __popc(bal);
    }
    if (a.calm_batched && lane < 27) a.rcalm[j * 27 + lane] = a.calm[b * 27 + lane];
}

__global__ void ransac_scatter_kernel(RansacArgs a, const int* __restrict__ plist, int m, const double* __restrict__ Rt2,
                                      const double* __restrict__ Rt3, const int* __restrict__ st) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)m * 12) return;
    const long long j = e / 12, r = e - j * 12, b = plist[j];
    a.refRt2[b * 12 + r] = Rt2[j * 12 + r];
    a.refRt3[b * 12 + r] = Rt3[j * 12 + r];
    if (r == 0) a.refst[b] = st[j];
}

// one warp per problem: the result rule of tvf_ransac_pose
__global__ void ransac_finish_kernel(RansacArgs a, int s) {
    const int lane = threadIdx.x & 31;
    const long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= a.B) return;
    const int bh = a.best_h[b], cb = a.cnt_best[b], cr = a.cnt_refit[b];
    const bool refit = bh >= 0 && cb >= s && a.refst[b] == 0 && cr >= cb;
    const unsigned char* mk = (refit ? a.mask_refit : a.mask_best) + b * a.n;
    for (int i = lane; i < a.n; i += 32) a.inliers[b * a.n + i] = mk[i];
    if (lane < 12) {
        a.Rt2[b * 12 + lane] = refit ? a.refRt2[b * 12 + lane] : a.bestRt2[b * 12 + lane];
        a.Rt3[b * 12 + lane] = refit ? a.refRt3[b * 12 + lane] : a.bestRt3[b * 12 + lane];
    }
    if (lane == 0) {
        a.n_inliers[b] = refit ? cr : cb;
        a.status[b] = bh >= 0 ? 0 : ST_RANSAC_FAILED;
        int idx[8];
        if (bh >= 0) ransac_sample(a.seeds[b], (uint32_t)bh, a.n, s, idx);
        for (int j = 0; j < s; ++j) a.sample[b * s + j] = bh >= 0 ? idx[j] : -1;
    }
}

}  // namespace

void launch_ransac_consensus(const double* corresp, const double* calm, int calm_batched, int n, long long Q, int H,
                             const double* Rt2, const double* Rt3, const int* hstatus, double th, int* count,
                             unsigned char* mask, int sm_count, cudaStream_t stream) {
    if (Q <= 0) return;
    ransac_consensus_kernel<<<blocks_for(Q * n, 256, (long long)sm_count * 64), 256, 0, stream>>>(
        corresp, calm, calm_batched, n, Q, H, Rt2, Rt3, hstatus, th, count, mask);
}

void launch_ransac_sample(const RansacArgs& a, int H, int s, cudaStream_t stream) {
    ransac_sample_kernel<<<blocks_for(a.B * H, 128, 1LL << 20), 128, 0, stream>>>(a, H, s);
}

void launch_ransac_select(const RansacArgs& a, int H, cudaStream_t stream) {
    ransac_select_kernel<<<blocks_for(a.B * 32, 128, 1LL << 30), 128, 0, stream>>>(a, H);
}

void launch_ransac_gather(const RansacArgs& a, const int* plist, int m, int k, cudaStream_t stream) {
    ransac_gather_kernel<<<blocks_for((long long)m * 32, 128, 1LL << 30), 128, 0, stream>>>(a, plist, m, k);
}

void launch_ransac_scatter(const RansacArgs& a, const int* plist, int m, const double* Rt2, const double* Rt3,
                           const int* st, cudaStream_t stream) {
    ransac_scatter_kernel<<<blocks_for((long long)m * 12, 128, 1LL << 30), 128, 0, stream>>>(a, plist, m, Rt2, Rt3, st);
}

void launch_ransac_finish(const RansacArgs& a, int s, cudaStream_t stream) {
    ransac_finish_kernel<<<blocks_for(a.B * 32, 128, 1LL << 30), 128, 0, stream>>>(a, s);
}

}  // namespace tvf
