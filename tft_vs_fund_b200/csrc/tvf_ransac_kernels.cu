// tvf_ransac_kernels.cu -- the RANSAC pose estimator's own kernels (tvf_ransac_pose[_refined], tvf_consensus):
// sampling, the three-view consensus (the hot path), selection, the refit's compaction, the LO rounds' acceptance and
// the result rule.  The hypotheses and the refit themselves are the pose path's kernels (run_pose_chunk in tvf_api.cu),
// their adjustments the bundle adjustment's (tvf_ba_kernels.cu).
#include "tvf_kernels.h"
#include "tvf_ransac.cuh"

namespace tvf {

namespace {

unsigned blocks_for(long long work, int threads, long long cap) {
    long long b = (work + threads - 1) / threads;
    if (b > cap) b = cap;
    return (unsigned)(b < 1 ? 1 : b);
}

// The ragged kernels below are the <true> instantiations of the uniform kernels' code written as templates; the uniform
// sample, gather, LO-accept and finish kernels keep that code in their own bodies, because moving a kernel's body into
// an inlined function changes its machine code (the consensus kernel's does not change, so both forms share it).
// Where problem b's matches start and how many there are: ragged (offs) or uniform (b * a.n, a.n)
template <bool Ragged> __device__ __forceinline__ long long first_match(const RansacArgs& a, const long long* offs, long long b) {
    return Ragged ? offs[b] : b * a.n;
}
template <bool Ragged> __device__ __forceinline__ int matches(const RansacArgs& a, const long long* offs, long long b) {
    return Ragged ? (int)(offs[b + 1] - offs[b]) : a.n;
}

// one thread per hypothesis q = b H + h; a ragged problem of fewer than s matches gets NaN columns (every hypothesis
// flagged)
template <bool Ragged> __device__ __forceinline__ void sample_hypotheses(const RansacArgs& a, int H, int s, const long long* offs) {
    const long long Q = a.B * H;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < Q; q += (long long)gridDim.x * blockDim.x) {
        const long long b = q / H;
        const int n = matches<Ragged>(a, offs, b);
        double* out = a.gin + q * 6 * s;
        if (Ragged && n < s) {
            for (int e = 0; e < 6 * s; ++e) out[e] = __longlong_as_double(0x7ff8000000000000LL);
        } else {
            int idx[8];
            ransac_sample(a.seeds[b], (uint32_t)(q - b * H), n, s, idx);
            for (int j = 0; j < s; ++j) {
                const double2* p = reinterpret_cast<const double2*>(a.corresp + (first_match<Ragged>(a, offs, b) + idx[j]) * 6);
                double2* o = reinterpret_cast<double2*>(out + 6 * j);
                o[0] = p[0]; o[1] = p[1]; o[2] = p[2];
            }
        }
        if (a.calm_batched)
            for (int e = 0; e < 27; ++e) a.gcalm[q * 27 + e] = a.calm[b * 27 + e];
    }
}

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

__global__ void ransac_sample_ragged_kernel(RansacArgs a, int H, int s, const long long* offs) { sample_hypotheses<true>(a, H, s, offs); }

// One thread per (pose, point) pair, pose-major, grid-stride with whole warps, so a warp holds one or a few poses.
// Each warp adds its inlier count per pose with one atomic (integers: the sum does not depend on the order).
// Ragged: problem b's H n_b pairs form the segment that starts at H offs[b] (B problems, `total` = H offs[B] pairs); a
// thread finds its problem by binary search over offs, and an empty problem owns no pair.
template <bool Ragged>
__device__ __forceinline__ void consensus_pairs(const double* __restrict__ corresp, const double* __restrict__ calm,
                                                int calm_batched, int n, long long total, int H,
                                                const double* __restrict__ Rt2, const double* __restrict__ Rt3,
                                                const int* __restrict__ hstatus, double th, int* count,
                                                unsigned char* mask, const long long* __restrict__ offs, long long B) {
    const int lane = threadIdx.x & 31;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long e0 = (long long)blockIdx.x * blockDim.x + threadIdx.x - lane; e0 < total; e0 += stride) {
        const long long e = e0 + lane;
        const bool live = e < total;
        long long q = -1, first = 0;
        int i = 0;
        if (Ragged) {
            if (live) {
                const long long t = e / H;                 // offs[b] <= t < offs[b + 1]: the last b with offs[b] <= t
                long long lo = 0, hi = B;
                while (hi - lo > 1) {
                    const long long mid = (lo + hi) >> 1;
                    if (offs[mid] <= t) lo = mid; else hi = mid;
                }
                first = offs[lo];
                const long long nb = offs[lo + 1] - first, r = e - H * first, h = r / nb;
                q = lo * H + h;
                i = (int)(r - h * nb);
            }
        } else {
            q = live ? e / n : -1;
            i = live ? (int)(e - q * n) : 0;
        }
        bool inl = false, flagged = false;
        if (live) {
            flagged = hstatus != nullptr && hstatus[q] != 0;
            if (!flagged) {
                const long long b = q / H;
                double P1[12], P2[12], P3[12], p6[6];
                ransac_cameras(calm + (calm_batched ? b * 27 : 0), Rt2 + q * 12, Rt3 + q * 12, P1, P2, P3);
                const double2* p = reinterpret_cast<const double2*>(corresp + ((Ragged ? first : b * n) + i) * 6);
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

__global__ void __launch_bounds__(256) ransac_consensus_kernel(const double* __restrict__ corresp, const double* __restrict__ calm,
                                                               int calm_batched, int n, long long Q, int H,
                                                               const double* __restrict__ Rt2, const double* __restrict__ Rt3,
                                                               const int* __restrict__ hstatus, double th, int* count,
                                                               unsigned char* mask) {
    consensus_pairs<false>(corresp, calm, calm_batched, n, Q * n, H, Rt2, Rt3, hstatus, th, count, mask, nullptr, 0);
}

__global__ void __launch_bounds__(256) ransac_consensus_ragged_kernel(const double* __restrict__ corresp,
                                                                      const double* __restrict__ calm, int calm_batched,
                                                                      const long long* __restrict__ offs, long long B,
                                                                      long long total, int H, const double* __restrict__ Rt2,
                                                                      const double* __restrict__ Rt3,
                                                                      const int* __restrict__ hstatus, double th,
                                                                      int* count, unsigned char* mask) {
    consensus_pairs<true>(corresp, calm, calm_batched, 0, total, H, Rt2, Rt3, hstatus, th, count, mask, offs, B);
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
template <bool Ragged>
__device__ __forceinline__ void gather_consensus(const RansacArgs& a, const int* __restrict__ plist, int m, int k, const long long* offs) {
    const int lane = threadIdx.x & 31;
    const long long j = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (j >= m) return;
    const long long b = plist[j];
    const long long o = first_match<Ragged>(a, offs, b);
    const int n = matches<Ragged>(a, offs, b);
    const unsigned char* mk = a.mask_best + o;
    double* out = a.rin + j * 6 * k;
    int base = 0;
    for (int i0 = 0; i0 < n; i0 += 32) {
        const int i = i0 + lane;
        const bool in = i < n && mk[i] != 0;
        const unsigned bal = __ballot_sync(0xffffffffu, in);
        if (in) {
            const int pos = base + __popc(bal & ((1u << lane) - 1u));
            const double* p = a.corresp + (o + i) * 6;
            for (int r = 0; r < 6; ++r) out[pos * 6 + r] = p[r];
        }
        base += __popc(bal);
    }
    if (a.calm_batched && lane < 27) a.rcalm[j * 27 + lane] = a.calm[b * 27 + lane];
    if (a.gRt2 && lane < 12) { a.gRt2[j * 12 + lane] = a.bestRt2[b * 12 + lane]; a.gRt3[j * 12 + lane] = a.bestRt3[b * 12 + lane]; }
}

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
    if (a.gRt2 && lane < 12) { a.gRt2[j * 12 + lane] = a.bestRt2[b * 12 + lane]; a.gRt3[j * 12 + lane] = a.bestRt3[b * 12 + lane]; }
}

__global__ void ransac_gather_ragged_kernel(RansacArgs a, const int* __restrict__ plist, int m, int k, const long long* offs) {
    gather_consensus<true>(a, plist, m, k, offs);
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

// st[q] <- 1 if pose_st[q] != 0 (pose_st may be null) or the adjustment's status st[q] has ST_NONFINITE, else 0
__global__ void ransac_flag_kernel(const int* __restrict__ pose_st, int* st, long long Q) {
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < Q; q += (long long)gridDim.x * blockDim.x)
        st[q] = ((pose_st && pose_st[q] != 0) || (st[q] & ST_NONFINITE)) ? 1 : 0;
}

// one warp per problem: an LO round's pose replaces the current one if its count is larger (a flagged one counts -1)
template <bool Ragged> __device__ __forceinline__ void lo_accept(const RansacArgs& a, const long long* offs) {
    const int lane = threadIdx.x & 31;
    const long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= a.B) return;
    const int c = a.cnt_refit[b];
    if (!(c > a.cnt_best[b])) return;
    const long long o = first_match<Ragged>(a, offs, b);
    const int n = matches<Ragged>(a, offs, b);
    for (int i = lane; i < n; i += 32) a.mask_best[o + i] = a.mask_refit[o + i];
    if (lane < 12) { a.bestRt2[b * 12 + lane] = a.refRt2[b * 12 + lane]; a.bestRt3[b * 12 + lane] = a.refRt3[b * 12 + lane]; }
    __syncwarp();
    if (lane == 0) { a.cnt_best[b] = c; a.lo_done[b] += 1; }
}

__global__ void ransac_lo_accept_kernel(RansacArgs a) {
    const int lane = threadIdx.x & 31;
    const long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= a.B) return;
    const int c = a.cnt_refit[b];
    if (!(c > a.cnt_best[b])) return;
    for (int i = lane; i < a.n; i += 32) a.mask_best[b * a.n + i] = a.mask_refit[b * a.n + i];
    if (lane < 12) { a.bestRt2[b * 12 + lane] = a.refRt2[b * 12 + lane]; a.bestRt3[b * 12 + lane] = a.refRt3[b * 12 + lane]; }
    __syncwarp();
    if (lane == 0) { a.cnt_best[b] = c; a.lo_done[b] += 1; }
}

__global__ void ransac_lo_accept_ragged_kernel(RansacArgs a, const long long* offs) { lo_accept<true>(a, offs); }

// one warp per problem: the result rule of tvf_ransac_pose; a ragged problem of fewer than s matches: Rt NaN, inliers 0,
// count 0, sample -1, TVF_ST_TOO_FEW_MATCHES
template <bool Ragged> __device__ __forceinline__ void finish(const RansacArgs& a, int s, const long long* offs) {
    const int lane = threadIdx.x & 31;
    const long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= a.B) return;
    const long long o = first_match<Ragged>(a, offs, b);
    const int n = matches<Ragged>(a, offs, b);
    if (Ragged && n < s) {
        for (int i = lane; i < n; i += 32) a.inliers[o + i] = 0;
        if (lane < 12) { a.Rt2[b * 12 + lane] = (double)NAN; a.Rt3[b * 12 + lane] = (double)NAN; }
        if (lane < s) a.sample[b * s + lane] = -1;
        if (lane == 0) { a.n_inliers[b] = 0; a.status[b] = ST_TOO_FEW_MATCHES; }
        return;
    }
    const int bh = a.best_h[b], cb = a.cnt_best[b], cr = a.cnt_refit[b];
    const bool refit = bh >= 0 && cb >= s && a.refst[b] == 0 && cr >= cb;
    const unsigned char* mk = (refit ? a.mask_refit : a.mask_best) + o;
    for (int i = lane; i < n; i += 32) a.inliers[o + i] = mk[i];
    if (lane < 12) {
        a.Rt2[b * 12 + lane] = refit ? a.refRt2[b * 12 + lane] : a.bestRt2[b * 12 + lane];
        a.Rt3[b * 12 + lane] = refit ? a.refRt3[b * 12 + lane] : a.bestRt3[b * 12 + lane];
    }
    if (lane == 0) {
        a.n_inliers[b] = refit ? cr : cb;
        a.status[b] = bh >= 0 ? 0 : ST_RANSAC_FAILED;
        int idx[8];
        if (bh >= 0) ransac_sample(a.seeds[b], (uint32_t)bh, n, s, idx);
        for (int j = 0; j < s; ++j) a.sample[b * s + j] = bh >= 0 ? idx[j] : -1;
    }
}

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

__global__ void ransac_finish_ragged_kernel(RansacArgs a, int s, const long long* offs) { finish<true>(a, s, offs); }

}  // namespace

void launch_ransac_consensus(const double* corresp, const double* calm, int calm_batched, int n, long long Q, int H,
                             const double* Rt2, const double* Rt3, const int* hstatus, double th, int* count,
                             unsigned char* mask, int sm_count, cudaStream_t stream) {
    if (Q <= 0) return;
    ransac_consensus_kernel<<<blocks_for(Q * n, 256, (long long)sm_count * 64), 256, 0, stream>>>(
        corresp, calm, calm_batched, n, Q, H, Rt2, Rt3, hstatus, th, count, mask);
}

void launch_ransac_consensus_ragged(const double* corresp, const double* calm, int calm_batched, const long long* offs,
                                    long long B, long long m, int H, const double* Rt2, const double* Rt3,
                                    const int* hstatus, double th, int* count, unsigned char* mask, int sm_count,
                                    cudaStream_t stream) {
    if (B <= 0 || m <= 0) return;
    ransac_consensus_ragged_kernel<<<blocks_for(H * m, 256, (long long)sm_count * 64), 256, 0, stream>>>(
        corresp, calm, calm_batched, offs, B, H * m, H, Rt2, Rt3, hstatus, th, count, mask);
}

void launch_ransac_sample(const RansacArgs& a, int H, int s, cudaStream_t stream, const long long* offs) {
    const unsigned g = blocks_for(a.B * H, 128, 1LL << 20);
    if (offs) ransac_sample_ragged_kernel<<<g, 128, 0, stream>>>(a, H, s, offs);
    else ransac_sample_kernel<<<g, 128, 0, stream>>>(a, H, s);
}

void launch_ransac_select(const RansacArgs& a, int H, cudaStream_t stream) {
    ransac_select_kernel<<<blocks_for(a.B * 32, 128, 1LL << 30), 128, 0, stream>>>(a, H);
}

void launch_ransac_gather(const RansacArgs& a, const int* plist, int m, int k, cudaStream_t stream, const long long* offs) {
    const unsigned g = blocks_for((long long)m * 32, 128, 1LL << 30);
    if (offs) ransac_gather_ragged_kernel<<<g, 128, 0, stream>>>(a, plist, m, k, offs);
    else ransac_gather_kernel<<<g, 128, 0, stream>>>(a, plist, m, k);
}

void launch_ransac_scatter(const RansacArgs& a, const int* plist, int m, const double* Rt2, const double* Rt3,
                           const int* st, cudaStream_t stream) {
    ransac_scatter_kernel<<<blocks_for((long long)m * 12, 128, 1LL << 30), 128, 0, stream>>>(a, plist, m, Rt2, Rt3, st);
}

void launch_ransac_flag(const int* pose_st, int* st, long long Q, cudaStream_t stream) {
    if (Q <= 0) return;
    ransac_flag_kernel<<<blocks_for(Q, 256, 1LL << 20), 256, 0, stream>>>(pose_st, st, Q);
}

void launch_ransac_lo_accept(const RansacArgs& a, cudaStream_t stream, const long long* offs) {
    const unsigned g = blocks_for(a.B * 32, 128, 1LL << 30);
    if (offs) ransac_lo_accept_ragged_kernel<<<g, 128, 0, stream>>>(a, offs);
    else ransac_lo_accept_kernel<<<g, 128, 0, stream>>>(a);
}

void launch_ransac_finish(const RansacArgs& a, int s, cudaStream_t stream, const long long* offs) {
    const unsigned g = blocks_for(a.B * 32, 128, 1LL << 30);
    if (offs) ransac_finish_ragged_kernel<<<g, 128, 0, stream>>>(a, s, offs);
    else ransac_finish_kernel<<<g, 128, 0, stream>>>(a, s);
}

}  // namespace tvf
