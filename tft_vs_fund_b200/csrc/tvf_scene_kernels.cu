// tvf_scene_kernels.cu -- batched trials of the synthetic sweep generated on the device (SURVEY.md 8 f1).
// One thread per trial; the MT19937 state and the 6 x (n+100) coordinate scratch live in local memory.
#include <cstdint>

#include "tvf_kernels.h"
#include "tvf_scene.cuh"

namespace tvf {

__global__ void __launch_bounds__(64)
sweep_trials_kernel(long long first_trial, long long B, int n, const double* __restrict__ noise_levels, int L,
                    const double* __restrict__ P, double hi_x, double hi_y, double* __restrict__ out) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const long long j = first_trial + b;                    // global trial index (experiments.m:74-95)
    const uint32_t seed = (uint32_t)(j / L + 1);
    const double noise = noise_levels[j % L];
    MT19937 rng;
    double c[6 * SCENE_MAX_POINTS];
    unsigned char arr[SCENE_MAX_POINTS];
    signed char outpos[SCENE_MAX_POINTS];
    double Pl[36];
    for (int i = 0; i < 36; ++i) Pl[i] = P[i];
    scene_trial(rng, Pl, n, noise, seed, hi_x, hi_y, out + b * 6 * n, c, arr, outpos);
}

// One thread per SEED: the L noise levels of a seed share the seeding, the sub-sample permutation and the whole
// first pass of the generator (scene_seed_levels), ~L times less work than one thread per trial.
__global__ void __launch_bounds__(64)
sweep_seeds_kernel(long long first_trial, long long B, int n, const double* __restrict__ noise_levels, int L,
                   const double* __restrict__ P, double hi_x, double hi_y, double* __restrict__ out) {
    const long long s0 = first_trial / L;
    const long long s = s0 + (long long)blockIdx.x * blockDim.x + threadIdx.x;       // 0-based seed index, seed = s + 1
    const long long j_lo = s * L, last = first_trial + B;
    if (j_lo >= last) return;
    const int lv_lo = (int)((first_trial > j_lo) ? first_trial - j_lo : 0);
    const int lv_hi = (int)((last - j_lo < L) ? last - j_lo : L);
    MT19937 rng, snap;
    double clean[6 * SCENE_MAX_POINTS], z[6 * SCENE_MAX_POINTS], c[6 * SCENE_MAX_POINTS];
    unsigned char arr[SCENE_MAX_POINTS];
    signed char outpos[SCENE_MAX_POINTS];
    double Pl[36];
    for (int i = 0; i < 36; ++i) Pl[i] = P[i];
    scene_seed_levels(rng, snap, Pl, n, noise_levels, lv_lo, lv_hi, (uint32_t)(s + 1), hi_x, hi_y,
                      out + (j_lo + lv_lo - first_trial) * 6 * n, clean, z, c, arr, outpos);
}

// ------------------------------------------------------------------------------------------------------------------
// One WARP per seed.  The thread-per-seed kernel above keeps ~23 KB of generator state per thread in local memory and
// runs 77 k serial threads for a 1 M-trial sweep: latency bound (27 ms, twice the time of the solver it feeds).  Here
// the warp shares one generator whose state lives in shared memory, and every phase that the reference's stream order
// allows is spread over the lanes -- with exactly the bits of scene_seed_levels:
//   * MT19937 state regeneration ("twist"): element i depends on old i, i+1 and on i+397 (old) or i-227 (new), so 32
//     consecutive elements are independent: 20 lane-parallel steps, out of place into the other half of a two-block ring.
//     The ring holds blocks [cur, cur+1] of the stream, so a consumer may look 624 words ahead and a noise level can
//     rewind to the position its refill passes start from; a rewind past the ring re-twists from the seeded state,
//     which every lane keeps in 20 registers (never needed at the reference's scene parameters, but exact if it is).
//   * uniforms (3-D points): fixed stream positions, lane = point.
//   * polar Gaussian pairs: lane = candidate pair (4 words); accepted pairs are ranked with a ballot / popcount, the
//     rank gives (view, point) in the reference's v-major order, and the stream position after the last needed pair
//     is where the next consumer continues.  log / sqrt / divide run only on accepted lanes.
//   * inside-image compaction: ballot ranks in point order -> position in the sub-sample (outpos) -> 48-byte store.
//   * the seeding recurrence (624 dependent steps) and the sub-sample shuffle (data-dependent swaps) are serial; the
//     shuffle runs on lane 0 over words that all lanes tempered beforehand.
#ifndef TVF_SW_MINB
#define TVF_SW_MINB 14                             // resident warps per SM the kernel is compiled for (128 registers)
#endif
constexpr int SW_WARPS = 1;                     // warps (= seeds) per CTA
constexpr int SW_CAP = 32;                      // points per chunk of a refill pass (one per lane)
constexpr int SW_CAP2 = 8;                      // memoised second refill pass: up to this many points
constexpr unsigned SW_FULL = 0xffffffffu;

struct WarpMT {
    uint32_t* raw;        // shared memory, 2 x 624 words: block b of the stream's state sits in raw[(b & 1) * 624]
    uint32_t init[20];    // this lane's words (32 q + lane) of the seeded state ("block -1")
    int cur;              // lowest block in the ring (-1: the seeded state itself)
    bool have_next;       // block cur + 1 is in the other half
    int lane;

    __device__ __forceinline__ void seed(uint32_t s) {                     // init_genrand
        uint32_t* dst = raw + 624;
        __syncwarp();
#pragma unroll 8
        for (int i = 0; i < 624; ++i) {
            if (lane == 0) dst[i] = s;
            s = 1812433253u * (s ^ (s >> 30)) + (uint32_t)i + 1u;
        }
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 20; ++q) init[q] = (32 * q + lane < 624) ? dst[32 * q + lane] : 0u;
        cur = -1; have_next = false;
    }
    __device__ __forceinline__ void reset() {
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 20; ++q)
            if (32 * q + lane < 624) raw[624 + 32 * q + lane] = init[q];
        __syncwarp();
        cur = -1; have_next = false;
    }
    __device__ __forceinline__ void make_next() {                           // block cur + 1 from block cur
        const uint32_t* src = raw + (cur & 1) * 624;
        uint32_t* dst = raw + ((cur + 1) & 1) * 624;
#pragma unroll 1
        for (int s = 0; s < 20; ++s) {
            const int i = 32 * s + lane;
            __syncwarp();                                                   // dst[i - 227], dst[0] of earlier steps
            if (i < 624) {
                const uint32_t a = src[i];
                const uint32_t b = (i < 623) ? src[i + 1] : dst[0];
                const uint32_t m = (i < 227) ? src[i + 397] : dst[i - 227];
                const uint32_t y = (a & 0x80000000u) | (b & 0x7fffffffu);
                dst[i] = m ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
            }
        }
        __syncwarp();
        have_next = true;
    }
    // make the words [pos_lo, pos_hi] readable (pos_hi - pos_lo < 624); all arguments warp-uniform
    __device__ __forceinline__ void prepare(int pos_lo, int pos_hi) {
        const int b_lo = pos_lo / 624, b_hi = pos_hi / 624;
        if (b_lo < cur) reset();
        while (b_hi > cur + 1) {
            if (!have_next) make_next();
            ++cur; have_next = false;
        }
        if (b_hi == cur + 1 && !have_next) make_next();
    }
    static __device__ __forceinline__ uint32_t temper(uint32_t y) {
        y ^= (y >> 11);
        y ^= (y << 7) & 0x9d2c5680u;
        y ^= (y << 15) & 0xefc60000u;
        y ^= (y >> 18);
        return y;
    }
    // genrand_int32 outputs number pos .. pos + K - 1
    template <int K>
    __device__ __forceinline__ void words(int pos, uint32_t (&w)[K]) const {
        const int b = pos / 624, off = pos - b * 624;
        const uint32_t* lo = raw + (b & 1) * 624 + off;
        const uint32_t* hi = raw + ((b + 1) & 1) * 624 + off - 624;
#pragma unroll
        for (int t = 0; t < K; ++t) w[t] = temper((off + t < 624) ? lo[t] : hi[t]);
    }
    static __device__ __forceinline__ double res53(uint32_t w0, uint32_t w1) {          // genrand_res53
        const uint32_t a = w0 >> 5, b = w1 >> 6;
        return (a * 67108864.0 + b) / 9007199254740992.0;
    }
};

// X = 400*rand(3,1)-200 from the six words at `pos`, projected by the three cameras (generateSyntheticScene.m:82-87)
__device__ __forceinline__ void sw_point(const WarpMT& mt, int pos, const double* __restrict__ P, double* __restrict__ dst) {
    uint32_t w[6];
    mt.words<6>(pos, w);
    const double X = TVF_ADD(TVF_MUL(400.0, WarpMT::res53(w[0], w[1])), -200.0);
    const double Y = TVF_ADD(TVF_MUL(400.0, WarpMT::res53(w[2], w[3])), -200.0);
    const double Z = TVF_ADD(TVF_MUL(400.0, WarpMT::res53(w[4], w[5])), -200.0);
#pragma unroll
    for (int v = 0; v < 3; ++v) {
        const double* Pv = P + 12 * v;
        double x[3];
#pragma unroll
        for (int r = 0; r < 3; ++r)
            x[r] = TVF_ADD(TVF_ADD(TVF_ADD(TVF_MUL(Pv[4 * r], X), TVF_MUL(Pv[4 * r + 1], Y)), TVF_MUL(Pv[4 * r + 2], Z)), Pv[4 * r + 3]);
        dst[2 * v] = TVF_DIV(x[0], x[2]);
        dst[2 * v + 1] = TVF_DIV(x[1], x[2]);
    }
}

// The 3*M accepted polar pairs that follow stream position `pos`, in the reference's order (view-major, then point;
// the first value returned for a pair is f*x2, the cached one f*x1).  The draws of the points i in [i_lo, i_hi) are
// stored at buf[6*(i - i_lo) + 2*view ..]; the others are only counted.  Returns the stream position after the last pair.
__device__ __forceinline__ int sw_normals(WarpMT& mt, int pos, int M, int i_lo, int i_hi, double* __restrict__ buf) {
    const int need = 3 * M, lane = mt.lane;
    const unsigned lt = (1u << lane) - 1u;
    int got = 0;
    while (got < need) {
        mt.prepare(pos, pos + 127);
        uint32_t w[4];
        mt.words<4>(pos + 4 * lane, w);
        const double x1 = TVF_ADD(TVF_MUL(2.0, WarpMT::res53(w[0], w[1])), -1.0);
        const double x2 = TVF_ADD(TVF_MUL(2.0, WarpMT::res53(w[2], w[3])), -1.0);
        const double r2 = TVF_ADD(TVF_MUL(x1, x1), TVF_MUL(x2, x2));
        const bool acc = !(r2 >= 1.0 || r2 == 0.0);
        const unsigned bal = __ballot_sync(SW_FULL, acc);
        const int idx = got + __popc(bal & lt);
        if (acc && idx < need) {
            const int v = idx / M, i = idx - v * M;
            if (i >= i_lo && i < i_hi) {
                const double f = TVF_SQRT(TVF_DIV(TVF_MUL(-2.0, tvf_log(r2)), r2));
                double* d = buf + 6 * (i - i_lo) + 2 * v;
                d[0] = TVF_MUL(f, x2); d[1] = TVF_MUL(f, x1);
            }
        }
        const unsigned last = __ballot_sync(SW_FULL, acc && idx == need - 1);
        if (last) { pos += 4 * __ffs(last); got = need; }
        else { got += __popc(bal); pos += 128; }
    }
    __syncwarp();
    return pos;
}

__device__ __forceinline__ bool sw_inside(const double* p, double hi_x, double hi_y) {      // :95-100
    bool inside = true;
#pragma unroll
    for (int v = 0; v < 3; ++v) {
        const double x = p[2 * v], y = p[2 * v + 1];
        inside = inside && (x <= hi_x) && (y <= hi_y) && (x >= 0.0) && (y >= 0.0);
    }
    return inside;
}

// x = clean + z*noise for this lane's point (:90-92); the inside-image points of the warp, in lane order, go to the
// sub-sample positions outpos[filled ...] (-1: not sampled).  Returns the number of inside points.
__device__ __forceinline__ int sw_emit(bool have, const double* __restrict__ cl, const double* __restrict__ zz, double noise,
                                       double hi_x, double hi_y, const signed char* __restrict__ outpos, int filled,
                                       unsigned lt, double* __restrict__ o) {
    double p[6];
    bool inside = false;
    if (have) {
#pragma unroll
        for (int q = 0; q < 6; ++q) p[q] = TVF_ADD(cl[q], TVF_MUL(zz[q], noise));
        inside = sw_inside(p, hi_x, hi_y);
    }
    const unsigned bal = __ballot_sync(SW_FULL, inside);
    if (inside) {
        const int k = outpos[filled + __popc(bal & lt)];
        if (k >= 0) {
            double2* d = reinterpret_cast<double2*>(o + 6 * k);
            d[0] = make_double2(p[0], p[1]); d[1] = make_double2(p[2], p[3]); d[2] = make_double2(p[4], p[5]);
        }
    }
    return __popc(bal);
}

__host__ __device__ inline size_t sw_warp_bytes(int N) {
    return 2 * 624 * 4 + (size_t)48 * N + (size_t)2 * 48 * (SW_CAP + SW_CAP2) + 2 * (size_t)((N + 15) & ~15);
}

// SLOTS = ceil(N / 32): the noise-free projections of a lane's points (32 q + lane) stay in registers.
template <int SLOTS>
__global__ void __launch_bounds__(SW_WARPS * 32, TVF_SW_MINB)
sweep_seeds_warp_kernel(long long first_trial, long long B, int n, const double* __restrict__ noise_levels, int L,
                        const double* __restrict__ Pg, double hi_x, double hi_y, double* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char sw_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int N = n + 100, Npad = (N + 15) & ~15;
    double* P = reinterpret_cast<double*>(sw_smem);                          // 36 doubles, shared by the CTA
    for (int i = threadIdx.x; i < 36; i += blockDim.x) P[i] = Pg[i];
    __syncthreads();
    unsigned char* base = sw_smem + 288 + (size_t)warp * sw_warp_bytes(N);
    double* z = reinterpret_cast<double*>(base);                             // first pass: the Gaussian draws
    double* cc = z + 6 * N;                                                  // refill chunk: projections  (shuffle: tempered words)
    double* cz = cc + 6 * SW_CAP;                                            // refill chunk: Gaussian draws (shuffle: swap list)
    double* cc2 = cz + 6 * SW_CAP;                                           // memoised second refill pass
    double* cz2 = cc2 + 6 * SW_CAP2;
    WarpMT mt;
    mt.raw = reinterpret_cast<uint32_t*>(cz2 + 6 * SW_CAP2);
    mt.lane = lane;
    unsigned char* arr = reinterpret_cast<unsigned char*>(mt.raw + 2 * 624);
    signed char* outpos = reinterpret_cast<signed char*>(arr + Npad);

    const long long s0 = first_trial / L;
    const long long s = s0 + (long long)blockIdx.x * SW_WARPS + warp;         // 0-based seed index, seed = s + 1
    const long long j_lo = s * L, last_trial = first_trial + B;
    if (j_lo >= last_trial) return;
    const int lv_lo = (int)((first_trial > j_lo) ? first_trial - j_lo : 0);
    const int lv_hi = (int)((last_trial - j_lo < L) ? last_trial - j_lo : L);
    double* out0 = out + (j_lo + lv_lo - first_trial) * 6 * n;
    const unsigned lt = (1u << lane) - 1u;

    // ---- experiments.m:94-95: rng(it); randsample(N+100, N) = first n entries of a legacy shuffle of 0..N-1
    for (int i = lane; i < N; i += 32) { arr[i] = (unsigned char)i; outpos[i] = -1; }
    mt.seed((uint32_t)(s + 1));
    {
        // random_interval(top) = first word w (masked to the smallest 2^k - 1 >= top) with w <= top, for top = N-1 .. 1.
        // Whether word l of a batch is accepted depends on how many words before it were: a triangular system, solved
        // by fixed-point iteration on the ballot (bits 0..t-1 are final after t rounds; 2-4 rounds in practice).  The
        // swaps themselves are order dependent and run on lane 0 from the compacted (top, j) list.
        unsigned short* swaps = reinterpret_cast<unsigned short*>(cz);
        int top = N - 1, pos = 0;
        while (top >= 1) {
            mt.prepare(pos, pos + 31);
            uint32_t w[1];
            mt.words<1>(pos + lane, w);
            unsigned acc = 0;
            int my_top; uint32_t v = 0;
            while (true) {
                my_top = top - __popc(acc & lt);
                bool a = false;
                if (my_top >= 1) { v = w[0] & (0xffffffffu >> __clz(my_top)); a = v <= (uint32_t)my_top; }
                const unsigned nacc = __ballot_sync(SW_FULL, a);
                if (nacc == acc) break;
                acc = nacc;
            }
            const unsigned past = __ballot_sync(SW_FULL, my_top < 1);       // words after the shuffle has finished
            const int used = past ? __ffs(past) - 1 : 32;
            const int cnt = __popc(acc);
            if ((acc >> lane) & 1u) swaps[__popc(acc & lt)] = (unsigned short)((my_top << 8) | (int)v);
            __syncwarp();
            if (lane == 0) {
                for (int r = 0; r < cnt; ++r) {
                    const int pr = swaps[r], t = pr >> 8, j = pr & 255;
                    const unsigned char tmp = arr[t]; arr[t] = arr[j]; arr[j] = tmp;
                }
            }
            __syncwarp();
            top -= cnt; pos += used;
        }
        for (int k = lane; k < n; k += 32) outpos[arr[k]] = (signed char)k;
        __syncwarp();
    }
    // ---- generateSyntheticScene.m:75-92, first pass (rng(seed) again: the same stream from its start)
    double clean[SLOTS][6];                                                  // first pass: projections without noise
#pragma unroll
    for (int q = 0; q < SLOTS; ++q) {
        const int i0 = 32 * q;
#pragma unroll
        for (int t = 0; t < 6; ++t) clean[q][t] = 0.0;
        if (i0 < N) {
            const int i1 = (i0 + 32 < N) ? i0 + 32 : N;
            mt.prepare(6 * i0, 6 * i1 - 1);
            if (i0 + lane < N) sw_point(mt, 6 * (i0 + lane), P, clean[q]);
        }
    }
    const int snap_pos = sw_normals(mt, 6 * N, N, 0, N, z);
    // ---- per noise level: scale the draws, inside-image mask + compaction, refill passes (:95-110).
    // The first refill pass of a level starts at snap_pos for every level, and its points and draws do not depend on
    // the noise level -- only their number M does; the second pass likewise depends only on where it starts and on its
    // size.  Levels that agree in those (the usual case) reuse them: memo slot 0 = first pass (<= SW_CAP points, in
    // cc/cz), slot 1 = second pass (<= SW_CAP2 points, in cc2/cz2).  Anything else is generated into cc/cz in chunks.
    int m0_M = -1, m0_end = 0, m1_M = -1, m1_pos = 0, m1_end = 0;
    for (int lv = lv_lo; lv < lv_hi; ++lv) {
        const double noise = noise_levels[lv];
        double* o = out0 + (size_t)(lv - lv_lo) * 6 * n;
        int filled = 0;
#pragma unroll
        for (int q = 0; q < SLOTS; ++q) {
            const int i0 = 32 * q;
            if (i0 < N) {
                const int i = (i0 + lane < N) ? i0 + lane : N - 1;
                filled += sw_emit(i0 + lane < N, clean[q], z + 6 * i, noise, hi_x, hi_y, outpos, filled, lt, o);
            }
        }
        int M = N - filled, pos = snap_pos, npass = 0;
        while (M > 0) {
            const bool s0 = npass == 0 && M <= SW_CAP, s1 = npass == 1 && M <= SW_CAP2;
            const bool reuse = (s0 && m0_M == M) || (s1 && m1_M == M && m1_pos == pos);
            double* bc = s1 ? cc2 : cc;
            double* bz = s1 ? cz2 : cz;
            const int lb = s1 ? (lane & (SW_CAP2 - 1)) : lane;
            int end_pos = s0 ? m0_end : m1_end;                 // valid when reuse
            if (!s0 && !s1) m0_M = -1;                          // the big buffers are about to be overwritten
            for (int c0 = 0; c0 < M; c0 += SW_CAP) {            // one chunk whenever a memo slot is involved
                const int c1 = (c0 + SW_CAP < M) ? c0 + SW_CAP : M;
                if (!reuse) {
                    __syncwarp();
                    mt.prepare(pos + 6 * c0, pos + 6 * c1 - 1);
                    if (c0 + lane < c1) sw_point(mt, pos + 6 * (c0 + lane), P, bc + 6 * lb);
                    __syncwarp();
                    end_pos = sw_normals(mt, pos + 6 * M, M, c0, c1, bz);
                }
                filled += sw_emit(c0 + lane < c1, bc + 6 * lb, bz + 6 * lb, noise, hi_x, hi_y, outpos, filled, lt, o);
            }
            if (s0) { m0_M = M; m0_end = end_pos; }
            if (s1) { m1_M = M; m1_pos = pos; m1_end = end_pos; }
            pos = end_pos; M = N - filled; ++npass;
        }
    }
}

void launch_sweep_trials(long long first_trial, long long B, int n, const double* d_noise_levels, int L, const double* d_P,
                         double hi_x, double hi_y, double* d_out, cudaStream_t stream) {
    if (B <= 0) return;
    const long long seeds = (first_trial + B - 1) / L - first_trial / L + 1;
    if ((reinterpret_cast<uintptr_t>(d_out) & 15) == 0) {
        const size_t smem = 288 + SW_WARPS * sw_warp_bytes(n + 100);
        const unsigned grid = (unsigned)((seeds + SW_WARPS - 1) / SW_WARPS);
        if (n + 100 <= 128)
            sweep_seeds_warp_kernel<4><<<grid, SW_WARPS * 32, smem, stream>>>(first_trial, B, n, d_noise_levels, L, d_P, hi_x, hi_y, d_out);
        else
            sweep_seeds_warp_kernel<5><<<grid, SW_WARPS * 32, smem, stream>>>(first_trial, B, n, d_noise_levels, L, d_P, hi_x, hi_y, d_out);
        return;
    }
    if (L >= 4) {
        sweep_seeds_kernel<<<(unsigned)((seeds + 63) / 64), 64, 0, stream>>>(first_trial, B, n, d_noise_levels, L, d_P, hi_x, hi_y, d_out);
        return;
    }
    sweep_trials_kernel<<<(unsigned)((B + 63) / 64), 64, 0, stream>>>(first_trial, B, n, d_noise_levels, L, d_P, hi_x, hi_y, d_out);
}

}  // namespace tvf
