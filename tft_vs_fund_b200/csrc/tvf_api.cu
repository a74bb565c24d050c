// tvf_api.cu -- the C ABI of include/tvf.h: handle, work-space arenas, chunked
// host-pointer entry points (H2D / kernels / D2H pipelined over three streams)
// and asynchronous device-pointer entry points.  No CPU fallback lives here:
// every entry point either runs the CUDA kernels or returns an error.
#include "../../include/tvf.h"

#include <cuda_runtime.h>
#include <sched.h>

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "tvf_kernels.h"
#include "tvf_pose.cuh"

using namespace tvf;

namespace {

#ifndef TVF_NSLOT
#define TVF_NSLOT 3
#endif
#ifndef TVF_RAMP
#define TVF_RAMP 0
#endif
constexpr int NSLOT = TVF_NSLOT;
constexpr int NSCRATCH = 24;
constexpr int64_t DEFAULT_CHUNK = 65536;        // host-pointer entry points: chunks are the H2D / kernels / D2H pipeline stages
constexpr int64_t DEFAULT_CHUNK_DEV = 1 << 20;  // device-pointer entry points: fewer, larger launches (less launch and wave-tail
                                                // overhead: 8.32e7 / 8.48e7 / 8.58e7 / 8.63e7 solves/s at 262 144 / 524 288 / 1 M /
                                                // 2 M problems per launch, profiles/r02_variants.md); the 2.3 GB of work space is
                                                // far from L2-resident, which costs nothing measurable (the path is FP64-bound)
constexpr size_t ARENA_BUDGET = 384u << 20;   // bytes of per-slot work space the automatic chunk aims for

struct Slot {
    cudaStream_t stream = nullptr;
    char* arena = nullptr;
    size_t cap = 0;
};

std::string g_create_error;

}  // namespace

struct tvf_context {
    int device = 0;
    int sm_count = 148;
    Slot slot[NSLOT];
    cudaStream_t user_stream = nullptr;
    bool use_user_stream = false;
    int64_t chunk_user = 0;
    void* scratch[NSCRATCH] = {};
    size_t scratch_cap[NSCRATCH] = {};
    std::string err;
    int64_t launches = 0;
    // optional per-kernel CUDA-event timing (tvf_profile_*): (kernel id, start, stop) per launch
    bool profiling = false;
    struct Ev { int id; cudaEvent_t a, b; };
    std::vector<Ev> events;
    std::vector<cudaEvent_t> free_events;
    double prof_ms[TVF_NUM_KERNELS] = {};
    int64_t prof_n[TVF_NUM_KERNELS] = {};
    // tvf_create_multi: further devices of a group handle (this context is member 0); the host-pointer pose entry points
    // shard B over the members, one host thread per device (experiments.m:91-143 is the loop that fans out)
    std::vector<tvf_context*> peers;
    // tvf_set_host_register: pin caller buffers that are pageable for the duration of a host-pointer pose call
    int host_register = 0;
    // pageable caller buffers (an mxArray's data): chunks travel through per-slot pinned staging buffers filled / drained by
    // a few host threads, so the DMA engines see pinned memory and the three-slot pipeline keeps overlapping
    int host_threads = 0;                 // 0 = automatic
    int group_size = 1;                   // members of the group handle this context belongs to
    void* stage[NSLOT] = {};
    size_t stage_cap[NSLOT] = {};
};

namespace {

int fail(tvf_handle_t h, int code, const std::string& msg) {
    if (h) h->err = msg; else g_create_error = msg;
    return code;
}

#define TVF_CK(call)                                                                              \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess)                                                                    \
            return fail(h, TVF_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));     \
    } while (0)

int ensure_arena(tvf_handle_t h, Slot& s, size_t bytes) {
    if (s.cap >= bytes) return TVF_OK;
    if (s.arena) { TVF_CK(cudaStreamSynchronize(s.stream)); TVF_CK(cudaFree(s.arena)); s.arena = nullptr; s.cap = 0; }
    const size_t want = bytes + (bytes >> 3);
    cudaError_t e = cudaMalloc(&s.arena, want);
    if (e != cudaSuccess) return fail(h, TVF_ERR_NOMEM, std::string("cudaMalloc(arena): ") + cudaGetErrorString(e));
    s.cap = want;
    return TVF_OK;
}

int ensure_scratch(tvf_handle_t h, int id, size_t bytes, void** out) {
    if (h->scratch_cap[id] < bytes) {
        if (h->scratch[id]) { TVF_CK(cudaDeviceSynchronize()); TVF_CK(cudaFree(h->scratch[id])); h->scratch[id] = nullptr; h->scratch_cap[id] = 0; }
        cudaError_t e = cudaMalloc(&h->scratch[id], bytes ? bytes : 8);
        if (e != cudaSuccess) return fail(h, TVF_ERR_NOMEM, std::string("cudaMalloc(scratch): ") + cudaGetErrorString(e));
        h->scratch_cap[id] = bytes ? bytes : 8;
    }
    *out = h->scratch[id];
    return TVF_OK;
}

// bump allocator over a slot arena (256-byte aligned pieces)
struct Carver {
    char* base; size_t off = 0;
    explicit Carver(char* b) : base(b) {}
    template <typename T> T* take(size_t count) {
        T* p = reinterpret_cast<T*>(base + off);
        off += (count * sizeof(T) + 255) & ~size_t(255);
        return p;
    }
};

struct ChunkBufs {
    double* in; double* calm; double* T; double* F; double* core; double* cand; int* votes; double* scale;
    double* Rt2; double* Rt3; double* reconst; double* repr; int* status; int* iters; int* iter_sum;
    // ba: the bundle adjustment of the chunk's poses (tvf_sweep_run_levels_ba)
    double* ba_Rt2; double* ba_Rt3; double* ba_X; double* ba_Xc; double* ba_repr; int* ba_iter; int* ba_status;
};

// per-problem bytes of the ba buffers: Rt2, Rt3, X, Xc, repr (+ iter, status in the last double)
inline size_t ba_chunk_bytes(int n) { return (size_t)(24 + 6 * n + 3) * sizeof(double); }

size_t carve(char* base, int n, int64_t C, bool host_io, bool calm_batched, bool ba, ChunkBufs* out) {
    Carver c(base);
    ChunkBufs b{};
    b.T = c.take<double>(27 * C);
    b.F = c.take<double>(18 * C);
    b.core = c.take<double>((size_t)CORE_WS_TFT * C);
    b.cand = c.take<double>((size_t)CAND_SIZE * C);
    b.votes = c.take<int>(10 * C);
    b.scale = c.take<double>(2 * C);
    b.status = c.take<int>(C);
    b.iters = c.take<int>(2 * C);
    b.iter_sum = c.take<int>(C);
    if (host_io) {
        b.in = c.take<double>((size_t)6 * n * C);
        b.calm = c.take<double>(calm_batched ? 27 * C : 27);
        b.Rt2 = c.take<double>(12 * C);
        b.Rt3 = c.take<double>(12 * C);
        b.reconst = c.take<double>((size_t)3 * n * C);
        b.repr = c.take<double>(C);
    }
    if (ba) {
        b.ba_Rt2 = c.take<double>(12 * C);
        b.ba_Rt3 = c.take<double>(12 * C);
        b.ba_X = c.take<double>((size_t)3 * n * C);
        b.ba_Xc = c.take<double>((size_t)3 * n * C);
        b.ba_repr = c.take<double>(C);
        b.ba_iter = c.take<int>(C);
        b.ba_status = c.take<int>(C);
    }
    if (out) *out = b;
    return c.off;
}

int64_t pick_chunk(tvf_handle_t h, int n, int64_t B, bool host_io, bool ba) {
    int64_t c = h->chunk_user > 0 ? h->chunk_user : (host_io ? DEFAULT_CHUNK : DEFAULT_CHUNK_DEV);
    if (h->chunk_user <= 0) {   // automatic: keep one slot's work space near ARENA_BUDGET
        size_t payload = (27 + 18 + CORE_WS_TFT + CAND_SIZE + 2) * 8 + 14 * 4;
        if (host_io) payload += (size_t)(6 * n + 27 + 24 + 3 * n + 1) * 8;
        if (ba) payload += ba_chunk_bytes(n);
        const int64_t fit = (int64_t)((host_io ? ARENA_BUDGET : 8 * ARENA_BUDGET) / payload);
        if (c > fit) c = fit;
    }
    if (c < 1) c = 1;
    if (c > B) c = B;
    return c;
}

enum Method { METHOD_TFT = 0, METHOD_F = 1, METHOD_OPTF = 2 };

cudaEvent_t get_event(tvf_handle_t h) {
    if (!h->free_events.empty()) { cudaEvent_t e = h->free_events.back(); h->free_events.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}

// launch `f` (one kernel) on `st`, bracketed by events when profiling is on
template <typename F>
void timed_launch(tvf_handle_t h, int id, cudaStream_t st, F f) {
    if (!h->profiling) { f(); h->launches += 1; return; }
    tvf_context::Ev ev{id, get_event(h), get_event(h)};
    cudaEventRecord(ev.a, st);
    f();
    cudaEventRecord(ev.b, st);
    h->events.push_back(ev);
    h->launches += 1;
}

int drain_events(tvf_handle_t h) {
    for (auto& ev : h->events) {
        TVF_CK(cudaEventSynchronize(ev.b));
        float ms = 0.f;
        TVF_CK(cudaEventElapsedTime(&ms, ev.a, ev.b));
        h->prof_ms[ev.id] += ms; h->prof_n[ev.id] += 1;
        h->free_events.push_back(ev.a); h->free_events.push_back(ev.b);
    }
    h->events.clear();
    return TVF_OK;
}

// kernels of one chunk; all pointers are device pointers
int run_pose_chunk(tvf_handle_t h, cudaStream_t st, Method method, const double* d_corresp, const double* d_calm,
                   int calm_batched, int n, int64_t Bc, double* d_T, double* d_F, double* d_core, double* d_cand, int* d_votes,
                   double* d_scale, double* d_Rt2, double* d_Rt3, double* d_reconst, double* d_repr, int* d_status,
                   int* d_iters = nullptr, int* d_iter_sum = nullptr) {
    CoreInput in{};
    in.p1 = d_corresp; in.p2 = nullptr; in.p3 = nullptr; in.packed = 1; in.rows = 2; in.n = n; in.B = Bc; in.normalize = 1;
    PoseTailArgs a{};
    a.corresp = d_corresp; a.calm = d_calm; a.calm_batched = calm_batched; a.n = n; a.B = Bc;
    a.cand = d_cand; a.votes = d_votes; a.scale = d_scale;
    a.Rt2 = d_Rt2; a.Rt3 = d_Rt3; a.reconst = d_reconst; a.repr_err = d_repr; a.status = d_status;
    const int sm = h->sm_count;
    if (method == METHOD_TFT) {
        bool large_done = false;
        if (n >= LARGE_N_MIN) {
            timed_launch(h, TVF_K_TFT_MOMENTS_LARGE, st, [&] {
                large_done = launch_tft_moments_large(d_corresp, n, Bc, 1, d_core, sm, st) != 0;
            });
            if (large_done)
                timed_launch(h, TVF_K_TFT_STAGE1_SOLVE, st, [&] { launch_tft_stage1_solve(Bc, d_core, d_status, sm, st); });
        }
        if (!large_done) {
            int need_solve = 0;
            timed_launch(h, TVF_K_TFT_STAGE1, st, [&] { need_solve = launch_tft_stage1(in, d_core, d_status, sm, st); });
            if (need_solve)
                timed_launch(h, TVF_K_TFT_STAGE1_SOLVE, st, [&] { launch_tft_stage1_solve(Bc, d_core, d_status, sm, st); });
        }
        timed_launch(h, TVF_K_TFT_EPIPOLES, st, [&] { launch_tft_epipoles(d_core, Bc, st); });
        timed_launch(h, TVF_K_TFT_STAGE2, st, [&] { launch_tft_stage2(in, d_core, d_T, nullptr, nullptr, d_status, sm, st); });
        timed_launch(h, TVF_K_CANDIDATES, st, [&] { launch_candidates(0, d_T, a, st); });
    } else if (method == METHOD_F) {
        timed_launch(h, TVF_K_F_STAGE1, st, [&] { launch_f_stage1(in, d_core, d_status, sm, st); });
        timed_launch(h, TVF_K_F_FINISH, st, [&] { launch_f_finish(d_core, 1, Bc, d_F, st); });
        timed_launch(h, TVF_K_CANDIDATES, st, [&] { launch_candidates(1, d_F, a, st); });
    } else {    // OptimFPoseEstimation.m:47-53: linearF start, Gauss-Helmert refinement, then the F pose tail
        timed_launch(h, TVF_K_F_STAGE1, st, [&] { launch_f_stage1(in, d_core, d_status, sm, st); });
        int ok = 1;
        timed_launch(h, TVF_K_OPTIMF_GH, st, [&] { ok = launch_optimf_gh(d_corresp, n, Bc, d_core, d_F, d_iters, d_status, sm, st); });
        if (!ok) return fail(h, TVF_ERR_ARG, "optimF: too many correspondences for the Gauss-Helmert kernel (see tvf_optim_f_max_n)");
        if (d_iter_sum) launch_sum_pairs(d_iters, Bc, d_iter_sum, st);
        timed_launch(h, TVF_K_CANDIDATES, st, [&] { launch_candidates(1, d_F, a, st); });
    }
    if (n >= TAIL_FUSED_MIN_N && n <= TAIL_FUSED_MAX_N) {
        timed_launch(h, TVF_K_TAIL_FUSED, st, [&] { launch_pose_tail_fused(a, sm, st); });
    } else {
        timed_launch(h, TVF_K_VOTES, st, [&] { launch_votes(a, sm, st); });
        timed_launch(h, TVF_K_SCALE, st, [&] { launch_scale(a, sm, st); });
        timed_launch(h, TVF_K_FINAL, st, [&] { launch_final(a, sm, st); });
    }
    if (method != METHOD_TFT && d_T != nullptr)
        timed_launch(h, TVF_K_TFT_FROM_POSE, st, [&] { launch_tft_from_pose(d_calm, calm_batched, d_Rt2, d_Rt3, Bc, d_T, st); });
    TVF_CK(cudaGetLastError());
    return TVF_OK;
}

int check_pose_args(tvf_handle_t h, const void* corresp, const void* calm, int n, int64_t B, Method m) {
    if (!h) return TVF_ERR_ARG;
    if (!corresp || !calm) return fail(h, TVF_ERR_ARG, "corresp/calm must not be NULL");
    if (B < 0 || n < 1) return fail(h, TVF_ERR_ARG, "need n >= 1 and B >= 0");
    if (m != METHOD_TFT && n < 8) return fail(h, TVF_ERR_TOO_FEW_POINTS, TVF_LINEARF_ERRMSG);
    if (m == METHOD_OPTF && n > optimf_max_n()) return fail(h, TVF_ERR_ARG, "optimF: too many correspondences for the Gauss-Helmert kernel (see tvf_optim_f_max_n)");
    return TVF_OK;
}

int count_flagged(const int32_t* st, int64_t B) {
    int64_t c = 0;
    for (int64_t i = 0; i < B; ++i) c += (st[i] != 0);
    return (int)(c > 0x7fffffff ? 0x7fffffff : c);
}

// copy `bytes` with `nthreads` host threads (a single memcpy stream reaches ~10 GB/s, far below what the PCIe link moves)
void par_memcpy(void* dst, const void* src, size_t bytes, int nthreads) {
    if (bytes == 0) return;
    if (nthreads <= 1 || bytes < (4u << 20)) { memcpy(dst, src, bytes); return; }
    const size_t part = ((bytes / (size_t)nthreads) + 4095) & ~size_t(4095);
    std::vector<std::thread> th;
    for (int t = 1; t < nthreads; ++t) {
        const size_t lo = (size_t)t * part;
        if (lo >= bytes) break;
        const size_t len = (lo + part <= bytes) ? part : bytes - lo;
        th.emplace_back([=] { memcpy((char*)dst + lo, (const char*)src + lo, len); });
    }
    memcpy(dst, src, part < bytes ? part : bytes);
    for (auto& t : th) t.join();
}

bool is_pageable(const void* p) {
    if (!p) return false;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeUnregistered;
}

int ensure_stage(tvf_handle_t h, int slot, size_t bytes) {
    if (h->stage_cap[slot] >= bytes) return TVF_OK;
    if (h->stage[slot]) { cudaFreeHost(h->stage[slot]); h->stage[slot] = nullptr; h->stage_cap[slot] = 0; }
    cudaError_t e = cudaHostAlloc(&h->stage[slot], bytes, cudaHostAllocPortable);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(h, TVF_ERR_NOMEM, std::string("cudaHostAlloc(staging): ") + cudaGetErrorString(e)); }
    h->stage_cap[slot] = bytes;
    return TVF_OK;
}

// outputs of a pose call (any may be null); `votes` = 10 int32 per problem: the 4 + 4 cheirality votes of
// R_t_from_TFT.m:91-104 in the reference's candidate order for the pairs (1,2) and (1,3), then the two NaN masks
struct PoseOut {
    double* Rt2; double* Rt3; double* reconst; double* T; double* repr_err; double* F21; double* F31;
    int32_t* iter; int32_t* votes; int32_t* status;
};

// caller buffers that are pageable get pinned for the duration of a call (tvf_set_host_register); RAII
struct HostPins {
    std::vector<void*> pinned;
    void add(const void* p, size_t bytes) {
        if (!p || bytes < (1u << 20)) return;
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return; }
        if (at.type != cudaMemoryTypeUnregistered) return;
        if (cudaHostRegister(const_cast<void*>(p), bytes, cudaHostRegisterPortable) == cudaSuccess) pinned.push_back(const_cast<void*>(p));
        else cudaGetLastError();
    }
    ~HostPins() { for (void* p : pinned) cudaHostUnregister(p); }
};

int pose_host_one(tvf_handle_t h, Method method, const double* corresp, const double* calm, int calm_batched, int n,
                  int64_t B, const PoseOut& o) {
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    const int64_t C = pick_chunk(h, n, B, true, false);
    const size_t need = carve(nullptr, n, C, true, calm_batched != 0, false, nullptr);
    std::vector<int32_t> st_tmp;
    int32_t* st_host = o.status;
    if (!st_host) { st_tmp.resize((size_t)B); st_host = st_tmp.data(); }
    // earlier asynchronous *_dev / sweep work of this handle may still be using slot 0's arena
    TVF_CK(cudaStreamSynchronize(h->slot[0].stream));
    if (h->use_user_stream) TVF_CK(cudaStreamSynchronize(h->user_stream));

    // Pageable caller memory (what a MEX gateway receives): cudaMemcpyAsync would fall back to synchronous copies through
    // the runtime's own bounce buffer and serialise the pipeline (measured 6.6e6 solves/s against 4.5e7 with pinned
    // buffers).  Instead every chunk goes through a pinned per-slot staging buffer that a few host threads fill and drain.
    const bool staged = !h->host_register && (size_t)B * 6 * n * sizeof(double) >= (size_t(4) << 20) &&
                        (is_pageable(corresp) || is_pageable(o.Rt2) || is_pageable(o.reconst) || is_pageable(o.T) || is_pageable(o.repr_err));
    int nthreads = h->host_threads;
    if (nthreads <= 0) {
        const int hw = (int)std::thread::hardware_concurrency();
        nthreads = hw / (h->group_size > 0 ? h->group_size : 1);
        nthreads = nthreads < 2 ? 2 : (nthreads > 8 ? 8 : nthreads);
    }
    struct Drain { void* dst; const void* src; size_t bytes; };
    std::vector<Drain> pending[NSLOT];
    auto drain = [&](int slot) {
        for (const Drain& d : pending[slot]) par_memcpy(d.dst, d.src, d.bytes, nthreads);
        pending[slot].clear();
    };
    const size_t in_bytes_max = (size_t)C * 6 * n * sizeof(double) + (calm_batched ? (size_t)C * 27 * sizeof(double) : 0);
    const size_t out_bytes_max = (size_t)C * ((24 + 3 * n + 27 + 1 + 18) * sizeof(double) + 12 * sizeof(int32_t)) + 16 * 256;   // + region alignment

    // Chunk schedule.  The call is bound by the host link (H2D of chunk i+1, kernels of chunk i and D2H of chunk i-1
    // overlap).  Quarter- and half-size chunks at both ends, meant to shorten the pipeline's fill and drain, were
    // measured SLOWER (4.31e7 vs 4.56e7 solves/s end to end at 1 M problems, profiles/r01_variants.md) and are off.
    const bool ramp = TVF_RAMP && B >= 6 * C && C >= 4096;
    int64_t done = 0; int ci = 0;
    int rc = TVF_OK;
    while (done < B) {
        const int64_t rem = B - done;
        int64_t Bc = (rem < C) ? rem : C;
        if (ramp) {
            const int64_t tail = C / 2 + C / 4;          // the last two chunks: C/2, then C/4
            if (rem > tail) {
                const int64_t body = rem - tail;
                if (ci == 0) Bc = C / 4;
                else if (ci == 1) Bc = C / 2;
                else if (body >= 2 * C) Bc = C;
                else if (body > C) Bc = (body + 1) / 2;
                else Bc = body;
            } else if (rem > C / 4) Bc = rem - C / 4;
            else Bc = rem;
        }
        const int si = ci % NSLOT;
        Slot& s = h->slot[si];
        TVF_CK(cudaStreamSynchronize(s.stream));        // slot reuse: its previous chunk (incl. D2H) is finished
        rc = ensure_arena(h, s, need); if (rc) return rc;
        ChunkBufs b; carve(s.arena, n, C, true, calm_batched != 0, false, &b);
        const double* src_in = corresp + done * 6 * n;
        const double* src_calm = calm + (calm_batched ? done * 27 : 0);
        char* stage_out = nullptr;
        if (staged) {
            drain(si);                                   // the slot's previous outputs leave the staging buffer first
            rc = ensure_stage(h, si, in_bytes_max + out_bytes_max); if (rc) return rc;
            char* st_in = (char*)h->stage[si];
            par_memcpy(st_in, src_in, (size_t)Bc * 6 * n * sizeof(double), nthreads);
            src_in = (const double*)st_in;
            if (calm_batched) {
                char* st_calm = st_in + (size_t)C * 6 * n * sizeof(double);
                memcpy(st_calm, src_calm, (size_t)Bc * 27 * sizeof(double));
                src_calm = (const double*)st_calm;
            }
            stage_out = st_in + in_bytes_max;
        }
        TVF_CK(cudaMemcpyAsync(b.in, src_in, (size_t)Bc * 6 * n * sizeof(double), cudaMemcpyHostToDevice, s.stream));
        // CalM travels on the chunk's own stream (ordered before the kernels that read it), shared 9x3 included
        TVF_CK(cudaMemcpyAsync(b.calm, src_calm, (size_t)(calm_batched ? Bc * 27 : 27) * sizeof(double), cudaMemcpyHostToDevice, s.stream));
        rc = run_pose_chunk(h, s.stream, method, b.in, b.calm, calm_batched, n, Bc,
                            (method == METHOD_TFT || o.T) ? b.T : nullptr, b.F, b.core, b.cand, b.votes, b.scale, b.Rt2, b.Rt3,
                            b.reconst, b.repr, b.status, b.iters, b.iter_sum);
        if (rc) return rc;
        // device -> host: straight into the caller's array, or into the staging buffer with a drain entry
        size_t soff = 0;
        auto back = [&](void* host_base, size_t per, const void* dev, size_t dev_pitch) -> cudaError_t {
            if (!host_base) return cudaSuccess;
            char* dst = (char*)host_base + (size_t)done * per;
            if (staged) {
                char* stg = stage_out + soff;
                soff += ((size_t)C * per + 255) & ~size_t(255);
                pending[si].push_back(Drain{dst, stg, (size_t)Bc * per});
                dst = stg;
            }
            if (dev_pitch == per) return cudaMemcpyAsync(dst, dev, (size_t)Bc * per, cudaMemcpyDeviceToHost, s.stream);
            return cudaMemcpy2DAsync(dst, per, dev, dev_pitch, per, (size_t)Bc, cudaMemcpyDeviceToHost, s.stream);
        };
        if (method == METHOD_OPTF) TVF_CK(back(o.iter, sizeof(int32_t), b.iter_sum, sizeof(int32_t)));
        TVF_CK(back(o.Rt2, 12 * sizeof(double), b.Rt2, 12 * sizeof(double)));
        TVF_CK(back(o.Rt3, 12 * sizeof(double), b.Rt3, 12 * sizeof(double)));
        TVF_CK(back(o.reconst, (size_t)3 * n * sizeof(double), b.reconst, (size_t)3 * n * sizeof(double)));
        TVF_CK(back(o.T, 27 * sizeof(double), b.T, 27 * sizeof(double)));
        TVF_CK(back(o.repr_err, sizeof(double), b.repr, sizeof(double)));
        TVF_CK(back(o.votes, 10 * sizeof(int32_t), b.votes, 10 * sizeof(int32_t)));
        if (method != METHOD_TFT) {
            TVF_CK(back(o.F21, 72, b.F, 144));
            TVF_CK(back(o.F31, 72, b.F + 9, 144));
        }
        TVF_CK(back(st_host, sizeof(int32_t), b.status, sizeof(int32_t)));
        done += Bc; ++ci;
    }
    for (int i = 0; i < NSLOT; ++i) {
        const int si = (ci + i) % NSLOT;                 // oldest chunk first
        TVF_CK(cudaStreamSynchronize(h->slot[si].stream));
        if (staged) drain(si);
    }
    return count_flagged(st_host, B);
}

// contiguous [lo, hi) of B problems for member g of G (remainder to the first members; same rule as sharding.shard_range)
inline void shard_of(int64_t B, int g, int G, int64_t* lo, int64_t* hi) {
    const int64_t base = B / G, rem = B % G;
    *lo = g * base + (g < rem ? g : rem);
    *hi = *lo + base + (g < rem ? 1 : 0);
}

int pose_host(tvf_handle_t h, Method method, const double* corresp, const double* calm, int calm_batched, int n,
              int64_t B, const PoseOut& o) {
    int rc = check_pose_args(h, corresp, calm, n, B, method);
    if (rc != TVF_OK) return rc;
    if (B == 0) return TVF_OK;
    HostPins pins;
    if (h->host_register) {
        TVF_CK(cudaSetDevice(h->device));
        pins.add(corresp, (size_t)B * 6 * n * 8);
        if (calm_batched) pins.add(calm, (size_t)B * 27 * 8);
        pins.add(o.Rt2, (size_t)B * 96); pins.add(o.Rt3, (size_t)B * 96); pins.add(o.reconst, (size_t)B * 3 * n * 8);
        pins.add(o.T, (size_t)B * 216); pins.add(o.repr_err, (size_t)B * 8); pins.add(o.votes, (size_t)B * 40);
        pins.add(o.F21, (size_t)B * 72); pins.add(o.F31, (size_t)B * 72); pins.add(o.status, (size_t)B * 4);
    }
    const int G = 1 + (int)h->peers.size();
    if (G == 1 || B < G) return pose_host_one(h, method, corresp, calm, calm_batched, n, B, o);
    // group handle: member g solves the contiguous range shard_of(B, g, G) on its own device from its own host thread;
    // problems are independent and a problem's result does not depend on its batch, so the outputs are bit-identical
    // to a single-device call
    std::vector<int> rcs((size_t)G, TVF_OK);
    auto run = [&](int g) {
        tvf_handle_t m = (g == 0) ? h : h->peers[(size_t)g - 1];
        int64_t lo, hi; shard_of(B, g, G, &lo, &hi);
        PoseOut s = o;
        if (s.Rt2) s.Rt2 += lo * 12;
        if (s.Rt3) s.Rt3 += lo * 12;
        if (s.reconst) s.reconst += lo * 3 * n;
        if (s.T) s.T += lo * 27;
        if (s.repr_err) s.repr_err += lo;
        if (s.F21) s.F21 += lo * 9;
        if (s.F31) s.F31 += lo * 9;
        if (s.iter) s.iter += lo;
        if (s.votes) s.votes += lo * 10;
        if (s.status) s.status += lo;
        m->chunk_user = h->chunk_user; m->host_threads = h->host_threads;
        rcs[(size_t)g] = pose_host_one(m, method, corresp + lo * 6 * n, calm + (calm_batched ? lo * 27 : 0), calm_batched, n, hi - lo, s);
    };
    std::vector<std::thread> th;
    for (int g = 1; g < G; ++g) th.emplace_back(run, g);
    run(0);
    for (auto& t : th) t.join();
    int64_t flagged = 0;
    for (int g = 0; g < G; ++g) {
        if (rcs[(size_t)g] < 0) {
            if (g > 0) h->err = "device " + std::to_string(h->peers[(size_t)g - 1]->device) + ": " + h->peers[(size_t)g - 1]->err;
            return rcs[(size_t)g];
        }
        flagged += rcs[(size_t)g];
    }
    cudaSetDevice(h->device);
    return (int)(flagged > 0x7fffffff ? 0x7fffffff : flagged);
}

int pose_dev(tvf_handle_t h, Method method, const double* corresp, const double* calm, int calm_batched, int n,
             int64_t B, const PoseOut& o) {
    int rc = check_pose_args(h, corresp, calm, n, B, method);
    if (rc != TVF_OK) return rc;
    // the kernels read the correspondences with 128-bit loads and bulk asynchronous copies: 16-byte alignment (every
    // cudaMalloc'ed buffer and every problem boundary inside one satisfies it: a problem is 48 n bytes)
    if ((reinterpret_cast<uintptr_t>(corresp) & 15u) != 0) return fail(h, TVF_ERR_ARG, "device pointer `corresp` must be 16-byte aligned");
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    Slot& s = h->slot[0];
    cudaStream_t st = h->use_user_stream ? h->user_stream : s.stream;
    const int64_t C = pick_chunk(h, n, B, false, false);
    // internal buffers only; Rt2/Rt3 are needed internally by the F method's TFT_from_P, so stage them if absent
    const size_t need = carve(nullptr, n, C, false, false, false, nullptr) + (size_t)(24 * C) * sizeof(double) + 512;
    rc = ensure_arena(h, s, need); if (rc) return rc;
    ChunkBufs b; const size_t used = carve(s.arena, n, C, false, false, false, &b);
    double* tmpRt2 = reinterpret_cast<double*>(s.arena + used);
    double* tmpRt3 = tmpRt2 + 12 * C;
    for (int64_t done = 0; done < B; done += C) {
        const int64_t Bc = (B - done < C) ? (B - done) : C;
        double* dT = o.T ? o.T + done * 27 : (method == METHOD_TFT ? b.T : nullptr);
        double* dRt2 = o.Rt2 ? o.Rt2 + done * 12 : tmpRt2;
        double* dRt3 = o.Rt3 ? o.Rt3 + done * 12 : tmpRt3;
        rc = run_pose_chunk(h, st, method, corresp + done * 6 * n, calm + (calm_batched ? done * 27 : 0), calm_batched, n,
                            Bc, dT, b.F, b.core, b.cand, o.votes ? o.votes + done * 10 : b.votes, b.scale, dRt2, dRt3,
                            o.reconst ? o.reconst + done * 3 * n : nullptr, o.repr_err ? o.repr_err + done : nullptr,
                            o.status ? o.status + done : b.status, b.iters, o.iter ? o.iter + done : nullptr);
        if (rc) return rc;
        if (method != METHOD_TFT && o.F21)
            TVF_CK(cudaMemcpy2DAsync(o.F21 + done * 9, 72, b.F, 144, 72, (size_t)Bc, cudaMemcpyDeviceToDevice, st));
        if (method != METHOD_TFT && o.F31)
            TVF_CK(cudaMemcpy2DAsync(o.F31 + done * 9, 72, b.F + 9, 144, 72, (size_t)Bc, cudaMemcpyDeviceToDevice, st));
    }
    return TVF_OK;
}

// ---- bundle adjustment (tvf_bundle_adjust[_dev]) and its covariance (tvf_ba_covariance[_dev]) ------------------------
// one call's arrays (host or device pointers).  Adjustment: outputs may be null except Rt2 / Rt3.  Covariance (cov):
// the state is Rt2_0, Rt3_0, X0 (all required) and the outputs cov_cam, cov_pts, sigma2, status may be null.
struct BaIo {
    const double* corresp; const double* calm; int calm_batched; int n;
    const double* Rt2_0; const double* Rt3_0; const double* X0;
    double* Rt2; double* Rt3; double* X; double* repr; int32_t* iter; int32_t* status;
    bool cov; double* cov_cam; double* cov_pts; double* sigma2;
    BaIo shifted(int64_t lo) const {           // problems [lo, ...)
        BaIo s = *this;
        s.corresp += lo * 6 * n;
        if (calm_batched) s.calm += lo * 27;
        s.Rt2_0 += lo * 12; s.Rt3_0 += lo * 12;
        if (s.Rt2) s.Rt2 += lo * 12;
        if (s.Rt3) s.Rt3 += lo * 12;
        if (s.X0) s.X0 += lo * 3 * n;
        if (s.X) s.X += lo * 3 * n;
        if (s.repr) s.repr += lo;
        if (s.iter) s.iter += lo;
        if (s.status) s.status += lo;
        if (s.cov_cam) s.cov_cam += lo * 144;
        if (s.cov_pts) s.cov_pts += lo * 9 * n;
        if (s.sigma2) s.sigma2 += lo;
        return s;
    }
};

int check_ba_args(tvf_handle_t h, const BaIo& io, int64_t B) {
    if (!h) return TVF_ERR_ARG;
    if (io.cov) {
        if (!io.corresp || !io.calm || !io.Rt2_0 || !io.Rt3_0 || !io.X0)
            return fail(h, TVF_ERR_ARG, "ba_covariance: corresp, calm, Rt2, Rt3 and reconst must not be NULL");
    } else if (!io.corresp || !io.calm || !io.Rt2_0 || !io.Rt3_0 || !io.Rt2 || !io.Rt3) {
        return fail(h, TVF_ERR_ARG, "bundle_adjust: corresp, calm, Rt2_0, Rt3_0, Rt2 and Rt3 must not be NULL");
    }
    if (B < 0) return fail(h, TVF_ERR_ARG, "bundle_adjust: B >= 0");
    if (io.n < 4) return fail(h, TVF_ERR_ARG, "bundle_adjust: needs n >= 4 points (11 + 3n unknowns, 6n residuals)");
    return TVF_OK;
}

// per-problem device bytes of a chunk: host_io -> inputs and outputs too; the adjustment always has its two point buffers
size_t ba_bytes_per_problem(int n, bool host_io, bool cov) {
    if (cov) return host_io ? (size_t)(6 * n + 27 + 24 + 3 * n + 144 + 9 * n + 1 + 1) * sizeof(double) : 0;
    size_t b = (size_t)2 * 3 * n * sizeof(double);
    if (host_io) b += (size_t)(6 * n + 27 + 24 + 3 * n + 24 + 1) * sizeof(double) + 2 * sizeof(int32_t);
    return b;
}

int64_t pick_chunk_ba(tvf_handle_t h, int n, int64_t B, bool host_io, bool cov = false) {
    int64_t c = h->chunk_user > 0 ? h->chunk_user : (host_io ? DEFAULT_CHUNK : DEFAULT_CHUNK_DEV);
    const size_t per = ba_bytes_per_problem(n, host_io, cov);
    if (h->chunk_user <= 0 && per > 0) {
        const int64_t fit = (int64_t)((host_io ? ARENA_BUDGET : 8 * ARENA_BUDGET) / per);
        if (c > fit) c = fit;
    }
    if (c < 1) c = 1;
    if (c > B) c = B;
    return c;
}

// device copies of one host chunk of C problems in a slot arena (base = nullptr: size only)
// (the covariance's chunk: inputs, cov_cam and cov_pts when the caller wants them, sigma2, status)
size_t carve_ba(char* base, int n, int64_t C, const BaIo& io, BaIo* d, double** Xc) {
    Carver c(base);
    *d = BaIo{};
    d->cov = io.cov;
    d->corresp = c.take<double>((size_t)6 * n * C); d->calm = c.take<double>(io.calm_batched ? 27 * C : 27);
    d->calm_batched = io.calm_batched; d->n = n;
    d->Rt2_0 = c.take<double>(12 * C); d->Rt3_0 = c.take<double>(12 * C); d->X0 = c.take<double>((size_t)3 * n * C);
    if (io.cov) {
        d->cov_cam = io.cov_cam ? c.take<double>(144 * C) : nullptr;
        d->cov_pts = io.cov_pts ? c.take<double>((size_t)9 * n * C) : nullptr;
        d->sigma2 = c.take<double>(C); d->status = c.take<int32_t>(C);
        *Xc = nullptr;
        return c.off;
    }
    d->Rt2 = c.take<double>(12 * C); d->Rt3 = c.take<double>(12 * C); d->X = c.take<double>((size_t)3 * n * C);
    *Xc = c.take<double>((size_t)3 * n * C);
    d->repr = c.take<double>(C); d->iter = c.take<int32_t>(C); d->status = c.take<int32_t>(C);
    return c.off;
}

int ba_launch(tvf_handle_t h, cudaStream_t st, const BaIo& d, int64_t Bc, double* Xc) {
    int ok;
    if (d.cov) {
        BaCovArgs a{d.corresp, d.calm, d.calm_batched, d.n, Bc, d.Rt2_0, d.Rt3_0, d.X0, d.cov_cam, d.cov_pts, d.sigma2, d.status};
        ok = launch_ba_covariance(a, st);
    } else {
        BaArgs a{d.corresp, d.calm, d.calm_batched, d.n, Bc, d.Rt2_0, d.Rt3_0, d.X0, d.Rt2, d.Rt3, d.X, Xc, d.repr, d.iter, d.status};
        ok = launch_bundle_adjust(a, st);
    }
    h->launches += 1;
    if (!ok) {
        cudaError_t e = cudaGetLastError();
        return fail(h, TVF_ERR_CUDA, std::string(d.cov ? "ba_covariance_kernel: " : "bundle_adjust_kernel: ") + cudaGetErrorString(e));
    }
    return TVF_OK;
}

int ba_host_one(tvf_handle_t h, const BaIo& io, int64_t B) {
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    const int n = io.n;
    const int64_t C = pick_chunk_ba(h, n, B, true, io.cov);
    std::vector<int32_t> st_tmp;
    int32_t* st_host = io.status;
    if (!st_host) { st_tmp.resize((size_t)B); st_host = st_tmp.data(); }
    TVF_CK(cudaStreamSynchronize(h->slot[0].stream));
    if (h->use_user_stream) TVF_CK(cudaStreamSynchronize(h->user_stream));
    int64_t done = 0; int ci = 0; int rc;
    while (done < B) {
        const int64_t Bc = (B - done < C) ? (B - done) : C;
        Slot& s = h->slot[ci % NSLOT];
        TVF_CK(cudaStreamSynchronize(s.stream));            // the slot's previous chunk (with its copies back) is done
        BaIo d{}; double* Xc;
        rc = ensure_arena(h, s, carve_ba(nullptr, n, C, io, &d, &Xc)); if (rc) return rc;
        carve_ba(s.arena, n, C, io, &d, &Xc);
        double* x0 = const_cast<double*>(d.X0);
        if (!io.X0) d.X0 = nullptr;
        double* in = const_cast<double*>(d.corresp); double* calm = const_cast<double*>(d.calm);
        double* r2 = const_cast<double*>(d.Rt2_0); double* r3 = const_cast<double*>(d.Rt3_0);
        const BaIo hio = io.shifted(done);
        auto up = [&](void* dst, const void* src, size_t bytes) { return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, s.stream); };
        auto down = [&](void* dst, const void* src, size_t bytes) {
            return dst ? cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, s.stream) : cudaSuccess;
        };
        TVF_CK(up(in, hio.corresp, (size_t)Bc * 6 * n * sizeof(double)));
        TVF_CK(up(calm, hio.calm, (size_t)(io.calm_batched ? Bc * 27 : 27) * sizeof(double)));
        TVF_CK(up(r2, hio.Rt2_0, (size_t)Bc * 12 * sizeof(double)));
        TVF_CK(up(r3, hio.Rt3_0, (size_t)Bc * 12 * sizeof(double)));
        if (io.X0) TVF_CK(up(x0, hio.X0, (size_t)Bc * 3 * n * sizeof(double)));
        rc = ba_launch(h, s.stream, d, Bc, Xc); if (rc) return rc;
        if (io.cov) {
            TVF_CK(down(hio.cov_cam, d.cov_cam, (size_t)Bc * 144 * sizeof(double)));
            TVF_CK(down(hio.cov_pts, d.cov_pts, (size_t)Bc * 9 * n * sizeof(double)));
            TVF_CK(down(hio.sigma2, d.sigma2, (size_t)Bc * sizeof(double)));
        } else {
            TVF_CK(down(hio.Rt2, d.Rt2, (size_t)Bc * 12 * sizeof(double)));
            TVF_CK(down(hio.Rt3, d.Rt3, (size_t)Bc * 12 * sizeof(double)));
            TVF_CK(down(hio.X, d.X, (size_t)Bc * 3 * n * sizeof(double)));
            TVF_CK(down(hio.repr, d.repr, (size_t)Bc * sizeof(double)));
            TVF_CK(down(hio.iter, d.iter, (size_t)Bc * sizeof(int32_t)));
        }
        TVF_CK(down(st_host + done, d.status, (size_t)Bc * sizeof(int32_t)));
        done += Bc; ++ci;
    }
    for (int i = 0; i < NSLOT; ++i) TVF_CK(cudaStreamSynchronize(h->slot[i].stream));
    return count_flagged(st_host, B);
}

// host pointers; a group handle shards B exactly as pose_host does (results bit-identical to one device)
int ba_host(tvf_handle_t h, const BaIo& io, int64_t B) {
    int rc = check_ba_args(h, io, B);
    if (rc != TVF_OK) return rc;
    if (B == 0) return TVF_OK;
    const int G = 1 + (int)h->peers.size();
    if (G == 1 || B < G) return ba_host_one(h, io, B);
    std::vector<int> rcs((size_t)G, TVF_OK);
    auto run = [&](int g) {
        tvf_handle_t m = (g == 0) ? h : h->peers[(size_t)g - 1];
        int64_t lo, hi; shard_of(B, g, G, &lo, &hi);
        m->chunk_user = h->chunk_user;
        rcs[(size_t)g] = ba_host_one(m, io.shifted(lo), hi - lo);
    };
    std::vector<std::thread> th;
    for (int g = 1; g < G; ++g) th.emplace_back(run, g);
    run(0);
    for (auto& t : th) t.join();
    int64_t flagged = 0;
    for (int g = 0; g < G; ++g) {
        if (rcs[(size_t)g] < 0) {
            if (g > 0) h->err = "device " + std::to_string(h->peers[(size_t)g - 1]->device) + ": " + h->peers[(size_t)g - 1]->err;
            return rcs[(size_t)g];
        }
        flagged += rcs[(size_t)g];
    }
    cudaSetDevice(h->device);
    return (int)(flagged > 0x7fffffff ? 0x7fffffff : flagged);
}

// device pointers, asynchronous on the handle's stream
int ba_dev(tvf_handle_t h, const BaIo& io, int64_t B) {
    int rc = check_ba_args(h, io, B);
    if (rc != TVF_OK) return rc;
    if ((reinterpret_cast<uintptr_t>(io.corresp) & 15u) != 0) return fail(h, TVF_ERR_ARG, "device pointer `corresp` must be 16-byte aligned");
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    Slot& s = h->slot[0];
    cudaStream_t st = h->use_user_stream ? h->user_stream : s.stream;
    const int64_t C = pick_chunk_ba(h, io.n, B, false, io.cov);
    double* Xc = nullptr; double* Xw = nullptr;
    if (!io.cov) {                                           // the adjustment's work space; the covariance needs none
        const size_t pts = (size_t)3 * io.n * C;
        rc = ensure_arena(h, s, 2 * pts * sizeof(double) + 512); if (rc) return rc;
        Carver c(s.arena);
        Xc = c.take<double>(pts);
        Xw = c.take<double>(pts);
    }
    for (int64_t done = 0; done < B; done += C) {
        const int64_t Bc = (B - done < C) ? (B - done) : C;
        BaIo d = io.shifted(done);
        if (!io.cov && !io.X) d.X = Xw;
        rc = ba_launch(h, st, d, Bc, Xc); if (rc) return rc;
    }
    return TVF_OK;
}

// small helper for the stand-alone functions: upload, run, download on slot 0
struct Up {
    tvf_handle_t h; cudaStream_t st; int rc = TVF_OK; int next = 1;
    explicit Up(tvf_handle_t hh) : h(hh), st(hh->slot[0].stream) {}
    template <typename T> T* in(const T* host, size_t count) {
        if (rc) return nullptr;
        void* p; rc = ensure_scratch(h, next++, count * sizeof(T), &p);
        if (rc) return nullptr;
        if (host && count) {
            cudaError_t e = cudaMemcpyAsync(p, host, count * sizeof(T), cudaMemcpyHostToDevice, st);
            if (e != cudaSuccess) { rc = fail(h, TVF_ERR_CUDA, cudaGetErrorString(e)); return nullptr; }
        }
        return (T*)p;
    }
    template <typename T> T* out(size_t count) { return in<T>(nullptr, count); }
    template <typename T> void back(T* host, const T* dev, size_t count) {
        if (rc || !host) return;
        cudaError_t e = cudaMemcpyAsync(host, dev, count * sizeof(T), cudaMemcpyDeviceToHost, st);
        if (e != cudaSuccess) rc = fail(h, TVF_ERR_CUDA, cudaGetErrorString(e));
    }
    int finish() {
        if (rc) return rc;
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) return fail(h, TVF_ERR_CUDA, cudaGetErrorString(e));
        return TVF_OK;
    }
};

// dense, dependency-free-ish DFMA loop: the FP64 roofline denominator measured on this very device
__global__ void __launch_bounds__(256) fp64_peak_kernel(double* out, int iters, double seed) {
    double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 0.999999, c = 1e-6;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
        a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
    const double r = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
    if (r == 123.456) out[0] = r;      // never true; keeps the loop alive
}

}  // namespace

// =========================================================================== C ABI
extern "C" {

int tvf_version(void) { return 201; }

int tvf_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int tvf_create(tvf_handle_t* out, int device) {
    tvf_handle_t h = nullptr;
    if (!out) return fail(nullptr, TVF_ERR_ARG, "out must not be NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, TVF_ERR_CUDA, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                                               " (libtvf has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(nullptr, TVF_ERR_ARG, "device index out of range");
    TVF_CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    TVF_CK(cudaGetDeviceProperties(&prop, device));
    h = new tvf_context();
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    for (int i = 0; i < NSLOT; ++i) {
        e = cudaStreamCreateWithFlags(&h->slot[i].stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) { std::string m = cudaGetErrorString(e); tvf_destroy(h); return fail(nullptr, TVF_ERR_CUDA, m); }
    }
    *out = h;
    return TVF_OK;
}

void tvf_destroy(tvf_handle_t h) {
    if (!h) return;
    for (tvf_handle_t m : h->peers) tvf_destroy(m);
    h->peers.clear();
    cudaSetDevice(h->device);
    for (int i = 0; i < NSLOT; ++i) {
        if (h->slot[i].stream) { cudaStreamSynchronize(h->slot[i].stream); cudaStreamDestroy(h->slot[i].stream); }
        if (h->slot[i].arena) cudaFree(h->slot[i].arena);
        if (h->stage[i]) cudaFreeHost(h->stage[i]);
    }
    for (int i = 0; i < NSCRATCH; ++i)
        if (h->scratch[i]) cudaFree(h->scratch[i]);
    for (auto& ev : h->events) { cudaEventDestroy(ev.a); cudaEventDestroy(ev.b); }
    for (auto e : h->free_events) cudaEventDestroy(e);
    delete h;
}

int tvf_create_multi(tvf_handle_t* out, const int* devices, int n_dev) {
    if (!out) return fail(nullptr, TVF_ERR_ARG, "out must not be NULL");
    *out = nullptr;
    if (!devices || n_dev < 1) return fail(nullptr, TVF_ERR_ARG, "need at least one device");
    tvf_handle_t h = nullptr;
    int rc = tvf_create(&h, devices[0]);
    if (rc != TVF_OK) return rc;
    for (int i = 1; i < n_dev; ++i) {
        tvf_handle_t m = nullptr;
        rc = tvf_create(&m, devices[i]);
        if (rc != TVF_OK) { tvf_destroy(h); return rc; }
        h->peers.push_back(m);
    }
    h->group_size = n_dev;
    for (tvf_handle_t m : h->peers) m->group_size = n_dev;
    cudaSetDevice(h->device);
    *out = h;
    return TVF_OK;
}

int tvf_num_devices(tvf_handle_t h) { return h ? 1 + (int)h->peers.size() : 0; }

int tvf_set_host_threads(tvf_handle_t h, int threads) {
    if (!h || threads < 0) return TVF_ERR_ARG;
    h->host_threads = threads;
    return TVF_OK;
}

int tvf_set_host_register(tvf_handle_t h, int on) {
    if (!h) return TVF_ERR_ARG;
    h->host_register = on ? 1 : 0;
    return TVF_OK;
}

const char* tvf_last_error(tvf_handle_t h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int tvf_device(tvf_handle_t h) { return h ? h->device : -1; }

int tvf_set_chunk(tvf_handle_t h, int64_t problems) {
    if (!h || problems < 0) return TVF_ERR_ARG;
    h->chunk_user = problems;
    return TVF_OK;
}

int tvf_set_stream(tvf_handle_t h, void* cuda_stream) {
    if (!h) return TVF_ERR_ARG;
    h->user_stream = (cudaStream_t)cuda_stream;   // NULL is the legacy default stream
    h->use_user_stream = true;
    return TVF_OK;
}

int tvf_use_own_stream(tvf_handle_t h) {
    if (!h) return TVF_ERR_ARG;
    h->use_user_stream = false;
    return TVF_OK;
}

int tvf_synchronize(tvf_handle_t h) {
    if (!h) return TVF_ERR_ARG;
    TVF_CK(cudaSetDevice(h->device));
    for (int i = 0; i < NSLOT; ++i) TVF_CK(cudaStreamSynchronize(h->slot[i].stream));
    if (h->use_user_stream) TVF_CK(cudaStreamSynchronize(h->user_stream));
    return TVF_OK;
}

// CPUs of the NUMA node the current device hangs off (sysfs local_cpulist of its PCI function) that this thread may run
// on; false when that cannot be determined (then nothing is changed).
static bool device_local_cpus(cpu_set_t* out) {
    int dev = 0;
    char bus[32] = {0};
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetPCIBusId(bus, (int)sizeof(bus), dev) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    for (char* c = bus; *c; ++c) if (*c >= 'A' && *c <= 'F') *c = (char)(*c - 'A' + 'a');      // sysfs names are lower case
    const std::string path = std::string("/sys/bus/pci/devices/") + bus + "/local_cpulist";
    FILE* f = fopen(path.c_str(), "r");
    if (!f) return false;
    char line[4096] = {0};
    const bool got = fgets(line, sizeof(line), f) != nullptr;
    fclose(f);
    if (!got) return false;
    cpu_set_t allowed;
    if (sched_getaffinity(0, sizeof(allowed), &allowed) != 0) return false;
    CPU_ZERO(out);
    int n_set = 0;
    for (const char* c = line; *c;) {                                   // "0-31,64-95"
        char* end = nullptr;
        long a = strtol(c, &end, 10);
        if (end == c) break;
        long b = a;
        c = end;
        if (*c == '-') { b = strtol(c + 1, &end, 10); if (end == c + 1) break; c = end; }
        for (long i = a; i <= b && i < CPU_SETSIZE; ++i)
            if (i >= 0 && CPU_ISSET((int)i, &allowed)) { CPU_SET((int)i, out); ++n_set; }
        while (*c == ',' || *c == ' ' || *c == '\n') ++c;
    }
    return n_set > 0;
}

// Pinned host memory on the NUMA node of the current CUDA device: the pages are placed where the allocating thread runs,
// and a buffer on the far socket costs the host-pointer entry points ~15 % of their link bandwidth.  The calling thread's
// CPU affinity is narrowed to the device-local CPUs for the duration of the allocation and then restored.
void* tvf_host_alloc(size_t bytes) {
    cpu_set_t saved, local;
    const bool have_saved = sched_getaffinity(0, sizeof(saved), &saved) == 0;
    const bool moved = have_saved && device_local_cpus(&local) && sched_setaffinity(0, sizeof(local), &local) == 0;
    void* p = nullptr;
    const cudaError_t e = cudaMallocHost(&p, bytes ? bytes : 1);
    if (e == cudaSuccess && p) memset(p, 0, bytes ? bytes : 1);       // first touch on the local node
    if (moved) sched_setaffinity(0, sizeof(saved), &saved);
    if (e != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}

void tvf_host_free(void* p) { if (p) cudaFreeHost(p); }

int64_t tvf_launch_count(tvf_handle_t h) {
    if (!h) return 0;
    int64_t n = h->launches;
    for (tvf_handle_t m : h->peers) n += m->launches;
    return n;
}

int tvf_profile_enable(tvf_handle_t h, int on) {
    if (!h) return TVF_ERR_ARG;
    if (!on && h->profiling) { int rc = drain_events(h); if (rc) return rc; }
    h->profiling = on != 0;
    return TVF_OK;
}

int tvf_profile_reset(tvf_handle_t h) {
    if (!h) return TVF_ERR_ARG;
    int rc = drain_events(h); if (rc) return rc;
    for (int i = 0; i < TVF_NUM_KERNELS; ++i) { h->prof_ms[i] = 0.0; h->prof_n[i] = 0; }
    return TVF_OK;
}

int tvf_profile_read(tvf_handle_t h, double* total_ms, int64_t* launches) {
    if (!h || !total_ms || !launches) return TVF_ERR_ARG;
    int rc = drain_events(h); if (rc) return rc;
    for (int i = 0; i < TVF_NUM_KERNELS; ++i) { total_ms[i] = h->prof_ms[i]; launches[i] = h->prof_n[i]; }
    return TVF_OK;
}

double tvf_fp64_peak_tflops(tvf_handle_t h) {
    if (!h) return -1.0;
    if (cudaSetDevice(h->device) != cudaSuccess) return -1.0;
    cudaStream_t st = h->slot[0].stream;
    void* p = nullptr;
    if (ensure_scratch(h, NSCRATCH - 1, 64, &p) != TVF_OK) return -1.0;
    const int iters = 1 << 15, blocks = h->sm_count * 8;
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    double best = 0.0;
    for (int rep = 0; rep < 4; ++rep) {
        cudaEventRecord(a, st);
        fp64_peak_kernel<<<blocks, 256, 0, st>>>((double*)p, iters, 1.0 + rep);
        cudaEventRecord(b, st);
        if (cudaEventSynchronize(b) != cudaSuccess) { best = -1.0; break; }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, a, b);
        const double tf = (double)blocks * 256.0 * iters * 8.0 * 2.0 / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;     // first repetition is warm-up
    }
    cudaEventDestroy(a); cudaEventDestroy(b);
    return best;
}

const char* tvf_kernel_name(int id) {
    static const char* names[TVF_NUM_KERNELS] = {"tft_stage1_kernel", "tft_epipoles_kernel", "tft_stage2_kernel",
                                                 "f_stage1_kernel", "f_finish_kernel", "candidates_kernel",
                                                 "votes_kernel", "scale_kernel", "final_kernel", "tft_from_pose_kernel",
                                                 "pose_tail_fused_kernel", "tft_moments_large_kernel",
                                                 "tft_stage1_solve_kernel", "optimf_gh_kernel"};
    return (id >= 0 && id < TVF_NUM_KERNELS) ? names[id] : "";
}

static bool method_of(int id, Method* m) {
    if (id == 1) { *m = METHOD_TFT; return true; }
    if (id == 7) { *m = METHOD_F; return true; }
    if (id == 8) { *m = METHOD_OPTF; return true; }
    return false;
}

static PoseOut pose_out_of(const tvf_pose_out* o) {
    PoseOut p{};
    if (o) { p.Rt2 = o->Rt2; p.Rt3 = o->Rt3; p.reconst = o->reconst; p.T = o->T; p.repr_err = o->repr_err; p.F21 = o->F21;
             p.F31 = o->F31; p.iter = o->iter; p.votes = o->votes; p.status = o->status; }
    return p;
}

int tvf_pose(tvf_handle_t h, int method, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
             const tvf_pose_out* out) {
    Method m;
    if (!h) return TVF_ERR_ARG;
    if (!method_of(method, &m)) return fail(h, TVF_ERR_ARG, "method must be 1 (linear TFT), 7 (linear F) or 8 (optimal F)");
    return pose_host(h, m, corresp, calm, calm_batched, n, B, pose_out_of(out));
}

int tvf_pose_dev(tvf_handle_t h, int method, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                 const tvf_pose_out* out) {
    Method m;
    if (!h) return TVF_ERR_ARG;
    if (!method_of(method, &m)) return fail(h, TVF_ERR_ARG, "method must be 1 (linear TFT), 7 (linear F) or 8 (optimal F)");
    return pose_dev(h, m, corresp, calm, calm_batched, n, B, pose_out_of(out));
}

int tvf_linear_tft_pose(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                        double* Rt2, double* Rt3, double* reconst, double* T, double* repr_err, int32_t* status) {
    return pose_host(h, METHOD_TFT, corresp, calm, calm_batched, n, B, PoseOut{Rt2, Rt3, reconst, T, repr_err, nullptr, nullptr, nullptr, nullptr, status});
}

int tvf_linear_f_pose(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                      double* Rt2, double* Rt3, double* reconst, double* T, double* repr_err, double* F21, double* F31,
                      int32_t* status) {
    return pose_host(h, METHOD_F, corresp, calm, calm_batched, n, B, PoseOut{Rt2, Rt3, reconst, T, repr_err, F21, F31, nullptr, nullptr, status});
}

int tvf_optim_f_pose(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                     double* Rt2, double* Rt3, double* reconst, double* T, double* repr_err, double* F21, double* F31,
                     int32_t* iter, int32_t* status) {
    return pose_host(h, METHOD_OPTF, corresp, calm, calm_batched, n, B, PoseOut{Rt2, Rt3, reconst, T, repr_err, F21, F31, iter, nullptr, status});
}

int tvf_optim_f_pose_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                         double* Rt2, double* Rt3, double* reconst, double* T, double* repr_err, double* F21, double* F31,
                         int32_t* iter, int32_t* status) {
    return pose_dev(h, METHOD_OPTF, corresp, calm, calm_batched, n, B, PoseOut{Rt2, Rt3, reconst, T, repr_err, F21, F31, iter, nullptr, status});
}

int tvf_optim_f_max_n(void) { return optimf_max_n(); }

int tvf_linear_tft_pose_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                            double* Rt2, double* Rt3, double* reconst, double* T, double* repr_err, int32_t* status) {
    return pose_dev(h, METHOD_TFT, corresp, calm, calm_batched, n, B, PoseOut{Rt2, Rt3, reconst, T, repr_err, nullptr, nullptr, nullptr, nullptr, status});
}

int tvf_linear_f_pose_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                          double* Rt2, double* Rt3, double* reconst, double* T, double* repr_err, double* F21, double* F31,
                          int32_t* status) {
    return pose_dev(h, METHOD_F, corresp, calm, calm_batched, n, B, PoseOut{Rt2, Rt3, reconst, T, repr_err, F21, F31, nullptr, nullptr, status});
}

int tvf_linear_tft(tvf_handle_t h, const double* p1, const double* p2, const double* p3, int rows, int n, int64_t B,
                   double* T, double* P2, double* P3, int32_t* status) {
    if (!h) return TVF_ERR_ARG;
    if (!p1 || !p2 || !p3 || !T) return fail(h, TVF_ERR_ARG, "p1,p2,p3,T must not be NULL");
    if ((rows != 2 && rows != 3) || n < 1 || B < 0) return fail(h, TVF_ERR_ARG, "rows must be 2 or 3, n >= 1, B >= 0");
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    Up u(h);
    const size_t np = (size_t)rows * n * B;
    CoreInput in{};
    in.p1 = u.in(p1, np); in.p2 = u.in(p2, np); in.p3 = u.in(p3, np);
    in.packed = 0; in.rows = rows; in.n = n; in.B = B; in.normalize = 0;
    double* dT = u.out<double>(27 * (size_t)B);
    double* dP2 = u.out<double>(12 * (size_t)B);
    double* dP3 = u.out<double>(12 * (size_t)B);
    int* dst = u.out<int>((size_t)B);
    double* dws = u.out<double>((size_t)CORE_WS_TFT * B);
    if (u.rc) return u.rc;
    if (launch_tft_stage1(in, dws, dst, h->sm_count, u.st)) { launch_tft_stage1_solve(B, dws, dst, h->sm_count, u.st); h->launches += 1; }
    launch_tft_epipoles(dws, B, u.st);
    launch_tft_stage2(in, dws, dT, dP2, dP3, dst, h->sm_count, u.st);
    h->launches += 3;
    std::vector<int32_t> tmp; int32_t* sth = status;
    if (!sth) { tmp.resize((size_t)B); sth = tmp.data(); }
    u.back(T, dT, 27 * (size_t)B); u.back(P2, dP2, 12 * (size_t)B); u.back(P3, dP3, 12 * (size_t)B);
    u.back(sth, (const int32_t*)dst, (size_t)B);
    int rc = u.finish();
    return rc ? rc : count_flagged(sth, B);
}

int tvf_linear_f(tvf_handle_t h, const double* p1, const double* p2, int rows, int n, int64_t B, double* F,
                 int32_t* status) {
    if (!h) return TVF_ERR_ARG;
    if (!p1 || !p2 || !F) return fail(h, TVF_ERR_ARG, "p1,p2,F must not be NULL");
    if ((rows != 2 && rows != 3) || B < 0) return fail(h, TVF_ERR_ARG, "rows must be 2 or 3, B >= 0");
    if (n < 8) return fail(h, TVF_ERR_TOO_FEW_POINTS, TVF_LINEARF_ERRMSG);
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    Up u(h);
    const size_t np = (size_t)rows * n * B;
    CoreInput in{};
    in.p1 = u.in(p1, np); in.p2 = u.in(p2, np); in.p3 = nullptr;
    in.packed = 0; in.rows = rows; in.n = n; in.B = B; in.normalize = 0;
    double* dF = u.out<double>(9 * (size_t)B);
    int* dst = u.out<int>((size_t)B);
    double* dws = u.out<double>((size_t)CORE_WS_F * B);
    if (u.rc) return u.rc;
    launch_f_stage1(in, dws, dst, h->sm_count, u.st);
    launch_f_finish(dws, 0, B, dF, u.st);
    h->launches += 2;
    std::vector<int32_t> tmp; int32_t* sth = status;
    if (!sth) { tmp.resize((size_t)B); sth = tmp.data(); }
    u.back(F, dF, 9 * (size_t)B);
    u.back(sth, (const int32_t*)dst, (size_t)B);
    int rc = u.finish();
    return rc ? rc : count_flagged(sth, B);
}

int tvf_optim_f(tvf_handle_t h, const double* p1, const double* p2, int rows, int n, int64_t B, double* F, int32_t* iter,
                int32_t* status) {
    if (!h) return TVF_ERR_ARG;
    if (!p1 || !p2 || !F || (rows != 2 && rows != 3) || B < 0) return fail(h, TVF_ERR_ARG, "optimF: bad argument");
    if (n < 8) return fail(h, TVF_ERR_TOO_FEW_POINTS, TVF_LINEARF_ERRMSG);                 // optimF.m:36-38
    if (n > optimf_max_n()) return fail(h, TVF_ERR_ARG, "optimF: too many correspondences for the Gauss-Helmert kernel (see tvf_optim_f_max_n)");
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    // the kernels work on packed 6 x n records; the pair (p1, p2) is stored as views 1 and 2 (and again as view 3)
    std::vector<double> packed((size_t)6 * n * B);
    for (size_t i = 0; i < (size_t)n * B; ++i) {
        double a0 = p1[i * rows], a1 = p1[i * rows + 1], b0 = p2[i * rows], b1 = p2[i * rows + 1];
        if (rows == 3) { a0 /= p1[i * 3 + 2]; a1 /= p1[i * 3 + 2]; b0 /= p2[i * 3 + 2]; b1 /= p2[i * 3 + 2]; }   // optimF.m:40-43
        double* q = &packed[6 * i];
        q[0] = a0; q[1] = a1; q[2] = b0; q[3] = b1; q[4] = b0; q[5] = b1;
    }
    Up u(h);
    CoreInput in{};
    in.p1 = u.in(packed.data(), packed.size()); in.packed = 1; in.rows = 2; in.n = n; in.B = B; in.normalize = 1;
    double* dF = u.out<double>(18 * (size_t)B);
    int* dst = u.out<int>((size_t)B);
    int* dit = u.out<int>(2 * (size_t)B);
    double* dws = u.out<double>((size_t)CORE_WS_F * B);
    if (u.rc) return u.rc;
    launch_f_stage1(in, dws, dst, h->sm_count, u.st);
    if (!launch_optimf_gh(in.p1, n, B, dws, dF, dit, dst, h->sm_count, u.st)) return fail(h, TVF_ERR_ARG, "optimF: n too large");
    h->launches += 3;
    std::vector<double> Fh(18 * (size_t)B);
    std::vector<int32_t> ith(2 * (size_t)B), tmp;
    int32_t* sth = status;
    if (!sth) { tmp.resize((size_t)B); sth = tmp.data(); }
    u.back(Fh.data(), dF, 18 * (size_t)B);
    u.back(ith.data(), (const int32_t*)dit, 2 * (size_t)B);
    u.back(sth, (const int32_t*)dst, (size_t)B);
    int rc = u.finish();
    if (rc) return rc;
    for (int64_t b = 0; b < B; ++b) {
        for (int q = 0; q < 9; ++q) F[9 * b + q] = Fh[18 * b + q];
        if (iter) iter[b] = ith[2 * b];
    }
    return count_flagged(sth, B);
}

int tvf_normalize2d(tvf_handle_t h, const double* points, int n, int64_t B, double* new_points, double* N_matrix) {
    if (!h) return TVF_ERR_ARG;
    if (!points || n < 1 || B < 0) return fail(h, TVF_ERR_ARG, "points must not be NULL, n >= 1");
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    Up u(h);
    const double* d = u.in(points, (size_t)2 * n * B);
    double* o = u.out<double>((size_t)2 * n * B);
    double* N = u.out<double>(9 * (size_t)B);
    if (u.rc) return u.rc;
    launch_normalize2d(d, n, B, o, N, u.st); h->launches += 1;
    u.back(new_points, o, (size_t)2 * n * B); u.back(N_matrix, N, 9 * (size_t)B);
    return u.finish();
}

int tvf_transform_tft(tvf_handle_t h, const double* T_old, const double* M1, const double* M2, const double* M3,
                      int mats_batched, int inverse, int64_t B, double* T_new) {
    if (!h) return TVF_ERR_ARG;
    if (!T_old || !M1 || !M2 || !M3 || !T_new || B < 0) return fail(h, TVF_ERR_ARG, "NULL argument");
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    Up u(h);
    const size_t nm = mats_batched ? 9 * (size_t)B : 9;
    const double* t = u.in(T_old, 27 * (size_t)B);
    const double* m1 = u.in(M1, nm); const double* m2 = u.in(M2, nm); const double* m3 = u.in(M3, nm);
    double* o = u.out<double>(27 * (size_t)B);
    if (u.rc) return u.rc;
    launch_transform_tft(t, m1, m2, m3, mats_batched, inverse, B, o, u.st); h->launches += 1;
    u.back(T_new, o, 27 * (size_t)B);
    return u.finish();
}

int tvf_rt_from_tft(tvf_handle_t h, const double* T, const double* calm, int calm_batched, const double* corresp, int n,
                    int64_t B, double* Rt2, double* Rt3, int32_t* votes, int32_t* status) {
    if (!h) return TVF_ERR_ARG;
    if (!T || !calm || !corresp || n < 1 || B < 0) return fail(h, TVF_ERR_ARG, "NULL argument or bad size");
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    Up u(h);
    PoseTailArgs a{};
    const double* dT = u.in(T, 27 * (size_t)B);
    a.corresp = u.in(corresp, (size_t)6 * n * B);
    a.calm = u.in(calm, calm_batched ? 27 * (size_t)B : 27);
    a.calm_batched = calm_batched; a.n = n; a.B = B;
    a.cand = u.out<double>((size_t)CAND_SIZE * B);
    a.votes = u.out<int>(10 * (size_t)B);
    a.scale = u.out<double>(2 * (size_t)B);
    a.Rt2 = u.out<double>(12 * (size_t)B); a.Rt3 = u.out<double>(12 * (size_t)B);
    a.status = u.out<int>((size_t)B);
    if (u.rc) return u.rc;
    TVF_CK(cudaMemsetAsync(a.status, 0, (size_t)B * sizeof(int), u.st));
    launch_candidates(0, dT, a, u.st);
    if (n >= TAIL_FUSED_MIN_N && n <= TAIL_FUSED_MAX_N) {
        launch_pose_tail_fused(a, h->sm_count, u.st);
        h->launches += 2;
    } else {
        launch_votes(a, h->sm_count, u.st);
        launch_scale(a, h->sm_count, u.st);
        launch_final(a, h->sm_count, u.st);
        h->launches += 4;
    }
    std::vector<int32_t> tmp; int32_t* sth = status;
    if (!sth) { tmp.resize((size_t)B); sth = tmp.data(); }
    u.back(Rt2, a.Rt2, 12 * (size_t)B); u.back(Rt3, a.Rt3, 12 * (size_t)B);
    u.back(votes, (const int32_t*)a.votes, 10 * (size_t)B);
    u.back(sth, (const int32_t*)a.status, (size_t)B);
    int rc = u.finish();
    return rc ? rc : count_flagged(sth, B);
}

int tvf_tft_from_p(tvf_handle_t h, const double* P1, const double* P2, const double* P3, int64_t B, double* T) {
    if (!h) return TVF_ERR_ARG;
    if (!P1 || !P2 || !P3 || !T || B < 0) return fail(h, TVF_ERR_ARG, "NULL argument");
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    Up u(h);
    const double* a = u.in(P1, 12 * (size_t)B); const double* b = u.in(P2, 12 * (size_t)B); const double* c = u.in(P3, 12 * (size_t)B);
    double* o = u.out<double>(27 * (size_t)B);
    if (u.rc) return u.rc;
    launch_tft_from_p(a, b, c, B, o, u.st); h->launches += 1;
    u.back(T, o, 27 * (size_t)B);
    return u.finish();
}

int tvf_triangulate(tvf_handle_t h, const double* P, int M, int cams_batched, const double* image_points, int rows, int n,
                    int64_t B, double* X) {
    if (!h) return TVF_ERR_ARG;
    if (!P || !image_points || !X || n < 1 || B < 0) return fail(h, TVF_ERR_ARG, "NULL argument or bad size");
    if (M != 2 && M != 3) return fail(h, TVF_ERR_ARG, "triangulation3D: only M = 2 or 3 views are supported");
    if (rows != 2 && rows != 3) return fail(h, TVF_ERR_ARG, "rows must be 2 or 3");   // triangulation3D.m:46-47
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    Up u(h);
    const double* dP = u.in(P, (size_t)12 * M * (cams_batched ? B : 1));
    const double* dp = u.in(image_points, (size_t)rows * M * n * B);
    double* o = u.out<double>((size_t)4 * n * B);
    if (u.rc) return u.rc;
    launch_triangulate(dP, M, cams_batched, dp, rows, n, B, o, u.st); h->launches += 1;
    u.back(X, o, (size_t)4 * n * B);
    return u.finish();
}

int tvf_repr_error(tvf_handle_t h, const double* P, int M, int cams_batched, const double* corresp, int rows, int n,
                   int64_t B, const double* points3d, int pts_rows, double* err) {
    if (!h) return TVF_ERR_ARG;
    if (!P || !corresp || !err || n < 1 || B < 0) return fail(h, TVF_ERR_ARG, "NULL argument or bad size");
    if (M != 2 && M != 3) return fail(h, TVF_ERR_ARG, "ReprError: only M = 2 or 3 views are supported");
    if (rows != 2 && rows != 3) return fail(h, TVF_ERR_ARG, "rows must be 2 or 3");
    if (points3d && pts_rows != 3 && pts_rows != 4) return fail(h, TVF_ERR_ARG, "pts_rows must be 3 or 4");
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    Up u(h);
    const double* dP = u.in(P, (size_t)12 * M * (cams_batched ? B : 1));
    const double* dc = u.in(corresp, (size_t)rows * M * n * B);
    const double* dx = points3d ? u.in(points3d, (size_t)pts_rows * n * B) : nullptr;
    double* o = u.out<double>((size_t)B);
    if (u.rc) return u.rc;
    launch_repr_error(dP, M, cams_batched, dc, rows, n, B, dx, pts_rows, o, u.st); h->launches += 1;
    u.back(err, o, (size_t)B);
    return u.finish();
}

int tvf_project3d(tvf_handle_t h, const double* points3d, const double* P, int M, int cams_batched, int n, int64_t B,
                  double* corresp) {
    if (!h) return TVF_ERR_ARG;
    if (!points3d || !P || !corresp || n < 1 || B < 0 || M < 1) return fail(h, TVF_ERR_ARG, "NULL argument or bad size");
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    Up u(h);
    const double* dx = u.in(points3d, (size_t)3 * n * B);
    const double* dP = u.in(P, (size_t)12 * M * (cams_batched ? B : 1));
    double* o = u.out<double>((size_t)2 * M * n * B);
    if (u.rc) return u.rc;
    launch_project3d(dx, dP, M, cams_batched, n, B, o, u.st); h->launches += 1;
    u.back(corresp, o, (size_t)2 * M * n * B);
    return u.finish();
}

static int sweep_common(tvf_handle_t h, int64_t first_trial, int64_t B, int n, const double* noise_levels, int L,
                        const double* P, double hi_x, double hi_y, double* d_out, cudaStream_t st) {
    void* p0; void* p1;
    int rc = ensure_scratch(h, NSCRATCH - 2, (size_t)L * sizeof(double), &p0); if (rc) return rc;
    rc = ensure_scratch(h, NSCRATCH - 3, 36 * sizeof(double), &p1); if (rc) return rc;
    TVF_CK(cudaMemcpyAsync(p0, noise_levels, (size_t)L * sizeof(double), cudaMemcpyHostToDevice, st));
    TVF_CK(cudaMemcpyAsync(p1, P, 36 * sizeof(double), cudaMemcpyHostToDevice, st));
    launch_sweep_trials(first_trial, B, n, (const double*)p0, L, (const double*)p1, hi_x, hi_y, d_out, st);
    h->launches += 1;
    TVF_CK(cudaGetLastError());
    return TVF_OK;
}

static int sweep_check(tvf_handle_t h, int64_t first_trial, int64_t B, int n, const double* noise_levels, int L,
                       const double* P, const double* out) {
    if (!h) return TVF_ERR_ARG;
    if (!noise_levels || !P || !out || L < 1 || B < 0 || first_trial < 0) return fail(h, TVF_ERR_ARG, "NULL argument or bad size");
    if (n < 1 || n > SWEEP_MAX_N) return fail(h, TVF_ERR_ARG, "device scene generator supports 1 <= n <= 60");
    if ((first_trial + B) / L + 1 > 0xffffffffLL) return fail(h, TVF_ERR_ARG, "seed exceeds 32 bits");
    return TVF_OK;
}

int tvf_generate_sweep_dev(tvf_handle_t h, int64_t first_trial, int64_t B, int n, const double* noise_levels, int L,
                           const double* P, double hi_x, double hi_y, double* d_corresp) {
    int rc = sweep_check(h, first_trial, B, n, noise_levels, L, P, d_corresp); if (rc) return rc;
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    cudaStream_t st = h->use_user_stream ? h->user_stream : h->slot[0].stream;
    // the two small host arrays are consumed by an async copy: make that copy complete before returning
    rc = sweep_common(h, first_trial, B, n, noise_levels, L, P, hi_x, hi_y, d_corresp, st); if (rc) return rc;
    TVF_CK(cudaStreamSynchronize(st));
    return TVF_OK;
}

int tvf_generate_sweep(tvf_handle_t h, int64_t first_trial, int64_t B, int n, const double* noise_levels, int L,
                       const double* P, double hi_x, double hi_y, double* corresp) {
    int rc = sweep_check(h, first_trial, B, n, noise_levels, L, P, corresp); if (rc) return rc;
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    Up u(h);
    double* o = u.out<double>((size_t)6 * n * B);
    if (u.rc) return u.rc;
    rc = sweep_common(h, first_trial, B, n, noise_levels, L, P, hi_x, hi_y, o, u.st); if (rc) return rc;
    u.back(corresp, o, (size_t)6 * n * B);
    return u.finish();
}

// experiments.m:74-124 for one method, device-resident: generate the trials of the sweep, solve them, and
// reduce ReprError / AngError per noise level.  Only the L x 5 table crosses the bus.
int tvf_sweep_run(tvf_handle_t h, int method, int64_t first_trial, int64_t B, int n, const double* noise_levels, int L,
                  const double* P, double hi_x, double hi_y, const double* calm, const double* Rt0_2, const double* Rt0_3,
                  double* table) {
    int rc = sweep_check(h, first_trial, B, n, noise_levels, L, P, table); if (rc) return rc;
    if (!calm || !Rt0_2 || !Rt0_3 || (method != 1 && method != 7 && method != 8))
        return fail(h, TVF_ERR_ARG, "method must be 1 (linear TFT), 7 (linear F) or 8 (optimal F); calm/Rt0 required");
    if (method != 1 && n < 8) return fail(h, TVF_ERR_TOO_FEW_POINTS, TVF_LINEARF_ERRMSG);
    TVF_CK(cudaSetDevice(h->device));
    Slot& s = h->slot[0];
    cudaStream_t st = s.stream;
    const int Q = 512;
    // nothing crosses the bus here, so the solver runs its large device-path launches (the per-problem output buffers of
    // the host-path layout are still needed: the evaluation kernels read them)
    const int64_t C = pick_chunk(h, n, B > 0 ? B : 1, false, false);
    const size_t need = carve(nullptr, n, C, true, false, false, nullptr);
    rc = ensure_arena(h, s, need); if (rc) return rc;
    ChunkBufs b; carve(s.arena, n, C, true, false, false, &b);
    void *pc, *pr, *pp, *pt;
    rc = ensure_scratch(h, 0, 27 * sizeof(double), &pc); if (rc) return rc;
    rc = ensure_scratch(h, NSCRATCH - 4, 24 * sizeof(double), &pr); if (rc) return rc;
    rc = ensure_scratch(h, NSCRATCH - 5, (size_t)L * Q * 5 * sizeof(double), &pp); if (rc) return rc;
    rc = ensure_scratch(h, NSCRATCH - 6, (size_t)L * 5 * sizeof(double), &pt); if (rc) return rc;
    TVF_CK(cudaMemcpyAsync(pc, calm, 27 * sizeof(double), cudaMemcpyHostToDevice, st));
    TVF_CK(cudaMemcpyAsync(pr, Rt0_2, 12 * sizeof(double), cudaMemcpyHostToDevice, st));
    TVF_CK(cudaMemcpyAsync((double*)pr + 12, Rt0_3, 12 * sizeof(double), cudaMemcpyHostToDevice, st));
    TVF_CK(cudaMemsetAsync(pp, 0, (size_t)L * Q * 5 * sizeof(double), st));
    // The generator shares one pass per seed among its L noise levels (one warp per seed), so it wants many seeds
    // per launch: trials are generated in super-chunks of up to 4 solver chunks into a staging buffer.
    const int64_t G = (B < 4 * C) ? B : 4 * C;
    void* pg;
    rc = ensure_scratch(h, NSCRATCH - 7, (size_t)G * 6 * n * sizeof(double), &pg); if (rc) return rc;
    for (int64_t gdone = 0; gdone < B; gdone += G) {
        const int64_t Gc = (B - gdone < G) ? (B - gdone) : G;
        rc = sweep_common(h, first_trial + gdone, Gc, n, noise_levels, L, P, hi_x, hi_y, (double*)pg, st); if (rc) return rc;
        for (int64_t off = 0; off < Gc; off += C) {
            const int64_t Bc = (Gc - off < C) ? (Gc - off) : C;
            const double* d_in = (const double*)pg + off * 6 * n;
            rc = run_pose_chunk(h, st, method == 1 ? METHOD_TFT : (method == 7 ? METHOD_F : METHOD_OPTF), d_in, (const double*)pc, 0, n,
                                Bc, b.T, b.F, b.core, b.cand, b.votes, b.scale, b.Rt2, b.Rt3, b.reconst, b.repr, b.status, b.iters, nullptr);
            if (rc) return rc;
            launch_sweep_eval_accumulate(b.Rt2, b.Rt3, b.repr, b.status, first_trial + gdone + off, Bc, L, Q, (const double*)pr, (double*)pp, st);
            h->launches += 1;
        }
    }
    launch_sweep_eval_finish((const double*)pp, L, Q, (double*)pt, st);
    h->launches += 1;
    TVF_CK(cudaGetLastError());
    TVF_CK(cudaMemcpyAsync(table, pt, (size_t)L * 5 * sizeof(double), cudaMemcpyDeviceToHost, st));
    TVF_CK(cudaStreamSynchronize(st));
    return TVF_OK;
}

// experiments.m:74-124 for any of its four options ('noise', 'focal', 'points', 'angle', :38-47): every level carries its
// own noise, point count, cameras, calibration and ground truth.  Level by level: the level's trials (one per seed) are
// generated with its cameras, solved with its n and CalM, and reduced into its row of the table -- all on the device.
// ba: each chunk's poses are then bundle-adjusted (experiments.m:127-141 with the library's adjustment) and reduced into
// columns 5-10 of an L x 11 table; without it the table is L x 5 and the chunk size, and so every sum, is unchanged.
static int sweep_levels(tvf_handle_t h, int method, int64_t first_trial, int64_t B, const tvf_sweep_level* levels, int L,
                        double hi_x, double hi_y, double* table, bool ba) {
    if (!h) return TVF_ERR_ARG;
    if (!levels || !table || L < 1 || B < 0 || first_trial < 0) return fail(h, TVF_ERR_ARG, "NULL argument or bad size");
    if (method != 1 && method != 7 && method != 8) return fail(h, TVF_ERR_ARG, "method must be 1 (linear TFT), 7 (linear F) or 8 (optimal F)");
    if ((first_trial + B) / L + 1 > 0xffffffffLL) return fail(h, TVF_ERR_ARG, "seed exceeds 32 bits");
    int n_max = 1;
    for (int l = 0; l < L; ++l) {
        if (levels[l].n < 1 || levels[l].n > SWEEP_MAX_N) return fail(h, TVF_ERR_ARG, "device scene generator supports 1 <= n <= 60");
        if (levels[l].n > n_max) n_max = levels[l].n;
    }
    TVF_CK(cudaSetDevice(h->device));
    Slot& s = h->slot[0];
    cudaStream_t st = s.stream;
    const int Q = 512;
    const int W = ba ? 11 : 5;                 // table columns
    const Method m = method == 1 ? METHOD_TFT : (method == 7 ? METHOD_F : METHOD_OPTF);
    const int64_t per_level = B / L + 1;
    const int64_t C = pick_chunk(h, n_max, per_level, false, ba);
    const size_t need = carve(nullptr, n_max, C, true, false, ba, nullptr);
    int rc = ensure_arena(h, s, need); if (rc) return rc;
    ChunkBufs b; carve(s.arena, n_max, C, true, false, ba, &b);
    void *pc, *pr, *pp, *pt, *pg, *pb = nullptr;
    rc = ensure_scratch(h, NSCRATCH - 8, (size_t)L * 27 * sizeof(double), &pc); if (rc) return rc;
    rc = ensure_scratch(h, NSCRATCH - 9, (size_t)L * 24 * sizeof(double), &pr); if (rc) return rc;
    rc = ensure_scratch(h, NSCRATCH - 5, (size_t)L * Q * 5 * sizeof(double), &pp); if (rc) return rc;
    rc = ensure_scratch(h, NSCRATCH - 6, (size_t)L * W * sizeof(double), &pt); if (rc) return rc;
    if (ba) { rc = ensure_scratch(h, NSCRATCH - 10, (size_t)L * Q * 6 * sizeof(double), &pb); if (rc) return rc; }
    const int64_t G = (per_level < 4 * C) ? per_level : 4 * C;
    rc = ensure_scratch(h, NSCRATCH - 7, (size_t)G * 6 * n_max * sizeof(double), &pg); if (rc) return rc;
    std::vector<double> hc((size_t)L * 27), hr((size_t)L * 24);
    for (int l = 0; l < L; ++l) {
        memcpy(&hc[(size_t)l * 27], levels[l].calm, 27 * sizeof(double));
        memcpy(&hr[(size_t)l * 24], levels[l].Rt0_2, 12 * sizeof(double));
        memcpy(&hr[(size_t)l * 24 + 12], levels[l].Rt0_3, 12 * sizeof(double));
    }
    TVF_CK(cudaMemcpyAsync(pc, hc.data(), hc.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    TVF_CK(cudaMemcpyAsync(pr, hr.data(), hr.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    TVF_CK(cudaMemsetAsync(pp, 0, (size_t)L * Q * 5 * sizeof(double), st));
    TVF_CK(cudaMemsetAsync(pt, 0, (size_t)L * W * sizeof(double), st));
    if (ba) TVF_CK(cudaMemsetAsync(pb, 0, (size_t)L * Q * 6 * sizeof(double), st));
    std::vector<char> skipped((size_t)L, 0);
    for (int l = 0; l < L; ++l) {
        // trials j = l + L*q of [first_trial, first_trial + B): 0-based seed index q in [q_lo, q_hi), seed = q + 1
        const int64_t q_lo = (first_trial > l) ? (first_trial - l + L - 1) / L : 0;
        const int64_t q_hi = (first_trial + B > l) ? (first_trial + B - l + L - 1) / L : 0;
        const int64_t Bl = q_hi - q_lo;
        const int n = levels[l].n;
        if ((method != 1 && n < 8) || n < 7) { skipped[(size_t)l] = 1; continue; }          // experiments.m:99-104: "not enough matches"
        if (Bl <= 0) continue;
        const double* calm_l = (const double*)pc + (size_t)l * 27;
        const double* gt_l = (const double*)pr + (size_t)l * 24;
        for (int64_t gdone = 0; gdone < Bl; gdone += G) {
            const int64_t Gc = (Bl - gdone < G) ? (Bl - gdone) : G;
            rc = sweep_common(h, q_lo + gdone, Gc, n, &levels[l].noise, 1, levels[l].P, hi_x, hi_y, (double*)pg, st); if (rc) return rc;
            for (int64_t off = 0; off < Gc; off += C) {
                const int64_t Bc = (Gc - off < C) ? (Gc - off) : C;
                const double* d_in = (const double*)pg + off * 6 * n;
                rc = run_pose_chunk(h, st, m, d_in, calm_l, 0, n, Bc, b.T, b.F, b.core,
                                    b.cand, b.votes, b.scale, b.Rt2, b.Rt3, b.reconst, b.repr, b.status, b.iters, nullptr);
                if (rc) return rc;
                launch_sweep_eval_accumulate(b.Rt2, b.Rt3, b.repr, b.status, q_lo + gdone + off, Bc, 1, Q, gt_l,
                                             (double*)pp + (size_t)l * Q * 5, st);
                h->launches += 1;
                if (!ba) continue;
                // a trial without a pose starts from NaN: the kernel copies it through with TVF_ST_NONFINITE and iter = 0
                rc = ba_launch(h, st, BaIo{d_in, calm_l, 0, n, b.Rt2, b.Rt3, b.reconst, b.ba_Rt2, b.ba_Rt3, b.ba_X, b.ba_repr,
                                           b.ba_iter, b.ba_status}, Bc, b.ba_Xc);
                if (rc) return rc;
                launch_sweep_eval_accumulate(b.ba_Rt2, b.ba_Rt3, b.ba_repr, b.status, q_lo + gdone + off, Bc, 1, Q, gt_l,
                                             (double*)pb + (size_t)l * Q * 6, st, b.ba_status, b.ba_iter);
                h->launches += 1;
            }
        }
        launch_sweep_eval_finish((const double*)pp + (size_t)l * Q * 5, 1, Q, (double*)pt + (size_t)l * W, st);
        h->launches += 1;
        if (ba) {
            launch_sweep_eval_finish((const double*)pb + (size_t)l * Q * 6, 1, Q, (double*)pt + (size_t)l * W + 5, st, 6);
            h->launches += 1;
        }
    }
    TVF_CK(cudaGetLastError());
    TVF_CK(cudaMemcpyAsync(table, pt, (size_t)L * W * sizeof(double), cudaMemcpyDeviceToHost, st));
    TVF_CK(cudaStreamSynchronize(st));
    const double inf = __builtin_huge_val();
    for (int l = 0; l < L; ++l) {
        if (!skipped[(size_t)l]) continue;
        double* row = table + (size_t)W * l;
        for (int c = 0; c < W; ++c) row[c] = 0.0;
        row[0] = row[1] = row[2] = inf;
        if (ba) row[5] = row[6] = row[7] = inf;
    }
    return TVF_OK;
}

int tvf_sweep_run_levels(tvf_handle_t h, int method, int64_t first_trial, int64_t B, const tvf_sweep_level* levels, int L,
                         double hi_x, double hi_y, double* table) {
    return sweep_levels(h, method, first_trial, B, levels, L, hi_x, hi_y, table, false);
}

int tvf_sweep_run_levels_ba(tvf_handle_t h, int method, int64_t first_trial, int64_t B, const tvf_sweep_level* levels, int L,
                            double hi_x, double hi_y, double* table) {
    return sweep_levels(h, method, first_trial, B, levels, L, hi_x, hi_y, table, true);
}

int tvf_bundle_adjust(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                      const double* Rt2_0, const double* Rt3_0, const double* reconst0, double* Rt2, double* Rt3,
                      double* reconst, double* repr_err, int32_t* iter, int32_t* status) {
    return ba_host(h, BaIo{corresp, calm, calm_batched, n, Rt2_0, Rt3_0, reconst0, Rt2, Rt3, reconst, repr_err, iter, status}, B);
}

int tvf_bundle_adjust_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                          const double* Rt2_0, const double* Rt3_0, const double* reconst0, double* Rt2, double* Rt3,
                          double* reconst, double* repr_err, int32_t* iter, int32_t* status) {
    return ba_dev(h, BaIo{corresp, calm, calm_batched, n, Rt2_0, Rt3_0, reconst0, Rt2, Rt3, reconst, repr_err, iter, status}, B);
}

int tvf_ba_covariance(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                      const double* Rt2, const double* Rt3, const double* reconst, double* cov_cam, double* cov_pts,
                      double* sigma2, int32_t* status) {
    return ba_host(h, BaIo{corresp, calm, calm_batched, n, Rt2, Rt3, reconst, nullptr, nullptr, nullptr, nullptr, nullptr,
                           status, true, cov_cam, cov_pts, sigma2}, B);
}

int tvf_ba_covariance_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                          const double* Rt2, const double* Rt3, const double* reconst, double* cov_cam, double* cov_pts,
                          double* sigma2, int32_t* status) {
    return ba_dev(h, BaIo{corresp, calm, calm_batched, n, Rt2, Rt3, reconst, nullptr, nullptr, nullptr, nullptr, nullptr,
                          status, true, cov_cam, cov_pts, sigma2}, B);
}

int tvf_ang_error(tvf_handle_t h, const double* Rt_true, int true_batched, const double* Rt_est, int64_t B,
                  double* rot_err, double* t_err) {
    if (!h) return TVF_ERR_ARG;
    if (!Rt_true || !Rt_est || !rot_err || !t_err || B < 0) return fail(h, TVF_ERR_ARG, "NULL argument");
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    Up u(h);
    const double* a = u.in(Rt_true, (size_t)12 * (true_batched ? B : 1));
    const double* e = u.in(Rt_est, 12 * (size_t)B);
    double* r = u.out<double>((size_t)B); double* t = u.out<double>((size_t)B);
    if (u.rc) return u.rc;
    launch_ang_error(a, true_batched, e, B, r, t, u.st); h->launches += 1;
    u.back(rot_err, r, (size_t)B); u.back(t_err, t, (size_t)B);
    return u.finish();
}

}  // extern "C"
