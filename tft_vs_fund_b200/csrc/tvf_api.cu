// tvf_api.cu -- the C ABI of include/tvf.h: handle, work-space arenas, chunked
// host-pointer entry points (H2D / kernels / D2H pipelined over three streams)
// and asynchronous device-pointer entry points.  No CPU fallback lives here:
// every entry point either runs the CUDA kernels or returns an error.
#include "../../include/tvf.h"

#include <cuda_runtime.h>
#include <sched.h>

#include <algorithm>
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
constexpr int NSLOT = TVF_NSLOT;
// per-handle device scratch buffers (ensure_scratch): Up's count up from SCR_UP, the named ones lie above them
constexpr int UP_SLOTS = 12;                    // Up: one buffer per array of a stand-alone call (tvf_rt_from_tft has 9)
enum Scratch {
    SCR_UP = 0,
    SCR_FP64_PEAK = SCR_UP + UP_SLOTS,          // tvf_fp64_peak_tflops' output
    SCR_SWEEP_NOISE, SCR_SWEEP_CAMS,            // the scene generator's noise levels and cameras
    SCR_SWEEP_CALM, SCR_SWEEP_GT,               // a sweep's calibrations and ground-truth poses
    SCR_SWEEP_PARTIAL, SCR_SWEEP_BA_PARTIAL,    // its per-level partial sums, of the poses and of their adjustment
    SCR_SWEEP_TABLE, SCR_SWEEP_TRIALS,          // its table and one generator call's trials
    NSCRATCH
};
static_assert(SCR_UP + UP_SLOTS <= SCR_FP64_PEAK && SCR_FP64_PEAK < NSCRATCH, "Up's scratch range meets the named ones");
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
    // tvf_create_multi: further devices of a group handle (this context is member 0); the host-pointer batched calls
    // (host_call) shard B over the members, one host thread per device (experiments.m:91-143 is the loop that fans out)
    std::vector<tvf_context*> peers;
    // tvf_set_host_register: pin caller buffers that are pageable for the duration of a host-pointer batched call
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

// the buffers of one pose chunk (run_pose_chunk; in and calm are the chunk's inputs)
struct ChunkBufs {
    const double* in; const double* calm; double* T; double* F; double* core; double* cand; int* votes; double* scale;
    double* Rt2; double* Rt3; double* reconst; double* repr; int* status; int* iters; int* iter_sum;
    // ba: the bundle adjustment of the chunk's poses (tvf_sweep_run_levels_ba)
    double* ba_Rt2; double* ba_Rt3; double* ba_X; double* ba_Xc; double* ba_repr; int* ba_iter; int* ba_status;
};

size_t carve_pose(char* base, int n, int64_t C, bool host_io, bool calm_batched, bool ba, ChunkBufs* out) {
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

// per-problem bytes of carve_pose's buffers, for the automatic chunk size (a batched calm counted either way)
size_t pose_budget(int n, bool host_io, bool ba) {
    size_t payload = (27 + 18 + CORE_WS_TFT + CAND_SIZE + 2) * 8 + 14 * 4;
    if (host_io) payload += (size_t)(6 * n + 27 + 24 + 3 * n + 1) * 8;
    if (ba) payload += (size_t)(24 + 6 * n + 3) * sizeof(double);   // Rt2, Rt3, X, Xc, repr (+ iter, status in the last double)
    return payload;
}

// problems per chunk: tvf_set_chunk's, else the default cut so that `per` bytes per problem stay within one slot's
// arena budget (eight budgets on the device-pointer path); per = 0: no cut
int64_t pick_chunk(tvf_handle_t h, int64_t B, bool host_io, size_t per) {
    int64_t c = h->chunk_user > 0 ? h->chunk_user : (host_io ? DEFAULT_CHUNK : DEFAULT_CHUNK_DEV);
    if (h->chunk_user <= 0 && per > 0) {
        const int64_t fit = (int64_t)((host_io ? ARENA_BUDGET : 8 * ARENA_BUDGET) / per);
        if (c > fit) c = fit;
    }
    if (c < 1) c = 1;
    if (c > B) c = B;
    return c;
}

enum Method { METHOD_TFT = 0, METHOD_F = 1, METHOD_OPTF = 2, METHOD_FIVEPT = 3 };   // FIVEPT: RANSAC hypotheses only

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

// kernels of one chunk of Bc problems; all pointers are device pointers.  b.T null: T is not wanted (the F methods
// then skip TFT_from_P); b.reconst, b.repr and b.iter_sum may be null.
int run_pose_chunk(tvf_handle_t h, cudaStream_t st, Method method, int calm_batched, int n, int64_t Bc, const ChunkBufs& b) {
    CoreInput in{};
    in.p1 = b.in; in.p2 = nullptr; in.p3 = nullptr; in.packed = 1; in.rows = 2; in.n = n; in.B = Bc; in.normalize = 1;
    PoseTailArgs a{};
    a.corresp = b.in; a.calm = b.calm; a.calm_batched = calm_batched; a.n = n; a.B = Bc;
    a.cand = b.cand; a.votes = b.votes; a.scale = b.scale;
    a.Rt2 = b.Rt2; a.Rt3 = b.Rt3; a.reconst = b.reconst; a.repr_err = b.repr; a.status = b.status;
    const int sm = h->sm_count;
    if (method == METHOD_TFT) {
        bool large_done = false;
        if (n >= LARGE_N_MIN) {
            timed_launch(h, TVF_K_TFT_MOMENTS_LARGE, st, [&] {
                large_done = launch_tft_moments_large(b.in, n, Bc, 1, b.core, sm, st) != 0;
            });
            if (large_done)
                timed_launch(h, TVF_K_TFT_STAGE1_SOLVE, st, [&] { launch_tft_stage1_solve(Bc, b.core, b.status, sm, st); });
        }
        if (!large_done) {
            int need_solve = 0;
            timed_launch(h, TVF_K_TFT_STAGE1, st, [&] { need_solve = launch_tft_stage1(in, b.core, b.status, sm, st); });
            if (need_solve)
                timed_launch(h, TVF_K_TFT_STAGE1_SOLVE, st, [&] { launch_tft_stage1_solve(Bc, b.core, b.status, sm, st); });
        }
        timed_launch(h, TVF_K_TFT_EPIPOLES, st, [&] { launch_tft_epipoles(b.core, Bc, st); });
        timed_launch(h, TVF_K_TFT_STAGE2, st, [&] { launch_tft_stage2(in, b.core, b.T, nullptr, nullptr, b.status, sm, st); });
        timed_launch(h, TVF_K_CANDIDATES, st, [&] { launch_candidates(0, b.T, a, st); });
    } else if (method == METHOD_F) {
        timed_launch(h, TVF_K_F_STAGE1, st, [&] { launch_f_stage1(in, b.core, b.status, sm, st); });
        timed_launch(h, TVF_K_F_FINISH, st, [&] { launch_f_finish(b.core, 1, Bc, b.F, st); });
        timed_launch(h, TVF_K_CANDIDATES, st, [&] { launch_candidates(1, b.F, a, st); });
    } else {    // OptimFPoseEstimation.m:47-53: linearF start, Gauss-Helmert refinement, then the F pose tail
        timed_launch(h, TVF_K_F_STAGE1, st, [&] { launch_f_stage1(in, b.core, b.status, sm, st); });
        int ok = 1;
        timed_launch(h, TVF_K_OPTIMF_GH, st, [&] { ok = launch_optimf_gh(b.in, n, Bc, b.core, b.F, b.iters, b.status, sm, st); });
        if (!ok) return fail(h, TVF_ERR_ARG, "optimF: too many correspondences for the Gauss-Helmert kernel (see tvf_optim_f_max_n)");
        if (b.iter_sum) launch_sum_pairs(b.iters, Bc, b.iter_sum, st);
        timed_launch(h, TVF_K_CANDIDATES, st, [&] { launch_candidates(1, b.F, a, st); });
    }
    if (n >= TAIL_FUSED_MIN_N && n <= TAIL_FUSED_MAX_N) {
        timed_launch(h, TVF_K_TAIL_FUSED, st, [&] { launch_pose_tail_fused(a, sm, st); });
    } else {
        timed_launch(h, TVF_K_VOTES, st, [&] { launch_votes(a, sm, st); });
        timed_launch(h, TVF_K_SCALE, st, [&] { launch_scale(a, sm, st); });
        timed_launch(h, TVF_K_FINAL, st, [&] { launch_final(a, sm, st); });
    }
    if (method != METHOD_TFT && b.T != nullptr)
        timed_launch(h, TVF_K_TFT_FROM_POSE, st, [&] { launch_tft_from_pose(b.calm, calm_batched, b.Rt2, b.Rt3, Bc, b.T, st); });
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

// caller buffers that are pageable get pinned for the duration of a call (tvf_set_host_register); RAII
struct HostPins {
    std::vector<void*> pinned;
    void add(const void* p, size_t bytes) {
        if (bytes < (1u << 20) || !is_pageable(p)) return;
        if (cudaHostRegister(const_cast<void*>(p), bytes, cudaHostRegisterPortable) == cudaSuccess) pinned.push_back(const_cast<void*>(p));
        else cudaGetLastError();
    }
    ~HostPins() { for (void* p : pinned) cudaHostUnregister(p); }
};

inline size_t align256(size_t bytes) { return (bytes + 255) & ~size_t(255); }

// ---- host-pointer calls -------------------------------------------------------------------------------------------
// A host-pointer entry point is a Call: its caller arrays, the device buffers of the chunk in flight (`d`), and
//   size_t budget(bool host_io)          per-problem bytes of a chunk, for pick_chunk
//   size_t budget_match(bool host_io)    per-match bytes of a chunk of a ragged call, for its match budget
//   size_t carve(char* base, int64_t C, int64_t M)   lays `d` out in a slot arena for C problems and, ragged, M matches
//                                        (base = nullptr: size only)
//   void arrays(F f)                     f(caller pointer, Arr) for every caller array: the one place their layout is written
//   int launch(h, stream, Bc)            the kernels of one chunk on `d`
//   int check(h, B), int32_t*& status()  argument checks; the per-problem status array
//   Ragged rg                            the offsets of a ragged call (uniform: none)

// A ragged call (include/tvf.h: problem b owns matches offs[b] .. offs[b+1]-1): its offsets in host memory from the
// call's first problem on, the chunk's offsets rebased to 0 on the device (carved with the chunk's buffers) and the
// chunk's match count
struct Ragged {
    const int64_t* offs = nullptr;     // null: a uniform call
    long long* d_offs = nullptr;
    int64_t m = 0;
};

int check_offsets(tvf_handle_t h, const char* what, const int64_t* offs, int64_t B) {
    if (B < 0) return fail(h, TVF_ERR_ARG, std::string(what) + ": B >= 0");
    if (!offs) return fail(h, TVF_ERR_ARG, std::string(what) + ": offsets must not be NULL");
    if (offs[0] != 0) return fail(h, TVF_ERR_ARG, std::string(what) + ": offsets[0] must be 0");
    for (int64_t b = 0; b < B; ++b) {
        const int64_t nb = offs[b + 1] - offs[b];
        if (nb < 0) return fail(h, TVF_ERR_ARG, std::string(what) + ": offsets must not decrease");
        if (nb > 0x7fffffffLL) return fail(h, TVF_ERR_ARG, std::string(what) + ": a problem has more than 2^31 - 1 matches");
    }
    return TVF_OK;
}

// One caller array beside its device buffer in the chunk's arena
struct Arr {
    bool out;         // false: host -> device before the chunk's kernels; true: device -> host after them
    size_t per;       // bytes per problem (per match when `match`); 0: one copy of `pitch` bytes that every problem
                      // shares (a 9 x 3 calm)
    const void* dev;  // the chunk's device buffer
    size_t pitch;     // bytes per problem in `dev` (F21 / F31: 72 bytes out of each 144-byte F record)
    bool match = false;   // a per-match array of a ragged call (corresp, reconst, inliers, ...)
    static Arr input(size_t per, const void* dev, bool shared = false) { return Arr{false, shared ? 0 : per, dev, per}; }
    static Arr output(size_t per, const void* dev, size_t pitch = 0) { return Arr{true, per, dev, pitch ? pitch : per}; }
    // `bytes` per match: per problem n x bytes (uniform), or per match (ragged)
    static Arr points(const Ragged& rg, int n, size_t bytes, const void* dev, bool out) {
        Arr a = out ? output(rg.offs ? bytes : n * bytes, dev) : input(rg.offs ? bytes : n * bytes, dev);
        a.match = rg.offs != nullptr;
        return a;
    }
    // byte offset of problem b in the caller's array (offs: the call's offsets, for a per-match array)
    size_t at(const int64_t* offs, int64_t b) const { return (size_t)(match ? offs[b] - offs[0] : b) * per; }
    // bytes of problems [lo, hi)
    size_t bytes(const int64_t* offs, int64_t lo, int64_t hi) const { return per ? at(offs, hi) - at(offs, lo) : pitch; }
};

// the caller arrays of `c` from problem `lo` on
template <class Call> void shift(Call& c, int64_t lo) {
    c.arrays([&](auto& p, const Arr& a) { if (p) p += (int64_t)(a.at(c.rg.offs, lo) / sizeof(*p)); });
    if (c.rg.offs) c.rg.offs += lo;
}

// The chunks of a call over B problems, as their ends.  Uniform: every C problems, C = pick_chunk.  Ragged: contiguous
// ranges cut greedily at C problems or at the match budget M (per-match bytes against the arena budget, the same budget
// pick_chunk uses), whichever comes first; a problem larger than M gets a chunk of its own.  *C, *M: the most problems
// and matches of one chunk, the shape its buffers are carved for.
template <class Call> std::vector<int64_t> plan_chunks(tvf_handle_t h, const Call& c, int64_t B, bool host_io, int64_t* C,
                                                       int64_t* M) {
    *C = pick_chunk(h, B, host_io, c.budget(host_io));
    *M = 0;
    std::vector<int64_t> ends;
    const int64_t* o = c.rg.offs;
    if (!o) {
        for (int64_t e = *C; e < B + *C; e += *C) ends.push_back(e < B ? e : B);
        return ends;
    }
    const size_t pm = c.budget_match(host_io);
    const int64_t cap = pm ? (int64_t)((host_io ? ARENA_BUDGET : 8 * ARENA_BUDGET) / pm) : INT64_MAX;
    int64_t most = 0;
    for (int64_t lo = 0; lo < B;) {
        int64_t hi = lo + 1;
        while (hi < B && hi - lo < *C && o[hi + 1] - o[lo] <= cap) ++hi;
        ends.push_back(hi);
        *M = std::max(*M, o[hi] - o[lo]);
        most = std::max(most, hi - lo);
        lo = hi;
    }
    *C = most;
    return ends;
}

// A ragged call's chunk [lo, hi): its offsets rebased to 0 to the chunk's device copy (ordered on `st` before the
// chunk's kernels; pageable, so the runtime stages them before it returns) and rg.m.  Uniform: nothing.
template <class Call> int put_offsets(tvf_handle_t h, Call& c, int64_t lo, int64_t hi, cudaStream_t st) {
    if (!c.rg.offs) return TVF_OK;
    std::vector<long long> v((size_t)(hi - lo + 1));
    for (int64_t b = lo; b <= hi; ++b) v[(size_t)(b - lo)] = c.rg.offs[b] - c.rg.offs[lo];
    c.rg.m = v.back();
    TVF_CK(cudaMemcpyAsync(c.rg.d_offs, v.data(), v.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
    return TVF_OK;
}

// One host-pointer call on one device.  Chunk i runs on slot i mod NSLOT (stream + arena), so its H2D, kernels and D2H
// overlap those of its neighbours.
template <class Call> int host_pipeline(tvf_handle_t h, Call c, int64_t B) {
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    int64_t C, M;
    const std::vector<int64_t> ends = plan_chunks(h, c, B, true, &C, &M);
    const size_t need = c.carve(nullptr, C, M);
    const int64_t* offs = c.rg.offs;
    // the staging buffer of one chunk holds C problems and M matches of each array
    auto cap = [&](const Arr& a) { return a.per ? (size_t)(a.match ? M : C) * a.per : a.pitch; };
    // Pageable caller memory (what a MEX gateway receives): cudaMemcpyAsync would fall back to synchronous copies through
    // the runtime's own bounce buffer and serialise the pipeline (measured 6.6e6 solves/s against 4.5e7 with pinned
    // buffers).  Instead every chunk goes through a pinned per-slot staging buffer that a few host threads fill and drain.
    // A shared array is one small copy and stays where it is.
    size_t moved = 0;
    bool pageable = false;
    c.arrays([&](const void* p, const Arr& a) {
        if (p && a.per) { moved += a.bytes(offs, 0, B); pageable = pageable || is_pageable(p); }
    });
    const bool staged = pageable && !h->host_register && moved >= (size_t(4) << 20);
    std::vector<int32_t> st_tmp;
    if (!c.status()) { st_tmp.resize((size_t)B); c.status() = st_tmp.data(); }
    size_t stage_bytes = 0;
    c.arrays([&](const void* p, const Arr& a) { if (p && a.per) stage_bytes += align256(cap(a)); });
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
    // earlier asynchronous *_dev / sweep work of this handle may still be using slot 0's arena
    TVF_CK(cudaStreamSynchronize(h->slot[0].stream));
    if (h->use_user_stream) TVF_CK(cudaStreamSynchronize(h->user_stream));

    // Chunk schedule: uniform chunks.  The call is bound by the host link (H2D of chunk i+1, kernels of chunk i and D2H of
    // chunk i-1 overlap).  Quarter- and half-size chunks at both ends, meant to shorten the pipeline's fill and drain, were
    // measured SLOWER (4.31e7 vs 4.56e7 solves/s end to end at 1 M problems, profiles/r01_variants.md).
    int64_t done = 0; int ci = 0;
    int rc = TVF_OK;
    for (const int64_t end : ends) {
        const int64_t Bc = end - done;
        const int si = ci % NSLOT;
        Slot& s = h->slot[si];
        TVF_CK(cudaStreamSynchronize(s.stream));        // slot reuse: its previous chunk (incl. D2H) is finished
        rc = ensure_arena(h, s, need); if (rc) return rc;
        c.carve(s.arena, C, M);
        rc = put_offsets(h, c, done, end, s.stream); if (rc) return rc;
        char* stage = nullptr;
        if (staged) {
            drain(si);                                   // the slot's previous outputs leave the staging buffer first
            rc = ensure_stage(h, si, stage_bytes); if (rc) return rc;
            stage = (char*)h->stage[si];
        }
        // straight from / into the caller's array, or through the slot's staging buffer (outputs with a drain entry)
        cudaError_t e = cudaSuccess;
        c.arrays([&](const void* p, const Arr& a) {
            if (!p || a.out || e != cudaSuccess) return;
            const char* src = (const char*)p + a.at(offs, done);
            if (staged && a.per) {
                par_memcpy(stage, src, a.bytes(offs, done, end), nthreads);
                src = stage;
                stage += align256(cap(a));
            }
            e = cudaMemcpyAsync(const_cast<void*>(a.dev), src, a.bytes(offs, done, end), cudaMemcpyHostToDevice, s.stream);
        });
        if (e != cudaSuccess) return fail(h, TVF_ERR_CUDA, std::string("cudaMemcpyAsync(host to device): ") + cudaGetErrorString(e));
        rc = c.launch(h, s.stream, Bc); if (rc) return rc;
        c.arrays([&](const void* p, const Arr& a) {
            if (!p || !a.out || e != cudaSuccess) return;
            char* dst = (char*)const_cast<void*>(p) + a.at(offs, done);
            if (staged) {
                pending[si].push_back(Drain{dst, stage, a.bytes(offs, done, end)});
                dst = stage;
                stage += align256(cap(a));
            }
            e = (a.pitch == a.per) ? cudaMemcpyAsync(dst, a.dev, a.bytes(offs, done, end), cudaMemcpyDeviceToHost, s.stream)
                                   : cudaMemcpy2DAsync(dst, a.per, a.dev, a.pitch, a.per, (size_t)Bc, cudaMemcpyDeviceToHost, s.stream);
        });
        if (e != cudaSuccess) return fail(h, TVF_ERR_CUDA, std::string("cudaMemcpyAsync(device to host): ") + cudaGetErrorString(e));
        done += Bc; ++ci;
    }
    for (int i = 0; i < NSLOT; ++i) {
        const int si = (ci + i) % NSLOT;                 // oldest chunk first
        TVF_CK(cudaStreamSynchronize(h->slot[si].stream));
        if (staged) drain(si);
    }
    return count_flagged(c.status(), B);
}

// contiguous [lo, hi) of B problems for member g of G (remainder to the first members; same rule as sharding.shard_range)
inline void shard_of(int64_t B, int g, int G, int64_t* lo, int64_t* hi) {
    const int64_t base = B / G, rem = B % G;
    *lo = g * base + (g < rem ? g : rem);
    *hi = *lo + base + (g < rem ? 1 : 0);
}

// the same for a ragged call (offs: B + 1 offsets from 0): member g starts at the first problem whose matches start at or
// after g / G of all matches, so the ranges hold about equal match counts
inline void shard_of_matches(const int64_t* offs, int64_t B, int g, int G, int64_t* lo, int64_t* hi) {
    auto start = [&](int k) -> int64_t {
        if (k == G) return B;
        const int64_t t = (int64_t)((__int128)offs[B] * k / G);
        return std::lower_bound(offs, offs + B, t) - offs;
    };
    *lo = start(g);
    *hi = start(g + 1);
}

// A host-pointer call: checks, page-locking (tvf_set_host_register), then the pipeline, on one device or sharded over the
// members of a group handle.  Member g solves the contiguous range shard_of(B, g, G) on its own device from its own host
// thread; problems are independent and a problem's result does not depend on its batch, so the outputs are
// bit-identical to a single-device call.
template <class Call> int host_call(tvf_handle_t h, Call c, int64_t B) {
    int rc = c.check(h, B);
    if (rc != TVF_OK) return rc;
    if (B == 0) return TVF_OK;
    HostPins pins;
    if (h->host_register) {
        TVF_CK(cudaSetDevice(h->device));
        c.arrays([&](const void* p, const Arr& a) { if (a.per) pins.add(p, a.bytes(c.rg.offs, 0, B)); });
    }
    const int G = 1 + (int)h->peers.size();
    if (G == 1 || B < G) return host_pipeline(h, c, B);
    std::vector<int> rcs((size_t)G, TVF_OK);
    auto run = [&](int g) {
        tvf_handle_t m = (g == 0) ? h : h->peers[(size_t)g - 1];
        int64_t lo, hi;
        if (c.rg.offs) shard_of_matches(c.rg.offs, B, g, G, &lo, &hi); else shard_of(B, g, G, &lo, &hi);
        Call s = c;
        shift(s, lo);
        m->chunk_user = h->chunk_user; m->host_threads = h->host_threads;
        rcs[(size_t)g] = host_pipeline(m, s, hi - lo);
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

// outputs of a pose call (any may be null); `votes` = 10 int32 per problem: the 4 + 4 cheirality votes of
// R_t_from_TFT.m:91-104 in the reference's candidate order for the pairs (1,2) and (1,3), then the two NaN masks
struct PoseOut {
    double* Rt2; double* Rt3; double* reconst; double* T; double* repr_err; double* F21; double* F31;
    int32_t* iter; int32_t* votes; int32_t* status;
};

// tvf_pose and the per-method pose calls
struct PoseCall {
    Method method; const double* corresp; const double* calm; int calm_batched; int n; PoseOut o;
    ChunkBufs d{};
    Ragged rg{};                          // always uniform
    int check(tvf_handle_t h, int64_t B) const { return check_pose_args(h, corresp, calm, n, B, method); }
    int32_t*& status() { return o.status; }
    size_t budget(bool host_io) const { return pose_budget(n, host_io, false); }
    size_t budget_match(bool) const { return 0; }
    size_t carve(char* base, int64_t C, int64_t) { return carve_pose(base, n, C, true, calm_batched != 0, false, &d); }
    template <class F> void arrays(F&& f) {
        f(corresp, Arr::input(8 * 6 * n, d.in));
        f(calm, Arr::input(8 * 27, d.calm, !calm_batched));
        f(o.Rt2, Arr::output(8 * 12, d.Rt2));
        f(o.Rt3, Arr::output(8 * 12, d.Rt3));
        f(o.reconst, Arr::output(8 * 3 * n, d.reconst));
        f(o.T, Arr::output(8 * 27, d.T));
        f(o.repr_err, Arr::output(8, d.repr));
        f(o.votes, Arr::output(4 * 10, d.votes));
        if (method != METHOD_TFT) {
            f(o.F21, Arr::output(8 * 9, d.F, 8 * 18));
            f(o.F31, Arr::output(8 * 9, d.F + 9, 8 * 18));
        }
        if (method == METHOD_OPTF) f(o.iter, Arr::output(4, d.iter_sum));
        f(o.status, Arr::output(4, d.status));
    }
    int launch(tvf_handle_t h, cudaStream_t st, int64_t Bc) {
        ChunkBufs k = d;
        if (method != METHOD_TFT && !o.T) k.T = nullptr;
        return run_pose_chunk(h, st, method, calm_batched, n, Bc, k);
    }
};

int pose_dev(tvf_handle_t h, const PoseCall& c, int64_t B) {
    int rc = c.check(h, B);
    if (rc != TVF_OK) return rc;
    // the kernels read the correspondences with 128-bit loads and bulk asynchronous copies: 16-byte alignment (every
    // cudaMalloc'ed buffer and every problem boundary inside one satisfies it: a problem is 48 n bytes)
    if ((reinterpret_cast<uintptr_t>(c.corresp) & 15u) != 0) return fail(h, TVF_ERR_ARG, "device pointer `corresp` must be 16-byte aligned");
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    Slot& s = h->slot[0];
    cudaStream_t st = h->use_user_stream ? h->user_stream : s.stream;
    const int n = c.n;
    const int64_t C = pick_chunk(h, B, false, c.budget(false));
    // internal buffers only; Rt2/Rt3 are needed internally by the F method's TFT_from_P, so stage them if absent
    const size_t need = carve_pose(nullptr, n, C, false, false, false, nullptr) + (size_t)(24 * C) * sizeof(double) + 512;
    rc = ensure_arena(h, s, need); if (rc) return rc;
    ChunkBufs b; const size_t used = carve_pose(s.arena, n, C, false, false, false, &b);
    double* tmpRt2 = reinterpret_cast<double*>(s.arena + used);
    double* tmpRt3 = tmpRt2 + 12 * C;
    for (int64_t done = 0; done < B; done += C) {
        const int64_t Bc = (B - done < C) ? (B - done) : C;
        PoseCall k = c;
        shift(k, done);
        const PoseOut& o = k.o;
        ChunkBufs d = b;                        // the caller's arrays; the work space for those it does not give
        d.in = k.corresp; d.calm = k.calm; d.reconst = o.reconst; d.repr = o.repr_err; d.iter_sum = o.iter;
        d.T = o.T ? o.T : (c.method == METHOD_TFT ? b.T : nullptr);
        d.Rt2 = o.Rt2 ? o.Rt2 : tmpRt2; d.Rt3 = o.Rt3 ? o.Rt3 : tmpRt3;
        d.votes = o.votes ? o.votes : b.votes; d.status = o.status ? o.status : b.status;
        rc = run_pose_chunk(h, st, c.method, c.calm_batched, n, Bc, d); if (rc) return rc;
        if (c.method != METHOD_TFT && o.F21)
            TVF_CK(cudaMemcpy2DAsync(o.F21, 72, b.F, 144, 72, (size_t)Bc, cudaMemcpyDeviceToDevice, st));
        if (c.method != METHOD_TFT && o.F31)
            TVF_CK(cudaMemcpy2DAsync(o.F31, 72, b.F + 9, 144, 72, (size_t)Bc, cudaMemcpyDeviceToDevice, st));
    }
    return TVF_OK;
}

// ---- bundle adjustment (tvf_bundle_adjust[_dev]) and its covariance (tvf_ba_covariance[_dev]) ------------------------
// `io` holds the caller's arrays (host or device pointers), `d` the chunk's kernel arguments: on the host path device
// copies carved from a slot arena, on the device path the caller's arrays themselves plus the work space.

// one kernel launch of the adjustment or the covariance: counted, and its launch error reported under the kernel's name
int ba_launched(tvf_handle_t h, int ok, const char* kernel) {
    h->launches += 1;
    if (ok) return TVF_OK;
    cudaError_t e = cudaGetLastError();
    return fail(h, TVF_ERR_CUDA, std::string(kernel) + ": " + cudaGetErrorString(e));
}

int check_ba_size(tvf_handle_t h, int n, int64_t B) {
    if (B < 0) return fail(h, TVF_ERR_ARG, "bundle_adjust: B >= 0");
    if (n < 4) return fail(h, TVF_ERR_ARG, "bundle_adjust: needs n >= 4 points (11 + 3n unknowns, 6n residuals)");
    return TVF_OK;
}

// outputs may be null except Rt2 / Rt3; X0 null: the kernel triangulates the start points
struct BundleAdjust {
    BaArgs io;
    BaArgs d{};
    Ragged rg{};                          // ragged: io.n = 0, every per-point array per match
    int check(tvf_handle_t h, int64_t B) const {
        if (!h) return TVF_ERR_ARG;
        if (!io.corresp || !io.calm || !io.Rt2_0 || !io.Rt3_0 || !io.Rt2 || !io.Rt3)
            return fail(h, TVF_ERR_ARG, "bundle_adjust: corresp, calm, Rt2_0, Rt3_0, Rt2 and Rt3 must not be NULL");
        return rg.offs ? check_offsets(h, "bundle_adjust", rg.offs, B) : check_ba_size(h, io.n, B);
    }
    int32_t*& status() { return io.status; }
    // the work space Xc (and X on the device path when the caller wants no points); the host path's inputs and outputs,
    // counting a batched calm and X0 whether or not the call has them
    size_t budget(bool host_io) const {
        const int n = io.n;
        size_t b = (size_t)2 * 3 * n * sizeof(double);
        if (host_io) b += (size_t)(6 * n + 27 + 24 + 3 * n + 24 + 1) * sizeof(double) + 2 * sizeof(int32_t);
        return b + (rg.offs ? sizeof(long long) : 0);
    }
    size_t budget_match(bool host_io) const { return (size_t)(2 * 3 + (host_io ? 9 : 0)) * sizeof(double); }
    size_t carve(char* base, int64_t C, int64_t M, bool host_io = true) {
        const int64_t P = rg.offs ? M : (int64_t)io.n * C;      // points of the chunk
        Carver c(base);
        d = io;
        if (host_io) {
            d.corresp = c.take<double>((size_t)6 * P); d.calm = c.take<double>(io.calm_batched ? 27 * C : 27);
            d.Rt2_0 = c.take<double>(12 * C); d.Rt3_0 = c.take<double>(12 * C);
            d.X0 = io.X0 ? c.take<double>((size_t)3 * P) : nullptr;
            d.Rt2 = c.take<double>(12 * C); d.Rt3 = c.take<double>(12 * C); d.X = c.take<double>((size_t)3 * P);
            d.repr_err = c.take<double>(C); d.iter = c.take<int>(C); d.status = c.take<int>(C);
        }
        if (!d.X) d.X = c.take<double>((size_t)3 * P);
        d.Xc = c.take<double>((size_t)3 * P);
        if (rg.offs) d.offs = rg.d_offs = c.take<long long>(C + 1);
        return c.off;
    }
    template <class F> void arrays(F&& f) {
        const int n = io.n;
        f(io.corresp, Arr::points(rg, n, 8 * 6, d.corresp, false));
        f(io.calm, Arr::input(8 * 27, d.calm, !io.calm_batched));
        f(io.Rt2_0, Arr::input(8 * 12, d.Rt2_0));
        f(io.Rt3_0, Arr::input(8 * 12, d.Rt3_0));
        f(io.X0, Arr::points(rg, n, 8 * 3, d.X0, false));
        f(io.Rt2, Arr::output(8 * 12, d.Rt2));
        f(io.Rt3, Arr::output(8 * 12, d.Rt3));
        f(io.X, Arr::points(rg, n, 8 * 3, d.X, true));
        f(io.repr_err, Arr::output(8, d.repr_err));
        f(io.iter, Arr::output(4, d.iter));
        f(io.status, Arr::output(4, d.status));
    }
    int launch(tvf_handle_t h, cudaStream_t st, int64_t Bc) {
        BaArgs a = d; a.B = Bc;
        return ba_launched(h, launch_bundle_adjust(a, st), rg.offs ? "bundle_adjust_ragged_kernel" : "bundle_adjust_kernel");
    }
};

// the robust-loss adjustment: BundleAdjust's arrays, work space and checks, plus the loss and two outputs that may be
// null, cost (per problem) and weights (per match).  BundleAdjust's own chunk budget is left as it is.
struct BundleAdjustRobust : BundleAdjust {
    BaRobustArgs rio;
    BaRobustArgs rd{};
    int check(tvf_handle_t h, int64_t B) const {
        if (!h) return TVF_ERR_ARG;
        if (rio.loss < TVF_LOSS_HUBER || rio.loss > TVF_LOSS_CAUCHY)
            return fail(h, TVF_ERR_ARG, "bundle_adjust_robust: loss must be TVF_LOSS_HUBER, TVF_LOSS_SOFT_L1 or TVF_LOSS_CAUCHY");
        const double c2 = rio.scale * rio.scale;       // the kernel divides by c^2: a normal number, so z = s / c^2 is exact
        if (!(rio.scale > 0.0) || !(c2 >= 2.2250738585072014e-308 && c2 <= 1.79769313486231570e308))
            return fail(h, TVF_ERR_ARG, "bundle_adjust_robust: scale must be finite and > 0 (1e-154 < scale < 1e154)");
        return BundleAdjust::check(h, B);
    }
    size_t budget(bool host_io) const {
        return BundleAdjust::budget(host_io) + (host_io ? (size_t)(1 + io.n) * sizeof(double) : 0);
    }
    size_t budget_match(bool host_io) const { return BundleAdjust::budget_match(host_io) + (host_io ? sizeof(double) : 0); }
    size_t carve(char* base, int64_t C, int64_t M, bool host_io = true) {
        Carver c(base);
        c.off = BundleAdjust::carve(base, C, M, host_io);
        rd = rio;
        if (host_io) {
            rd.cost = c.take<double>(C);
            rd.weights = rio.weights ? c.take<double>((size_t)(rg.offs ? M : (int64_t)io.n * C)) : nullptr;
        }
        return c.off;
    }
    template <class F> void arrays(F&& f) {
        BundleAdjust::arrays(f);
        f(rio.cost, Arr::output(8, rd.cost));
        f(rio.weights, Arr::points(rg, io.n, 8, rd.weights, true));
    }
    int launch(tvf_handle_t h, cudaStream_t st, int64_t Bc) {
        BaArgs a = d; a.B = Bc;
        return ba_launched(h, launch_bundle_adjust_robust(a, rd, st),
                           rg.offs ? "bundle_adjust_robust_ragged_kernel" : "bundle_adjust_robust_kernel");
    }
};

// the state Rt2, Rt3, X is required; every output may be null
struct Covariance {
    BaCovArgs io;
    BaCovArgs d{};
    Ragged rg{};                          // ragged: io.n = 0, every per-point array per match
    int check(tvf_handle_t h, int64_t B) const {
        if (!h) return TVF_ERR_ARG;
        if (!io.corresp || !io.calm || !io.Rt2 || !io.Rt3 || !io.X)
            return fail(h, TVF_ERR_ARG, "ba_covariance: corresp, calm, Rt2, Rt3 and reconst must not be NULL");
        return rg.offs ? check_offsets(h, "ba_covariance", rg.offs, B) : check_ba_size(h, io.n, B);
    }
    int32_t*& status() { return io.status; }
    // the host path's inputs and outputs, counting a batched calm and cov_pts whether or not the call has them; the
    // device path needs no work space
    size_t budget(bool host_io) const {
        const int n = io.n;
        return (host_io ? (size_t)(6 * n + 27 + 24 + 3 * n + 144 + 9 * n + 1 + 1) * sizeof(double) : 0) +
               (rg.offs ? sizeof(long long) : 0);
    }
    size_t budget_match(bool host_io) const { return host_io ? (size_t)(6 + 3 + 9) * sizeof(double) : 0; }
    size_t carve(char* base, int64_t C, int64_t M, bool host_io = true) {
        const int64_t P = rg.offs ? M : (int64_t)io.n * C;      // points of the chunk
        Carver c(base);
        d = io;
        if (host_io) {
            d.corresp = c.take<double>((size_t)6 * P); d.calm = c.take<double>(io.calm_batched ? 27 * C : 27);
            d.Rt2 = c.take<double>(12 * C); d.Rt3 = c.take<double>(12 * C); d.X = c.take<double>((size_t)3 * P);
            d.cov_cam = io.cov_cam ? c.take<double>(144 * C) : nullptr;
            d.cov_pts = io.cov_pts ? c.take<double>((size_t)9 * P) : nullptr;
            d.sigma2 = c.take<double>(C); d.status = c.take<int>(C);
        }
        if (rg.offs) d.offs = rg.d_offs = c.take<long long>(C + 1);
        return c.off;
    }
    template <class F> void arrays(F&& f) {
        const int n = io.n;
        f(io.corresp, Arr::points(rg, n, 8 * 6, d.corresp, false));
        f(io.calm, Arr::input(8 * 27, d.calm, !io.calm_batched));
        f(io.Rt2, Arr::input(8 * 12, d.Rt2));
        f(io.Rt3, Arr::input(8 * 12, d.Rt3));
        f(io.X, Arr::points(rg, n, 8 * 3, d.X, false));
        f(io.cov_cam, Arr::output(8 * 144, d.cov_cam));
        f(io.cov_pts, Arr::points(rg, n, 8 * 9, d.cov_pts, true));
        f(io.sigma2, Arr::output(8, d.sigma2));
        f(io.status, Arr::output(4, d.status));
    }
    int launch(tvf_handle_t h, cudaStream_t st, int64_t Bc) {
        BaCovArgs a = d; a.B = Bc;
        return ba_launched(h, launch_ba_covariance(a, st), rg.offs ? "ba_covariance_ragged_kernel" : "ba_covariance_kernel");
    }
};

// device pointers, asynchronous on the handle's stream
template <class Call> int ba_dev(tvf_handle_t h, const Call& c, int64_t B) {
    int rc = c.check(h, B);
    if (rc != TVF_OK) return rc;
    if ((reinterpret_cast<uintptr_t>(c.io.corresp) & 15u) != 0) return fail(h, TVF_ERR_ARG, "device pointer `corresp` must be 16-byte aligned");
    if (B == 0) return TVF_OK;
    TVF_CK(cudaSetDevice(h->device));
    Slot& s = h->slot[0];
    cudaStream_t st = h->use_user_stream ? h->user_stream : s.stream;
    int64_t C, M;
    const std::vector<int64_t> ends = plan_chunks(h, c, B, false, &C, &M);
    Call k = c;
    rc = ensure_arena(h, s, k.carve(nullptr, C, M, false)); if (rc) return rc;
    int64_t done = 0;
    for (const int64_t end : ends) {
        k = c;
        shift(k, done);
        k.carve(s.arena, C, M, false);
        rc = put_offsets(h, k, 0, end - done, st); if (rc) return rc;
        rc = k.launch(h, st, end - done); if (rc) return rc;
        done = end;
    }
    return TVF_OK;
}

// ---- RANSAC pose (tvf_ransac_pose[_dev]) and consensus (tvf_consensus) ----------------------------------------------

int ransac_launched(tvf_handle_t h) {
    h->launches += 1;
    TVF_CK(cudaGetLastError());
    return TVF_OK;
}

// outputs may be null: on the device path the work space stands in for them
struct Ransac {
    Method method; int s; int H; double th;
    RansacArgs io;
    RansacArgs d{};
    ChunkBufs w{};                       // the pose path's work space, for the B H hypotheses and then the refit
    Ragged rg{};                         // ragged: io.n = 0, corresp and inliers per match
    int check(tvf_handle_t h, int64_t B) const {
        if (!h) return TVF_ERR_ARG;
        if (!io.corresp || !io.calm || !io.seeds) return fail(h, TVF_ERR_ARG, "ransac_pose: corresp, calm and seeds must not be NULL");
        if (B < 0) return fail(h, TVF_ERR_ARG, "ransac_pose: B >= 0");
        if (rg.offs) {                   // a problem of fewer than s matches is flagged, not an error
            const int rc = check_offsets(h, "ransac_pose", rg.offs, B);
            if (rc != TVF_OK) return rc;
        } else if (io.n < s) {
            if (method == METHOD_F) return fail(h, TVF_ERR_TOO_FEW_POINTS, TVF_LINEARF_ERRMSG);
            if (method == METHOD_FIVEPT) return fail(h, TVF_ERR_ARG, "ransac_pose: method 9 needs n >= 5 points");
            return fail(h, TVF_ERR_ARG, "ransac_pose: method 1 needs n >= 7 points");
        }
        if (H < 1 || H > (1 << 24)) return fail(h, TVF_ERR_ARG, "ransac_pose: hypotheses must be in 1 .. 2^24");
        if (!(th > 0.0) || !(th < __builtin_huge_val())) return fail(h, TVF_ERR_ARG, "ransac_pose: threshold must be finite and > 0");
        return TVF_OK;
    }
    int32_t*& status() { return io.status; }
    // H hypotheses (the pose path's work space at n = s, the minimal problem, its calm, pose and count), the refit's
    // compacted problem, the best and the refit pose with their masks and counters, and the host path's inputs and
    // outputs; a batched calm counted either way
    size_t budget(bool host_io) const {
        const int n = io.n;
        size_t b = (size_t)H * (pose_budget(s, false, false) + (size_t)(6 * s + 27 + 24) * 8 + 4);
        b += (size_t)(6 * n + 27 + 48) * 8 + 2 * (size_t)n + 6 * 4;
        if (host_io) b += (size_t)(6 * n + 27 + 1 + 24) * 8 + n + 4 * (size_t)(s + 2);
        return b + (rg.offs ? sizeof(long long) : 0);
    }
    size_t budget_match(bool host_io) const { return (size_t)6 * 8 + 2 + (host_io ? 6 * 8 + 1 : 0); }
    size_t carve(char* base, int64_t C, int64_t M, bool host_io = true) {
        const int64_t P = rg.offs ? M : (int64_t)io.n * C;      // matches of the chunk
        const int64_t Q = C * H;
        Carver c(base);
        d = io;
        if (host_io) {
            d.corresp = c.take<double>((size_t)6 * P); d.calm = c.take<double>(io.calm_batched ? 27 * C : 27);
            d.seeds = c.take<uint64_t>(C);
        }
        if (host_io || !d.Rt2) d.Rt2 = c.take<double>(12 * C);
        if (host_io || !d.Rt3) d.Rt3 = c.take<double>(12 * C);
        if (host_io || !d.inliers) d.inliers = c.take<unsigned char>((size_t)P);
        if (host_io || !d.n_inliers) d.n_inliers = c.take<int>(C);
        if (host_io || !d.sample) d.sample = c.take<int>((size_t)s * C);
        if (host_io || !d.status) d.status = c.take<int>(C);
        c.off += carve_pose(base ? base + c.off : nullptr, s, Q, false, false, false, &w);
        d.gin = c.take<double>((size_t)6 * s * Q); d.gcalm = io.calm_batched ? c.take<double>(27 * Q) : nullptr;
        d.hRt2 = c.take<double>(12 * Q); d.hRt3 = c.take<double>(12 * Q); d.hstatus = w.status; d.hcount = c.take<int>(Q);
        d.best_h = c.take<int>(C); d.cnt_best = c.take<int>(C); d.mask_best = c.take<unsigned char>((size_t)P);
        d.bestRt2 = c.take<double>(12 * C); d.bestRt3 = c.take<double>(12 * C);
        d.refst = c.take<int>(C); d.cnt_refit = c.take<int>(C); d.mask_refit = c.take<unsigned char>((size_t)P);
        d.refRt2 = c.take<double>(12 * C); d.refRt3 = c.take<double>(12 * C);
        d.rin = c.take<double>((size_t)6 * P); d.rcalm = io.calm_batched ? c.take<double>(27 * C) : nullptr;
        d.plist = c.take<int>(C);
        if (rg.offs) rg.d_offs = c.take<long long>(C + 1);
        return c.off;
    }
    template <class F> void arrays(F&& f) {
        const int n = io.n;
        f(io.corresp, Arr::points(rg, n, 8 * 6, d.corresp, false));
        f(io.calm, Arr::input(8 * 27, d.calm, !io.calm_batched));
        f(io.seeds, Arr::input(8, d.seeds));
        f(io.Rt2, Arr::output(8 * 12, d.Rt2));
        f(io.Rt3, Arr::output(8 * 12, d.Rt3));
        f(io.inliers, Arr::points(rg, n, 1, d.inliers, true));
        f(io.n_inliers, Arr::output(4, d.n_inliers));
        f(io.sample, Arr::output(4 * s, d.sample));
        f(io.status, Arr::output(4, d.status));
    }
    // consensus counts of the poses of a.B problems, hyp per problem (into count, zeroed before; mask may be null)
    void consensus(tvf_handle_t h, cudaStream_t st, const RansacArgs& a, int hyp, const double* Rt2, const double* Rt3,
                   const int* hst, int* count, unsigned char* mask) const {
        if (rg.offs)
            launch_ransac_consensus_ragged(a.corresp, a.calm, a.calm_batched, rg.d_offs, a.B, rg.m, hyp, Rt2, Rt3, hst, th,
                                           count, mask, h->sm_count, st);
        else
            launch_ransac_consensus(a.corresp, a.calm, a.calm_batched, a.n, a.B * hyp, hyp, Rt2, Rt3, hst, th, count, mask,
                                    h->sm_count, st);
    }
    // sample and solve the hypotheses, score them, select; refit on the consensus of the best, grouped by its size
    // (the one read-back of the call); rescore; the result rule
    // the Q = Bc H minimal problems (gin, gcalm) and their poses (hRt2, hRt3, hstatus); k: the pose path's buffers
    int hypotheses(tvf_handle_t h, cudaStream_t st, const RansacArgs& a, ChunkBufs& k) const {
        launch_ransac_sample(a, H, s, st, rg.d_offs);
        int rc = ransac_launched(h); if (rc) return rc;
        k = w;
        k.in = a.gin; k.calm = a.calm_batched ? a.gcalm : a.calm; k.Rt2 = a.hRt2; k.Rt3 = a.hRt3;
        if (method == METHOD_FIVEPT) {
            launch_five_point_pose(k.in, k.calm, a.calm_batched, a.B * H, a.hRt2, a.hRt3, nullptr, nullptr, a.hstatus, st);
            return ransac_launched(h);
        }
        if (method != METHOD_TFT) k.T = nullptr;
        return run_pose_chunk(h, st, method, a.calm_batched, s, a.B * H, k);
    }
    // the refit's method and the least consensus it needs: method 9 refits with linear F on >= 8 columns
    Method refit_method() const { return method == METHOD_FIVEPT ? METHOD_F : method; }
    int refit_min() const { return method == METHOD_FIVEPT ? 8 : s; }
    int launch(tvf_handle_t h, cudaStream_t st, int64_t Bc) {
        RansacArgs a = d; a.B = Bc;
        const int64_t Q = Bc * H;
        ChunkBufs k;
        int rc = hypotheses(h, st, a, k); if (rc) return rc;
        TVF_CK(cudaMemsetAsync(a.hcount, 0, (size_t)Q * sizeof(int), st));
        consensus(h, st, a, H, a.hRt2, a.hRt3, a.hstatus, a.hcount, nullptr);
        rc = ransac_launched(h); if (rc) return rc;
        launch_ransac_select(a, H, st);
        rc = ransac_launched(h); if (rc) return rc;
        TVF_CK(cudaMemsetAsync(a.cnt_best, 0, (size_t)Bc * sizeof(int), st));
        consensus(h, st, a, 1, a.bestRt2, a.bestRt3, nullptr, a.cnt_best, a.mask_best);
        rc = ransac_launched(h); if (rc) return rc;
        std::vector<int> cnt((size_t)Bc);
        TVF_CK(cudaMemcpyAsync(cnt.data(), a.cnt_best, (size_t)Bc * sizeof(int), cudaMemcpyDeviceToHost, st));
        TVF_CK(cudaStreamSynchronize(st));
        TVF_CK(cudaMemsetAsync(a.refst, 0xff, (size_t)Bc * sizeof(int), st));      // -1: no refit
        std::vector<int> order;
        for (int64_t b = 0; b < Bc; ++b) if (cnt[(size_t)b] >= refit_min()) order.push_back((int)b);
        std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return cnt[(size_t)x] < cnt[(size_t)y]; });
        if (!order.empty())
            TVF_CK(cudaMemcpyAsync(a.plist, order.data(), order.size() * sizeof(int), cudaMemcpyHostToDevice, st));
        for (size_t g0 = 0; g0 < order.size();) {
            const int size = cnt[(size_t)order[g0]];
            size_t g1 = g0;
            while (g1 < order.size() && cnt[(size_t)order[g1]] == size) ++g1;
            const int m = (int)(g1 - g0);
            launch_ransac_gather(a, a.plist + g0, m, size, st, rg.d_offs);
            rc = ransac_launched(h); if (rc) return rc;
            ChunkBufs r = k;                      // the hypotheses' buffers, free again
            r.in = a.rin; r.calm = a.calm_batched ? a.rcalm : a.calm;
            rc = run_pose_chunk(h, st, refit_method(), a.calm_batched, size, m, r); if (rc) return rc;
            launch_ransac_scatter(a, a.plist + g0, m, r.Rt2, r.Rt3, r.status, st);
            rc = ransac_launched(h); if (rc) return rc;
            g0 = g1;
        }
        TVF_CK(cudaMemsetAsync(a.cnt_refit, 0, (size_t)Bc * sizeof(int), st));
        consensus(h, st, a, 1, a.refRt2, a.refRt3, a.refst, a.cnt_refit, a.mask_refit);
        rc = ransac_launched(h); if (rc) return rc;
        launch_ransac_finish(a, s, st, rg.d_offs);
        return ransac_launched(h);
    }
};

// tvf_ransac_pose_refined: Ransac's layout and hypotheses, each hypothesis adjusted on its own sample (the packed
// adjustment), and LO rounds of the adjustment on the current consensus
struct RansacRefined : Ransac {
    int lo_rounds;
    double *aRt2 = nullptr, *aRt3 = nullptr, *X = nullptr, *Xc = nullptr;
    int* ast = nullptr;
    int check(tvf_handle_t h, int64_t B) const {
        const int rc = Ransac::check(h, B);
        if (rc != TVF_OK) return rc;
        if (lo_rounds < 0 || lo_rounds > 32) return fail(h, TVF_ERR_ARG, "ransac_pose_refined: lo_rounds must be in 0 .. 32");
        return TVF_OK;
    }
    // Ransac's, lo_done, the adjusted hypotheses (pose, status), the adjustment's points and candidates for the larger
    // of the hypotheses (3 x s each) and an LO round (3 x n), and the LO round's start poses
    size_t budget(bool host_io) const {
        const size_t pts = (size_t)3 * (s * (size_t)H > (size_t)io.n ? s * (size_t)H : (size_t)io.n);
        return Ransac::budget(host_io) + 4 + (size_t)H * (24 * 8 + 4) + 2 * pts * 8 + 24 * 8;
    }
    // an LO round's points (3 per match), counted beside the hypotheses' rather than overlapping them
    size_t budget_match(bool host_io) const { return Ransac::budget_match(host_io) + 2 * 3 * 8; }
    size_t carve(char* base, int64_t C, int64_t M, bool host_io = true) {
        Carver c(base);
        c.off = Ransac::carve(base, C, M, host_io);
        const int64_t Q = C * H;
        const int64_t P = rg.offs ? M : (int64_t)io.n * C;      // matches of the chunk
        if (host_io || !d.lo_done) d.lo_done = c.take<int>(C);
        aRt2 = c.take<double>(12 * Q); aRt3 = c.take<double>(12 * Q); ast = c.take<int>(Q);
        const size_t pts = (size_t)3 * (s * Q > P ? s * Q : P);
        X = c.take<double>(pts); Xc = c.take<double>(pts);
        d.gRt2 = c.take<double>(12 * C); d.gRt3 = c.take<double>(12 * C);
        return c.off;
    }
    template <class F> void arrays(F&& f) {
        Ransac::arrays(f);
        f(io.lo_done, Arr::output(4, d.lo_done));
    }
    // Hypotheses; each adjusted from its pose on its sample (X0 null) and scored (flagged: -1); select; then per LO
    // round read the counts back (the call's one read-back per round), adjust every problem whose count grew in the
    // previous round (all in the first) and has >= 4 matches on its consensus, grouped by its size, rescore, accept;
    // the result rule with no refit.  aRt2, aRt3 and ast hold the hypotheses' adjustments, then an LO round's.
    int launch(tvf_handle_t h, cudaStream_t st, int64_t Bc) {
        RansacArgs a = d; a.B = Bc;
        const int64_t Q = Bc * H;
        ChunkBufs k;
        int rc = hypotheses(h, st, a, k); if (rc) return rc;
        const BaArgs hb{a.gin, a.calm_batched ? a.gcalm : a.calm, a.calm_batched, s, Q, a.hRt2, a.hRt3, nullptr, aRt2, aRt3,
                        X, Xc, nullptr, nullptr, ast};
        rc = ba_launched(h, launch_bundle_adjust_small(hb, st), "bundle_adjust_small_kernel"); if (rc) return rc;
        launch_ransac_flag(a.hstatus, ast, Q, st);
        rc = ransac_launched(h); if (rc) return rc;
        TVF_CK(cudaMemsetAsync(a.hcount, 0, (size_t)Q * sizeof(int), st));
        consensus(h, st, a, H, aRt2, aRt3, ast, a.hcount, nullptr);
        rc = ransac_launched(h); if (rc) return rc;
        RansacArgs sel = a; sel.hRt2 = aRt2; sel.hRt3 = aRt3;
        launch_ransac_select(sel, H, st);
        rc = ransac_launched(h); if (rc) return rc;
        TVF_CK(cudaMemsetAsync(a.cnt_best, 0, (size_t)Bc * sizeof(int), st));
        consensus(h, st, a, 1, a.bestRt2, a.bestRt3, nullptr, a.cnt_best, a.mask_best);
        rc = ransac_launched(h); if (rc) return rc;
        TVF_CK(cudaMemsetAsync(a.lo_done, 0, (size_t)Bc * sizeof(int), st));
        std::vector<int> cnt((size_t)Bc), prev;
        for (int r = 1; r <= lo_rounds; ++r) {
            TVF_CK(cudaMemcpyAsync(cnt.data(), a.cnt_best, (size_t)Bc * sizeof(int), cudaMemcpyDeviceToHost, st));
            TVF_CK(cudaStreamSynchronize(st));
            std::vector<int> order;
            for (int64_t b = 0; b < Bc; ++b)
                if (cnt[(size_t)b] >= 4 && (r == 1 || cnt[(size_t)b] > prev[(size_t)b])) order.push_back((int)b);
            if (order.empty()) break;
            std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return cnt[(size_t)x] < cnt[(size_t)y]; });
            TVF_CK(cudaMemcpyAsync(a.plist, order.data(), order.size() * sizeof(int), cudaMemcpyHostToDevice, st));
            TVF_CK(cudaMemsetAsync(a.refst, 0xff, (size_t)Bc * sizeof(int), st));      // -1: not adjusted this round
            for (size_t g0 = 0; g0 < order.size();) {
                const int size = cnt[(size_t)order[g0]];
                size_t g1 = g0;
                while (g1 < order.size() && cnt[(size_t)order[g1]] == size) ++g1;
                const int m = (int)(g1 - g0);
                launch_ransac_gather(a, a.plist + g0, m, size, st, rg.d_offs);
                rc = ransac_launched(h); if (rc) return rc;
                const BaArgs lb{a.rin, a.calm_batched ? a.rcalm : a.calm, a.calm_batched, size, m, a.gRt2, a.gRt3, nullptr,
                                aRt2, aRt3, X, Xc, nullptr, nullptr, ast};
                rc = ba_launched(h, launch_bundle_adjust(lb, st), "bundle_adjust_kernel"); if (rc) return rc;
                launch_ransac_scatter(a, a.plist + g0, m, aRt2, aRt3, ast, st);
                rc = ransac_launched(h); if (rc) return rc;
                g0 = g1;
            }
            launch_ransac_flag(nullptr, a.refst, Bc, st);                           // -1 and TVF_ST_NONFINITE: count -1
            rc = ransac_launched(h); if (rc) return rc;
            TVF_CK(cudaMemsetAsync(a.cnt_refit, 0, (size_t)Bc * sizeof(int), st));
            consensus(h, st, a, 1, a.refRt2, a.refRt3, a.refst, a.cnt_refit, a.mask_refit);
            rc = ransac_launched(h); if (rc) return rc;
            launch_ransac_lo_accept(a, st, rg.d_offs);
            rc = ransac_launched(h); if (rc) return rc;
            prev.swap(cnt);
            cnt.resize((size_t)Bc);
        }
        TVF_CK(cudaMemsetAsync(a.refst, 0xff, (size_t)Bc * sizeof(int), st));          // the result rule without a refit
        launch_ransac_finish(a, s, st, rg.d_offs);
        return ransac_launched(h);
    }
};

// tvf_five_point_pose: the minimal pose of each problem, the kernel RANSAC method 9 runs on its hypotheses
struct FivePoint {
    struct Io {
        const double* corresp; const double* calm; int calm_batched;
        double* Rt2; double* Rt3; double* E; int32_t* n_E; int32_t* status;
    } io;
    Io d{};
    Ragged rg{};                          // always uniform
    int check(tvf_handle_t h, int64_t B) const {
        if (!h) return TVF_ERR_ARG;
        if (!io.corresp || !io.calm) return fail(h, TVF_ERR_ARG, "five_point_pose: corresp and calm must not be NULL");
        if (B < 0) return fail(h, TVF_ERR_ARG, "five_point_pose: B >= 0");
        return TVF_OK;
    }
    int32_t*& status() { return io.status; }
    size_t budget(bool host_io) const { return host_io ? (size_t)(30 + 27 + 24 + 9 * 10) * 8 + 2 * 4 : 0; }
    size_t budget_match(bool) const { return 0; }
    size_t carve(char* base, int64_t C, int64_t, bool host_io = true) {
        Carver c(base);
        d = io;
        if (host_io) {
            d.corresp = c.take<double>(30 * C); d.calm = c.take<double>(io.calm_batched ? 27 * C : 27);
            d.Rt2 = io.Rt2 ? c.take<double>(12 * C) : nullptr; d.Rt3 = io.Rt3 ? c.take<double>(12 * C) : nullptr;
            d.E = io.E ? c.take<double>(90 * C) : nullptr; d.n_E = io.n_E ? c.take<int32_t>(C) : nullptr;
            d.status = c.take<int32_t>(C);
        }
        return c.off;
    }
    template <class F> void arrays(F&& f) {
        f(io.corresp, Arr::input(8 * 30, d.corresp));
        f(io.calm, Arr::input(8 * 27, d.calm, !io.calm_batched));
        f(io.Rt2, Arr::output(8 * 12, d.Rt2));
        f(io.Rt3, Arr::output(8 * 12, d.Rt3));
        f(io.E, Arr::output(8 * 90, d.E));
        f(io.n_E, Arr::output(4, d.n_E));
        f(io.status, Arr::output(4, d.status));
    }
    int launch(tvf_handle_t h, cudaStream_t st, int64_t Bc) {
        launch_five_point_pose(d.corresp, d.calm, d.calm_batched, Bc, d.Rt2, d.Rt3, d.E, d.n_E, d.status, st);
        return ransac_launched(h);
    }
};

// tvf_consensus: no status word, so host_pipeline's temporary one stays zero
struct Consensus {
    const double* corresp; const double* calm; int calm_batched; int n; const double* Rt2; const double* Rt3; double th;
    uint8_t* inliers; int32_t* n_inliers;
    int32_t* no_status = nullptr;
    const double *d_corresp = nullptr, *d_calm = nullptr, *d_Rt2 = nullptr, *d_Rt3 = nullptr;
    uint8_t* d_inliers = nullptr; int32_t* d_count = nullptr;
    Ragged rg{};                          // ragged: n = 0, corresp and inliers per match
    int check(tvf_handle_t h, int64_t B) const {
        if (!h) return TVF_ERR_ARG;
        if (!corresp || !calm || !Rt2 || !Rt3) return fail(h, TVF_ERR_ARG, "consensus: corresp, calm, Rt2 and Rt3 must not be NULL");
        if (rg.offs) {
            const int rc = check_offsets(h, "consensus", rg.offs, B);
            if (rc != TVF_OK) return rc;
        } else if (B < 0 || n < 1) return fail(h, TVF_ERR_ARG, "consensus: need n >= 1 and B >= 0");
        if (!(th > 0.0) || !(th < __builtin_huge_val())) return fail(h, TVF_ERR_ARG, "consensus: threshold must be finite and > 0");
        return TVF_OK;
    }
    int32_t*& status() { return no_status; }
    size_t budget(bool) const { return (size_t)(6 * n + 27 + 24) * 8 + n + 4 + (rg.offs ? 8 : 0); }
    size_t budget_match(bool) const { return (size_t)6 * 8 + 1; }
    size_t carve(char* base, int64_t C, int64_t M) {
        const int64_t P = rg.offs ? M : (int64_t)n * C;      // matches of the chunk
        Carver c(base);
        d_corresp = c.take<double>((size_t)6 * P); d_calm = c.take<double>(calm_batched ? 27 * C : 27);
        d_Rt2 = c.take<double>(12 * C); d_Rt3 = c.take<double>(12 * C);
        d_inliers = c.take<uint8_t>((size_t)P); d_count = c.take<int32_t>(C);
        if (rg.offs) rg.d_offs = c.take<long long>(C + 1);
        return c.off;
    }
    template <class F> void arrays(F&& f) {
        f(corresp, Arr::points(rg, n, 8 * 6, d_corresp, false));
        f(calm, Arr::input(8 * 27, d_calm, !calm_batched));
        f(Rt2, Arr::input(8 * 12, d_Rt2));
        f(Rt3, Arr::input(8 * 12, d_Rt3));
        f(inliers, Arr::points(rg, n, 1, d_inliers, true));
        f(n_inliers, Arr::output(4, d_count));
    }
    int launch(tvf_handle_t h, cudaStream_t st, int64_t Bc) {
        TVF_CK(cudaMemsetAsync(d_count, 0, (size_t)Bc * sizeof(int32_t), st));
        if (rg.offs)
            launch_ransac_consensus_ragged(d_corresp, d_calm, calm_batched, rg.d_offs, Bc, rg.m, 1, d_Rt2, d_Rt3, nullptr, th,
                                           d_count, d_inliers, h->sm_count, st);
        else
            launch_ransac_consensus(d_corresp, d_calm, calm_batched, n, Bc, 1, d_Rt2, d_Rt3, nullptr, th, d_count, d_inliers,
                                    h->sm_count, st);
        return ransac_launched(h);
    }
};

// small helper for the stand-alone functions: upload, run, download on slot 0
struct Up {
    tvf_handle_t h; cudaStream_t st; int rc = TVF_OK; int next = SCR_UP;
    explicit Up(tvf_handle_t hh) : h(hh), st(hh->slot[0].stream) {}
    template <typename T> T* in(const T* host, size_t count) {
        if (rc) return nullptr;
        if (next == SCR_UP + UP_SLOTS) { rc = fail(h, TVF_ERR_ARG, "internal: more arrays than UP_SLOTS"); return nullptr; }
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
    if (ensure_scratch(h, SCR_FP64_PEAK, 64, &p) != TVF_OK) return -1.0;
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
    return host_call(h, PoseCall{m, corresp, calm, calm_batched, n, pose_out_of(out)}, B);
}

int tvf_pose_dev(tvf_handle_t h, int method, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                 const tvf_pose_out* out) {
    Method m;
    if (!h) return TVF_ERR_ARG;
    if (!method_of(method, &m)) return fail(h, TVF_ERR_ARG, "method must be 1 (linear TFT), 7 (linear F) or 8 (optimal F)");
    return pose_dev(h, PoseCall{m, corresp, calm, calm_batched, n, pose_out_of(out)}, B);
}

int tvf_linear_tft_pose(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                        double* Rt2, double* Rt3, double* reconst, double* T, double* repr_err, int32_t* status) {
    return host_call(h, PoseCall{METHOD_TFT, corresp, calm, calm_batched, n, PoseOut{Rt2, Rt3, reconst, T, repr_err, nullptr, nullptr, nullptr, nullptr, status}}, B);
}

int tvf_linear_f_pose(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                      double* Rt2, double* Rt3, double* reconst, double* T, double* repr_err, double* F21, double* F31,
                      int32_t* status) {
    return host_call(h, PoseCall{METHOD_F, corresp, calm, calm_batched, n, PoseOut{Rt2, Rt3, reconst, T, repr_err, F21, F31, nullptr, nullptr, status}}, B);
}

int tvf_optim_f_pose(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                     double* Rt2, double* Rt3, double* reconst, double* T, double* repr_err, double* F21, double* F31,
                     int32_t* iter, int32_t* status) {
    return host_call(h, PoseCall{METHOD_OPTF, corresp, calm, calm_batched, n, PoseOut{Rt2, Rt3, reconst, T, repr_err, F21, F31, iter, nullptr, status}}, B);
}

int tvf_optim_f_pose_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                         double* Rt2, double* Rt3, double* reconst, double* T, double* repr_err, double* F21, double* F31,
                         int32_t* iter, int32_t* status) {
    return pose_dev(h, PoseCall{METHOD_OPTF, corresp, calm, calm_batched, n, PoseOut{Rt2, Rt3, reconst, T, repr_err, F21, F31, iter, nullptr, status}}, B);
}

int tvf_optim_f_max_n(void) { return optimf_max_n(); }

int tvf_linear_tft_pose_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                            double* Rt2, double* Rt3, double* reconst, double* T, double* repr_err, int32_t* status) {
    return pose_dev(h, PoseCall{METHOD_TFT, corresp, calm, calm_batched, n, PoseOut{Rt2, Rt3, reconst, T, repr_err, nullptr, nullptr, nullptr, nullptr, status}}, B);
}

int tvf_linear_f_pose_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                          double* Rt2, double* Rt3, double* reconst, double* T, double* repr_err, double* F21, double* F31,
                          int32_t* status) {
    return pose_dev(h, PoseCall{METHOD_F, corresp, calm, calm_batched, n, PoseOut{Rt2, Rt3, reconst, T, repr_err, F21, F31, nullptr, nullptr, status}}, B);
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
    int rc = ensure_scratch(h, SCR_SWEEP_NOISE, (size_t)L * sizeof(double), &p0); if (rc) return rc;
    rc = ensure_scratch(h, SCR_SWEEP_CAMS, 36 * sizeof(double), &p1); if (rc) return rc;
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

// What a device-resident sweep keeps over its chunks: trials are generated G at a time into `trials` (the generator
// shares one pass per seed among its noise levels, one warp per seed, so it wants many seeds per launch) and solved C at
// a time in `b`.
struct Sweep {
    tvf_handle_t h; cudaStream_t st; Method m; double hi_x, hi_y;
    static constexpr int Q = 512;              // partial sums per level
    ChunkBufs b; int64_t C, G; double* trials;

    // buffers for chunks of problems of up to n points and `count` trials per generator range; ba: the adjustment's too
    int init(int n, int64_t count, bool ba) {
        // nothing crosses the bus, so the solver runs the device path's large chunks; the carve is the host path's because
        // the evaluation kernels read its per-problem outputs
        C = pick_chunk(h, count > 0 ? count : 1, false, pose_budget(n, false, ba));
        Slot& s = h->slot[0];
        int rc = ensure_arena(h, s, carve_pose(nullptr, n, C, true, false, ba, nullptr)); if (rc) return rc;
        carve_pose(s.arena, n, C, true, false, ba, &b);
        G = (count < 4 * C) ? count : 4 * C;
        void* p;
        rc = ensure_scratch(h, SCR_SWEEP_TRIALS, (size_t)G * 6 * n * sizeof(double), &p);
        trials = (double*)p;
        return rc;
    }

    // trials [first, first + count) of the L noise levels `noise` with cameras P and n points: generate them, solve them
    // with `calm` and reduce them against the ground truth `gt` into the partial sums `pp`; with `pb`, also bundle-adjust
    // each chunk's poses (experiments.m:127-141 with the library's adjustment) and reduce those into `pb`
    int run(int64_t first, int64_t count, int n, const double* noise, int L, const double* P, const double* calm,
            const double* gt, double* pp, double* pb) const {
        for (int64_t gdone = 0; gdone < count; gdone += G) {
            const int64_t Gc = (count - gdone < G) ? (count - gdone) : G;
            int rc = sweep_common(h, first + gdone, Gc, n, noise, L, P, hi_x, hi_y, trials, st); if (rc) return rc;
            for (int64_t off = 0; off < Gc; off += C) {
                const int64_t Bc = (Gc - off < C) ? (Gc - off) : C;
                ChunkBufs k = b;
                k.in = trials + off * 6 * n; k.calm = calm; k.iter_sum = nullptr;
                rc = run_pose_chunk(h, st, m, 0, n, Bc, k); if (rc) return rc;
                launch_sweep_eval_accumulate(b.Rt2, b.Rt3, b.repr, b.status, first + gdone + off, Bc, L, Q, gt, pp, st);
                h->launches += 1;
                if (!pb) continue;
                // a trial without a pose starts from NaN: the kernel copies it through with TVF_ST_NONFINITE and iter = 0
                const BaArgs a{k.in, calm, 0, n, Bc, b.Rt2, b.Rt3, b.reconst, b.ba_Rt2, b.ba_Rt3, b.ba_X, b.ba_Xc, b.ba_repr,
                               b.ba_iter, b.ba_status};
                rc = ba_launched(h, launch_bundle_adjust(a, st), "bundle_adjust_kernel"); if (rc) return rc;
                launch_sweep_eval_accumulate(b.ba_Rt2, b.ba_Rt3, b.ba_repr, b.status, first + gdone + off, Bc, L, Q, gt, pb, st,
                                             b.ba_status, b.ba_iter);
                h->launches += 1;
            }
        }
        return TVF_OK;
    }
};

// experiments.m:74-124 for one method, device-resident: generate the trials of the sweep, solve them, and
// reduce ReprError / AngError per noise level.  Only the L x 5 table crosses the bus.
int tvf_sweep_run(tvf_handle_t h, int method, int64_t first_trial, int64_t B, int n, const double* noise_levels, int L,
                  const double* P, double hi_x, double hi_y, const double* calm, const double* Rt0_2, const double* Rt0_3,
                  double* table) {
    int rc = sweep_check(h, first_trial, B, n, noise_levels, L, P, table); if (rc) return rc;
    Method m;
    if (!calm || !Rt0_2 || !Rt0_3 || !method_of(method, &m))
        return fail(h, TVF_ERR_ARG, "method must be 1 (linear TFT), 7 (linear F) or 8 (optimal F); calm/Rt0 required");
    if (m != METHOD_TFT && n < 8) return fail(h, TVF_ERR_TOO_FEW_POINTS, TVF_LINEARF_ERRMSG);
    TVF_CK(cudaSetDevice(h->device));
    Sweep sw{h, h->slot[0].stream, m, hi_x, hi_y};
    const cudaStream_t st = sw.st;
    const int Q = Sweep::Q;
    rc = sw.init(n, B, false); if (rc) return rc;
    void *pc, *pr, *pp, *pt;
    rc = ensure_scratch(h, SCR_SWEEP_CALM, 27 * sizeof(double), &pc); if (rc) return rc;
    rc = ensure_scratch(h, SCR_SWEEP_GT, 24 * sizeof(double), &pr); if (rc) return rc;
    rc = ensure_scratch(h, SCR_SWEEP_PARTIAL, (size_t)L * Q * 5 * sizeof(double), &pp); if (rc) return rc;
    rc = ensure_scratch(h, SCR_SWEEP_TABLE, (size_t)L * 5 * sizeof(double), &pt); if (rc) return rc;
    TVF_CK(cudaMemcpyAsync(pc, calm, 27 * sizeof(double), cudaMemcpyHostToDevice, st));
    TVF_CK(cudaMemcpyAsync(pr, Rt0_2, 12 * sizeof(double), cudaMemcpyHostToDevice, st));
    TVF_CK(cudaMemcpyAsync((double*)pr + 12, Rt0_3, 12 * sizeof(double), cudaMemcpyHostToDevice, st));
    TVF_CK(cudaMemsetAsync(pp, 0, (size_t)L * Q * 5 * sizeof(double), st));
    rc = sw.run(first_trial, B, n, noise_levels, L, P, (const double*)pc, (const double*)pr, (double*)pp, nullptr);
    if (rc) return rc;
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
// ba: each chunk's poses are then bundle-adjusted and reduced into columns 5-10 of an L x 11 table; without it the table
// is L x 5 and the chunk size, and so every sum, is unchanged.
static int sweep_levels(tvf_handle_t h, int method, int64_t first_trial, int64_t B, const tvf_sweep_level* levels, int L,
                        double hi_x, double hi_y, double* table, bool ba) {
    if (!h) return TVF_ERR_ARG;
    if (!levels || !table || L < 1 || B < 0 || first_trial < 0) return fail(h, TVF_ERR_ARG, "NULL argument or bad size");
    Method m;
    if (!method_of(method, &m)) return fail(h, TVF_ERR_ARG, "method must be 1 (linear TFT), 7 (linear F) or 8 (optimal F)");
    if ((first_trial + B) / L + 1 > 0xffffffffLL) return fail(h, TVF_ERR_ARG, "seed exceeds 32 bits");
    int n_max = 1;
    for (int l = 0; l < L; ++l) {
        if (levels[l].n < 1 || levels[l].n > SWEEP_MAX_N) return fail(h, TVF_ERR_ARG, "device scene generator supports 1 <= n <= 60");
        if (levels[l].n > n_max) n_max = levels[l].n;
    }
    TVF_CK(cudaSetDevice(h->device));
    Sweep sw{h, h->slot[0].stream, m, hi_x, hi_y};
    const cudaStream_t st = sw.st;
    const int Q = Sweep::Q;
    const int W = ba ? 11 : 5;                 // table columns
    int rc = sw.init(n_max, B / L + 1, ba); if (rc) return rc;
    void *pc, *pr, *pp, *pt, *pb = nullptr;
    rc = ensure_scratch(h, SCR_SWEEP_CALM, (size_t)L * 27 * sizeof(double), &pc); if (rc) return rc;
    rc = ensure_scratch(h, SCR_SWEEP_GT, (size_t)L * 24 * sizeof(double), &pr); if (rc) return rc;
    rc = ensure_scratch(h, SCR_SWEEP_PARTIAL, (size_t)L * Q * 5 * sizeof(double), &pp); if (rc) return rc;
    rc = ensure_scratch(h, SCR_SWEEP_TABLE, (size_t)L * W * sizeof(double), &pt); if (rc) return rc;
    if (ba) { rc = ensure_scratch(h, SCR_SWEEP_BA_PARTIAL, (size_t)L * Q * 6 * sizeof(double), &pb); if (rc) return rc; }
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
        const int n = levels[l].n;
        if ((m != METHOD_TFT && n < 8) || n < 7) { skipped[(size_t)l] = 1; continue; }          // experiments.m:99-104: "not enough matches"
        if (q_hi <= q_lo) continue;
        rc = sw.run(q_lo, q_hi - q_lo, n, &levels[l].noise, 1, levels[l].P, (const double*)pc + (size_t)l * 27,
                    (const double*)pr + (size_t)l * 24, (double*)pp + (size_t)l * Q * 5, ba ? (double*)pb + (size_t)l * Q * 6 : nullptr);
        if (rc) return rc;
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
    return host_call(h, BundleAdjust{BaArgs{corresp, calm, calm_batched, n, 0, Rt2_0, Rt3_0, reconst0, Rt2, Rt3, reconst, nullptr,
                                            repr_err, iter, status}}, B);
}

int tvf_bundle_adjust_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                          const double* Rt2_0, const double* Rt3_0, const double* reconst0, double* Rt2, double* Rt3,
                          double* reconst, double* repr_err, int32_t* iter, int32_t* status) {
    return ba_dev(h, BundleAdjust{BaArgs{corresp, calm, calm_batched, n, 0, Rt2_0, Rt3_0, reconst0, Rt2, Rt3, reconst, nullptr,
                                         repr_err, iter, status}}, B);
}

int tvf_ba_covariance(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                      const double* Rt2, const double* Rt3, const double* reconst, double* cov_cam, double* cov_pts,
                      double* sigma2, int32_t* status) {
    return host_call(h, Covariance{BaCovArgs{corresp, calm, calm_batched, n, 0, Rt2, Rt3, reconst, cov_cam, cov_pts, sigma2, status}}, B);
}

int tvf_ba_covariance_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                          const double* Rt2, const double* Rt3, const double* reconst, double* cov_cam, double* cov_pts,
                          double* sigma2, int32_t* status) {
    return ba_dev(h, Covariance{BaCovArgs{corresp, calm, calm_batched, n, 0, Rt2, Rt3, reconst, cov_cam, cov_pts, sigma2, status}}, B);
}

int tvf_bundle_adjust_ragged(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, const int64_t* offsets,
                             int64_t B, const double* Rt2_0, const double* Rt3_0, const double* reconst0, double* Rt2,
                             double* Rt3, double* reconst, double* repr_err, int32_t* iter, int32_t* status) {
    BundleAdjust c{BaArgs{corresp, calm, calm_batched, 0, 0, Rt2_0, Rt3_0, reconst0, Rt2, Rt3, reconst, nullptr, repr_err, iter,
                          status}};
    c.rg.offs = offsets;
    return host_call(h, c, B);
}

int tvf_bundle_adjust_ragged_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched,
                                 const int64_t* offsets, int64_t B, const double* Rt2_0, const double* Rt3_0,
                                 const double* reconst0, double* Rt2, double* Rt3, double* reconst, double* repr_err,
                                 int32_t* iter, int32_t* status) {
    BundleAdjust c{BaArgs{corresp, calm, calm_batched, 0, 0, Rt2_0, Rt3_0, reconst0, Rt2, Rt3, reconst, nullptr, repr_err, iter,
                          status}};
    c.rg.offs = offsets;
    return ba_dev(h, c, B);
}

static int ba_robust_call(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                          int loss, double scale, const double* Rt2_0, const double* Rt3_0, const double* reconst0,
                          double* Rt2, double* Rt3, double* reconst, double* repr_err, double* cost, double* weights,
                          int32_t* iter, int32_t* status, bool dev, const int64_t* offsets = nullptr) {
    BundleAdjustRobust c{};
    c.io = BaArgs{corresp, calm, calm_batched, n, 0, Rt2_0, Rt3_0, reconst0, Rt2, Rt3, reconst, nullptr, repr_err, iter,
                  status};
    c.rio = BaRobustArgs{loss, scale, cost, weights};
    c.rg.offs = offsets;
    return dev ? ba_dev(h, c, B) : host_call(h, c, B);
}

int tvf_bundle_adjust_robust(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                             int loss, double scale, const double* Rt2_0, const double* Rt3_0, const double* reconst0,
                             double* Rt2, double* Rt3, double* reconst, double* repr_err, double* cost, double* weights,
                             int32_t* iter, int32_t* status) {
    return ba_robust_call(h, corresp, calm, calm_batched, n, B, loss, scale, Rt2_0, Rt3_0, reconst0, Rt2, Rt3, reconst,
                          repr_err, cost, weights, iter, status, false);
}

int tvf_bundle_adjust_robust_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n,
                                 int64_t B, int loss, double scale, const double* Rt2_0, const double* Rt3_0,
                                 const double* reconst0, double* Rt2, double* Rt3, double* reconst, double* repr_err,
                                 double* cost, double* weights, int32_t* iter, int32_t* status) {
    return ba_robust_call(h, corresp, calm, calm_batched, n, B, loss, scale, Rt2_0, Rt3_0, reconst0, Rt2, Rt3, reconst,
                          repr_err, cost, weights, iter, status, true);
}

int tvf_bundle_adjust_robust_ragged(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched,
                                    const int64_t* offsets, int64_t B, int loss, double scale, const double* Rt2_0,
                                    const double* Rt3_0, const double* reconst0, double* Rt2, double* Rt3, double* reconst,
                                    double* repr_err, double* cost, double* weights, int32_t* iter, int32_t* status) {
    return ba_robust_call(h, corresp, calm, calm_batched, 0, B, loss, scale, Rt2_0, Rt3_0, reconst0, Rt2, Rt3, reconst,
                          repr_err, cost, weights, iter, status, false, offsets);
}

int tvf_bundle_adjust_robust_ragged_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched,
                                        const int64_t* offsets, int64_t B, int loss, double scale, const double* Rt2_0,
                                        const double* Rt3_0, const double* reconst0, double* Rt2, double* Rt3,
                                        double* reconst, double* repr_err, double* cost, double* weights, int32_t* iter,
                                        int32_t* status) {
    return ba_robust_call(h, corresp, calm, calm_batched, 0, B, loss, scale, Rt2_0, Rt3_0, reconst0, Rt2, Rt3, reconst,
                          repr_err, cost, weights, iter, status, true, offsets);
}

int tvf_ba_covariance_ragged(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, const int64_t* offsets,
                             int64_t B, const double* Rt2, const double* Rt3, const double* reconst, double* cov_cam,
                             double* cov_pts, double* sigma2, int32_t* status) {
    Covariance c{BaCovArgs{corresp, calm, calm_batched, 0, 0, Rt2, Rt3, reconst, cov_cam, cov_pts, sigma2, status}};
    c.rg.offs = offsets;
    return host_call(h, c, B);
}

int tvf_ba_covariance_ragged_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched,
                                 const int64_t* offsets, int64_t B, const double* Rt2, const double* Rt3,
                                 const double* reconst, double* cov_cam, double* cov_pts, double* sigma2, int32_t* status) {
    Covariance c{BaCovArgs{corresp, calm, calm_batched, 0, 0, Rt2, Rt3, reconst, cov_cam, cov_pts, sigma2, status}};
    c.rg.offs = offsets;
    return ba_dev(h, c, B);
}

static Method ransac_method(int method) { return method == 1 ? METHOD_TFT : (method == 7 ? METHOD_F : METHOD_FIVEPT); }
static int ransac_sample_size(int method) { return method == 1 ? 7 : (method == 7 ? 8 : 5); }

static int ransac_call(tvf_handle_t h, int method, const double* corresp, const double* calm, int calm_batched, int n,
                       int64_t B, int hypotheses, double threshold, const uint64_t* seeds, double* Rt2, double* Rt3,
                       uint8_t* inliers, int32_t* n_inliers, int32_t* sample, int32_t* status, bool dev,
                       const int64_t* offsets = nullptr) {
    if (!h) return TVF_ERR_ARG;
    if (method != 1 && method != 7 && method != 9)
        return fail(h, TVF_ERR_ARG, "ransac_pose: method must be 1 (linear TFT), 7 (linear F) or 9 (five-point)");
    RansacArgs io{};
    io.corresp = corresp; io.calm = calm; io.calm_batched = calm_batched; io.n = n; io.seeds = seeds;
    io.Rt2 = Rt2; io.Rt3 = Rt3; io.inliers = inliers; io.n_inliers = n_inliers; io.sample = sample; io.status = status;
    Ransac c{ransac_method(method), ransac_sample_size(method), hypotheses, threshold, io};
    c.rg.offs = offsets;
    return dev ? ba_dev(h, c, B) : host_call(h, c, B);
}

int tvf_ransac_pose(tvf_handle_t h, int method, const double* corresp, const double* calm, int calm_batched, int n,
                    int64_t B, int hypotheses, double threshold, const uint64_t* seeds, double* Rt2, double* Rt3,
                    uint8_t* inliers, int32_t* n_inliers, int32_t* sample, int32_t* status) {
    return ransac_call(h, method, corresp, calm, calm_batched, n, B, hypotheses, threshold, seeds, Rt2, Rt3, inliers,
                       n_inliers, sample, status, false);
}

int tvf_ransac_pose_dev(tvf_handle_t h, int method, const double* corresp, const double* calm, int calm_batched, int n,
                        int64_t B, int hypotheses, double threshold, const uint64_t* seeds, double* Rt2, double* Rt3,
                        uint8_t* inliers, int32_t* n_inliers, int32_t* sample, int32_t* status) {
    return ransac_call(h, method, corresp, calm, calm_batched, n, B, hypotheses, threshold, seeds, Rt2, Rt3, inliers,
                       n_inliers, sample, status, true);
}

static int ransac_refined_call(tvf_handle_t h, int method, const double* corresp, const double* calm, int calm_batched,
                               int n, int64_t B, int hypotheses, double threshold, const uint64_t* seeds, int lo_rounds,
                               double* Rt2, double* Rt3, uint8_t* inliers, int32_t* n_inliers, int32_t* sample,
                               int32_t* lo_done, int32_t* status, bool dev, const int64_t* offsets = nullptr) {
    if (!h) return TVF_ERR_ARG;
    if (method != 1 && method != 7 && method != 9)
        return fail(h, TVF_ERR_ARG, "ransac_pose: method must be 1 (linear TFT), 7 (linear F) or 9 (five-point)");
    RansacArgs io{};
    io.corresp = corresp; io.calm = calm; io.calm_batched = calm_batched; io.n = n; io.seeds = seeds;
    io.Rt2 = Rt2; io.Rt3 = Rt3; io.inliers = inliers; io.n_inliers = n_inliers; io.sample = sample; io.status = status;
    io.lo_done = lo_done;
    RansacRefined c{Ransac{ransac_method(method), ransac_sample_size(method), hypotheses, threshold, io}, lo_rounds};
    c.rg.offs = offsets;
    return dev ? ba_dev(h, c, B) : host_call(h, c, B);
}

int tvf_ransac_pose_refined(tvf_handle_t h, int method, const double* corresp, const double* calm, int calm_batched, int n,
                            int64_t B, int hypotheses, double threshold, const uint64_t* seeds, int lo_rounds, double* Rt2,
                            double* Rt3, uint8_t* inliers, int32_t* n_inliers, int32_t* sample, int32_t* lo_done,
                            int32_t* status) {
    return ransac_refined_call(h, method, corresp, calm, calm_batched, n, B, hypotheses, threshold, seeds, lo_rounds, Rt2,
                               Rt3, inliers, n_inliers, sample, lo_done, status, false);
}

int tvf_ransac_pose_refined_dev(tvf_handle_t h, int method, const double* corresp, const double* calm, int calm_batched,
                                int n, int64_t B, int hypotheses, double threshold, const uint64_t* seeds, int lo_rounds,
                                double* Rt2, double* Rt3, uint8_t* inliers, int32_t* n_inliers, int32_t* sample,
                                int32_t* lo_done, int32_t* status) {
    return ransac_refined_call(h, method, corresp, calm, calm_batched, n, B, hypotheses, threshold, seeds, lo_rounds, Rt2,
                               Rt3, inliers, n_inliers, sample, lo_done, status, true);
}

int tvf_ransac_pose_ragged(tvf_handle_t h, int method, const double* corresp, const double* calm, int calm_batched,
                           const int64_t* offsets, int64_t B, int hypotheses, double threshold, const uint64_t* seeds,
                           double* Rt2, double* Rt3, uint8_t* inliers, int32_t* n_inliers, int32_t* sample, int32_t* status) {
    return ransac_call(h, method, corresp, calm, calm_batched, 0, B, hypotheses, threshold, seeds, Rt2, Rt3, inliers,
                       n_inliers, sample, status, false, offsets);
}

int tvf_ransac_pose_ragged_dev(tvf_handle_t h, int method, const double* corresp, const double* calm, int calm_batched,
                               const int64_t* offsets, int64_t B, int hypotheses, double threshold, const uint64_t* seeds,
                               double* Rt2, double* Rt3, uint8_t* inliers, int32_t* n_inliers, int32_t* sample,
                               int32_t* status) {
    return ransac_call(h, method, corresp, calm, calm_batched, 0, B, hypotheses, threshold, seeds, Rt2, Rt3, inliers,
                       n_inliers, sample, status, true, offsets);
}

int tvf_ransac_pose_refined_ragged(tvf_handle_t h, int method, const double* corresp, const double* calm, int calm_batched,
                                   const int64_t* offsets, int64_t B, int hypotheses, double threshold, const uint64_t* seeds,
                                   int lo_rounds, double* Rt2, double* Rt3, uint8_t* inliers, int32_t* n_inliers,
                                   int32_t* sample, int32_t* lo_done, int32_t* status) {
    return ransac_refined_call(h, method, corresp, calm, calm_batched, 0, B, hypotheses, threshold, seeds, lo_rounds, Rt2,
                               Rt3, inliers, n_inliers, sample, lo_done, status, false, offsets);
}

int tvf_ransac_pose_refined_ragged_dev(tvf_handle_t h, int method, const double* corresp, const double* calm,
                                       int calm_batched, const int64_t* offsets, int64_t B, int hypotheses, double threshold,
                                       const uint64_t* seeds, int lo_rounds, double* Rt2, double* Rt3, uint8_t* inliers,
                                       int32_t* n_inliers, int32_t* sample, int32_t* lo_done, int32_t* status) {
    return ransac_refined_call(h, method, corresp, calm, calm_batched, 0, B, hypotheses, threshold, seeds, lo_rounds, Rt2,
                               Rt3, inliers, n_inliers, sample, lo_done, status, true, offsets);
}

int tvf_five_point_pose(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int64_t B, double* Rt2,
                        double* Rt3, double* E, int32_t* n_E, int32_t* status) {
    return host_call(h, FivePoint{{corresp, calm, calm_batched, Rt2, Rt3, E, n_E, status}}, B);
}

int tvf_five_point_pose_dev(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int64_t B,
                            double* Rt2, double* Rt3, double* E, int32_t* n_E, int32_t* status) {
    return ba_dev(h, FivePoint{{corresp, calm, calm_batched, Rt2, Rt3, E, n_E, status}}, B);
}

int tvf_consensus(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, int n, int64_t B,
                  const double* Rt2, const double* Rt3, double threshold, uint8_t* inliers, int32_t* n_inliers) {
    return host_call(h, Consensus{corresp, calm, calm_batched, n, Rt2, Rt3, threshold, inliers, n_inliers}, B);
}

int tvf_consensus_ragged(tvf_handle_t h, const double* corresp, const double* calm, int calm_batched, const int64_t* offsets,
                         int64_t B, const double* Rt2, const double* Rt3, double threshold, uint8_t* inliers,
                         int32_t* n_inliers) {
    Consensus c{corresp, calm, calm_batched, 0, Rt2, Rt3, threshold, inliers, n_inliers};
    c.rg.offs = offsets;
    return host_call(h, c, B);
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
