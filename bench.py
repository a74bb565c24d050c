#!/usr/bin/env python
"""bench.py -- throughput of the linear three-view pose path on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's algorithm on host cores (oracle port)
    python bench.py ... --dump-outputs DIR                   # + a seeded sample of the last timed step's outputs as .npy

A "step" is one pass of LinearTFTPoseEstimation (+ ReprError) over one batch of synthetic trials
of BASELINE.json config 3: experiments.m's noise sweep, n = 20 points, `--trials` (default
1 000 000) independent trials per GPU, inputs resident in HBM when the timed region starts.
Multi-GPU: one process per GPU (torchrun), contiguous ranges of the global trial index per rank,
no data-path collective (weak scaling: per-GPU work fixed); NCCL only carries the barrier and the
max-over-ranks of the device time.  Prints ONE JSON line on rank 0.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "3-view linear TFT pose solves/sec (LinearTFTPoseEstimation + ReprError, n=20)"
UNIT = "solves/s"


# ---- work model (SURVEY.md 8(d) / App. B): algorithmic figures per solve ------------------------
def tft_flops(n):
    return 19458 * n + 438212


def f_flops(n):
    return 8974 * n + 20995


def pose_bytes(n):
    return 72 * n + 416


def kernel_flops(n):
    """App. B.1 rows attributed to the kernels of the TFT method (sums to tft_flops(n))."""
    return {
        "tft_stage1_kernel": 77 * n,             # normalise x3 + design matrix (the moments half of the split stage 1)
        "tft_stage1_solve_kernel": 5832 * n + 216513,  # null vector of A (4n x 27) (the solve half)
        "tft_epipoles_kernel": 2592,             # 8 svd3 (linearTFT.m:71-79)
        "tft_stage2_kernel": 5040 * n + 214000,  # svd(E), A*Up, its null vector, Up*tp, a; undo normalisation
        "candidates_kernel": 4922,               # de-calibrate, 8 svd3, E21/E31, 2 x svd(E) -> R, Rp, t
        "votes_kernel": 6632 * n,                # 8 two-view DLTs per point + signs
        "scale_kernel": 846 * n + 60,            # two-view DLT per point + closed-form lambda
        "final_kernel": 1031 * n + 125,          # three-view DLT per point + ReprError
        "pose_tail_fused_kernel": 8509 * n + 185,  # votes + scale + final in one launch (n <= 256)
    }


# ---- oracle-based CPU legs (the only place bench.py touches oracle/) -----------------------------
def _cpu_worker(args):
    import oracle as o
    Cs, CalM = args
    K = [CalM[0:3], CalM[3:6], CalM[6:9]]
    acc = 0.0
    for C_ in Cs:
        R2, R3, Rec, T, _ = o.LinearTFTPoseEstimation(C_, CalM)
        acc += o.ReprError([K[0] @ np.eye(3, 4), K[1] @ R2, K[2] @ R3], C_, Rec)
    return acc


def _pool_init():
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)
    except Exception:
        pass


def cpu_solves_per_sec(Corresp, CalM, cores, pool):
    """Oracle port of LinearTFTPoseEstimation+ReprError over `Corresp` (S,6,n) on `cores` processes."""
    S = Corresp.shape[0]
    parts = np.array_split(np.arange(S), cores * 4)
    jobs = [(Corresp[p], CalM) for p in parts if p.size]
    t0 = time.perf_counter()
    if pool is None:
        for j in jobs:
            _cpu_worker(j)
    else:
        pool.map(_cpu_worker, jobs)
    dt = time.perf_counter() - t0
    return S / dt, dt


def make_pool(cores):
    if cores <= 1:
        return None
    import multiprocessing as mp
    return mp.get_context("fork").Pool(cores, initializer=_pool_init)


# ---- clocks --------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.path = tempfile.mktemp(prefix="tvf_clocks_", suffix=".csv")
        self.proc = None
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(device), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, pw = [], [], []
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1])); mx.append(float(p[2])); pw.append(float(p[3]))
                except ValueError:
                    continue
                for nm, val in zip(names, p[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(nm)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            # "under load": samples in the upper half of the observed power range
            thr = (max(pw) + min(pw)) / 2.0
            load = [s for s, w in zip(sm, pw) if w >= thr] or sm
            out = {"sm_mhz": float(np.median(load)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm), "power_w_max": float(max(pw))}
        return out


def ncu_counters():
    """Per-kernel hardware counters of the committed ncu captures (profiles/*_counters.json, written by
    tools/ncu_summary.py from separate profiled runs of this same bench command): kernel name ->
    counters + the number of problems its captured launch processed."""
    import glob
    out = {}
    for f in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_counters.json"))):
        try:
            d = json.load(open(f))
        except Exception:
            continue
        for name, c in d.get("kernels", {}).items():
            c = dict(c); c["problems_per_launch"] = d["problems_per_launch"]; c["file"] = os.path.relpath(f, ROOT)
            out[name] = c
    return out


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


# ---- reference arm -------------------------------------------------------------------------------
def run_reference(args, rank, world):
    if rank != 0:
        return
    from tft_vs_fund_b200 import scene
    cores = os.cpu_count() or 1
    S = args.cpu_sample if args.cpu_sample > 0 else 250 * cores       # ~2.5 s of oracle work per core and step
    d = scene.sweep_batch(S, args.n, workers=min(cores, 16))
    pool = make_pool(cores)
    for _ in range(args.warmup):
        cpu_solves_per_sec(d["Corresp"][: max(cores * 8, S // 8)], d["CalM"], cores, pool)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_solves_per_sec(d["Corresp"], d["CalM"], cores, pool)
    dt = time.perf_counter() - t0
    if pool is not None:
        pool.close()
    value = S * args.steps / dt
    sample = "first %d trials of the sweep per step (of %d in the GPU arm's step)" % (S, args.trials)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "experiments.m noise sweep, n=%d, %d trials per GPU (BASELINE config 3)" % (args.n, args.trials),
                   "method": "LinearTFTPoseEstimation", "n_points": args.n, "trials_per_gpu": args.trials},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "note": "NumPy/LAPACK restatement of the reference's MATLAB (oracle/), not MATLAB itself: "
                                 "neither MATLAB nor Octave exists in this image"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---- GPU arm -------------------------------------------------------------------------------------
def run_gpu(args, rank, local_rank, world):
    from tft_vs_fund_b200 import scene, _lib
    n, B = args.n, args.trials
    cores = os.cpu_count() or 1

    # 1. a host-generated sample of the step's first trials: CPU-baseline input and cross-check of the device generator
    CalM = scene.sweep_batch(1, n)["CalM"]
    S = 0
    sample = None
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        S = args.cpu_sample if args.cpu_sample > 0 else min(B, 200 * cores)
        sample = scene.sweep_batch(S, n, first_trial=rank * B, workers=max(1, min(16, cores)))
        # 2. CPU baseline beside it (rank 0, N=1 only), before CUDA is initialised (the pool forks)
        pool = make_pool(cores)
        cpu_solves_per_sec(sample["Corresp"][: max(8, S // 10)], CalM, cores, pool)      # warm the pool
        v, dt = cpu_solves_per_sec(sample["Corresp"][:S], CalM, cores, pool)
        if pool is not None:
            pool.close()
        cpu_baseline = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": "first %d of the step's %d trials, %.1f s wall" % (S, B, dt),
                        "note": "oracle/ NumPy+LAPACK restatement of the MATLAB reference, one process per core"}

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    h = _lib.Handle(local_rank)
    lib = h.lib
    stream = torch.cuda.Stream(device=dev)
    h.call("tvf_set_stream", C.c_void_p(stream.cuda_stream))
    if args.chunk > 0:
        h.call("tvf_set_chunk", args.chunk)

    # 3. inputs generated on the device (tvf_generate_sweep_dev: one thread per trial), outputs preallocated
    t_gen = time.perf_counter()
    d_corresp = torch.empty((B, n, 6), dtype=torch.float64, device=dev)
    scene.sweep_batch_device(B, n, first_trial=rank * B, device=local_rank, out_ptr=d_corresp.data_ptr(), meta=False)
    torch.cuda.synchronize(dev)
    t_gen = time.perf_counter() - t_gen
    t_gen2 = time.perf_counter()                                             # second call: no first-launch set-up cost
    scene.sweep_batch_device(B, n, first_trial=rank * B, device=local_rank, out_ptr=d_corresp.data_ptr(), meta=False)
    torch.cuda.synchronize(dev)
    t_gen2 = time.perf_counter() - t_gen2
    corresp_host = d_corresp.cpu().numpy()                                   # for the end-to-end (host-pointer) leg
    gen_check = None
    if sample is not None:
        dd = np.abs(corresp_host[:S] - sample["Corresp"].transpose(0, 2, 1))
        gen_check = {"trials": int(S), "max_abs_diff_vs_host_generator": float(dd.max()), "bitwise_equal_fraction": float(np.mean(dd == 0.0))}
    d_calm = torch.from_numpy(np.ascontiguousarray(CalM.T)).to(dev)
    d_Rt2 = torch.empty((B, 12), dtype=torch.float64, device=dev)
    d_Rt3 = torch.empty((B, 12), dtype=torch.float64, device=dev)
    d_rec = torch.empty((B, 3 * n), dtype=torch.float64, device=dev)
    d_T = torch.empty((B, 27), dtype=torch.float64, device=dev)
    d_rep = torch.empty((B,), dtype=torch.float64, device=dev)
    d_st = torch.zeros((B,), dtype=torch.int32, device=dev)
    ptr = lambda t: C.c_void_p(t.data_ptr())

    def step_tft():
        h.call("tvf_linear_tft_pose_dev", ptr(d_corresp), ptr(d_calm), 0, n, B, ptr(d_Rt2), ptr(d_Rt3), ptr(d_rec),
               ptr(d_T), ptr(d_rep), ptr(d_st))

    def step_f():
        h.call("tvf_linear_f_pose_dev", ptr(d_corresp), ptr(d_calm), 0, n, B, ptr(d_Rt2), ptr(d_Rt3), ptr(d_rec),
               ptr(d_T), ptr(d_rep), None, None, ptr(d_st))

    d_iter = torch.zeros((B,), dtype=torch.int32, device=dev)

    def step_optf():
        h.call("tvf_optim_f_pose_dev", ptr(d_corresp), ptr(d_calm), 0, n, B, ptr(d_Rt2), ptr(d_Rt3), ptr(d_rec),
               ptr(d_T), ptr(d_rep), None, None, ptr(d_iter), ptr(d_st))

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def timed(step, steps, profile=False):
        """K steps on `stream`, bracketed by barrier + synchronize, timed with CUDA events on that stream."""
        if profile:
            h.call("tvf_profile_reset"); h.call("tvf_profile_enable", 1)
        barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(steps):
                step()
            e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        prof = None
        if profile:
            tot = (C.c_double * _lib.NUM_KERNELS)(); cnt = (C.c_int64 * _lib.NUM_KERNELS)()
            h.call("tvf_profile_read", tot, cnt)
            h.call("tvf_profile_enable", 0)
            prof = {lib.tvf_kernel_name(i).decode(): (tot[i], cnt[i]) for i in range(_lib.NUM_KERNELS) if cnt[i]}
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, prof

    fp64_peak = lib.tvf_fp64_peak_tflops(h._h)

    # 4. warm-up, then the timed region (with the clock sampler running)
    for _ in range(max(3, args.warmup)):
        step_tft()
    torch.cuda.synchronize(dev)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    l0 = lib.tvf_launch_count(h._h)
    ms, prof = timed(step_tft, args.steps, profile=True)
    launches = lib.tvf_launch_count(h._h) - l0
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:            # before the other legs reuse the output buffers
        dump_outputs(args.dump_outputs, B, n, {"R_t_2": d_Rt2, "R_t_3": d_Rt3, "Reconst": d_rec, "T": d_T,
                                                "repr_err": d_rep, "status": d_st})
    flagged = int(torch.count_nonzero(d_st).item())
    flagged_detail = None
    if flagged:
        idxs = torch.nonzero(d_st).reshape(-1)[:8].cpu().numpy()
        flagged_detail = [{"trial": int(rank * B + i), "status": int(d_st[int(i)].item())} for i in idxs]
    value = world * B * args.steps / (ms * 1e-3)
    rep_device_path = d_rep.cpu().numpy()

    full = args.legs == "all"
    f_value = ms_f = optf_value = ms_o = optf_iters = e2e_value = e2e_check = sweep_value = None
    e2e_variants = link = shard_check = e2e_pageable_check = None
    optf_steps = e2e_steps = 0
    gh_ms = (float("nan"), 1)
    h2d = B * n * 6 * 8 + 27 * 8
    d2h = B * (12 + 12 + 3 * n + 27 + 1) * 8 + B * 4
    table = np.zeros((13, 5))
    if full:
        # F method, same inputs (reported beside the headline)
        for _ in range(3):
            step_f()
        ms_f, _ = timed(step_f, max(3, args.steps // 2))
        f_value = world * B * max(3, args.steps // 2) / (ms_f * 1e-3)

        # OptimFPoseEstimation (Gauss-Helmert refinement of both F; SURVEY 8 f4), same inputs
        optf_steps = max(3, args.steps // 4)
        for _ in range(2):
            step_optf()
        ms_o, prof_o = timed(step_optf, optf_steps, profile=True)
        optf_value = world * B * optf_steps / (ms_o * 1e-3)
        optf_iters = float(d_iter.double().mean().item())
        gh_ms = prof_o.get("optimf_gh_kernel", (float("nan"), 1)) if prof_o else (float("nan"), 1)

        # 5. end to end through the host-pointer C ABI: host buffers, H2D + kernels + D2H inside the timed region.
        #    Headline `e2e`: pinned buffers (tvf_host_alloc), every output of the reference signature.  Beside it:
        #    `lean` (Reconst and T not requested -- the ABI takes NULL; 204 B instead of 900 B back per solve),
        #    `pageable` (plain malloc'ed buffers, what a MEX caller's mxArrays are) and `registered` (the same pageable
        #    buffers page-locked by tvf_set_host_register for the duration of each call).
        lib.tvf_host_alloc.restype = C.c_void_p

        def pinned(shape, dtype=np.float64):
            nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
            p = lib.tvf_host_alloc(nbytes)
            if not p:
                raise RuntimeError("tvf_host_alloc failed")
            buf = (C.c_char * nbytes).from_address(p)
            return np.frombuffer(buf, dtype=dtype).reshape(shape), p

        h_in, p0 = pinned((B, n, 6)); h_in[...] = corresp_host
        h_calm = np.ascontiguousarray(CalM.T)
        h_Rt2, p1 = pinned((B, 12)); h_Rt3, p2 = pinned((B, 12)); h_rec, p3 = pinned((B, 3 * n))
        h_T, p4 = pinned((B, 27)); h_rep, p5 = pinned((B,)); h_st, p6 = pinned((B,), np.int32)
        dp = lambda a: a.ctypes.data_as(_lib.c_double_p) if a is not None else None

        def make_step(bufs, lean):
            i_, r2_, r3_, rec_, T_, rep_, st_ = bufs
            def step():
                return h.call("tvf_linear_tft_pose", dp(i_), dp(h_calm), 0, n, B, dp(r2_), dp(r3_), None if lean else dp(rec_),
                              None if lean else dp(T_), dp(rep_), st_.ctypes.data_as(_lib.c_int32_p))
            return step

        def time_e2e(step, steps):
            for _ in range(2):
                step()
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                step()
            torch.cuda.synchronize(dev)
            dt = time.perf_counter() - t0
            if world > 1:
                t = torch.tensor([dt], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            barrier()
            return world * B * steps / dt

        pinned_bufs = (h_in, h_Rt2, h_Rt3, h_rec, h_T, h_rep, h_st)
        e2e_steps = max(3, min(args.steps, 10))
        e2e_value = time_e2e(make_step(pinned_bufs, False), e2e_steps)
        e2e_check = float(np.abs(h_rep - rep_device_path).max())       # host path and device path agree bit for bit
        h2d = B * n * 6 * 8 + 27 * 8
        d2h = B * (12 + 12 + 3 * n + 27 + 1) * 8 + B * 4
        e2e_variants = {"pinned_all_outputs": {"value": e2e_value, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h}}
        e2e_variants["pinned_lean"] = {"value": time_e2e(make_step(pinned_bufs, True), e2e_steps), "h2d_bytes_per_step": h2d,
                                       "d2h_bytes_per_step": B * (12 + 12 + 1) * 8 + B * 4,
                                       "note": "Reconst and T not requested (NULL): R_t_2, R_t_3, repr_err, status only"}
        # pageable buffers (np.empty): a MEX caller's situation
        pg = (corresp_host.copy(), np.empty((B, 12)), np.empty((B, 12)), np.empty((B, 3 * n)), np.empty((B, 27)), np.empty(B),
              np.zeros(B, dtype=np.int32))
        steps_pg = max(2, min(args.steps, 4))
        e2e_variants["pageable"] = {"value": time_e2e(make_step(pg, False), steps_pg), "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                                    "note": "np.empty buffers: the CUDA runtime stages every copy through its own pinned buffer"}
        e2e_pageable_check = float(np.abs(pg[5] - rep_device_path).max())
        h.call("tvf_set_host_register", 1)
        e2e_variants["pageable_registered_per_call"] = {
            "value": time_e2e(make_step(pg, False), steps_pg), "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "note": "same buffers, page-locked by cudaHostRegister inside every call and released before it returns (TVF_HOST_REGISTER=1 in the MEX gateways)"}
        h.call("tvf_set_host_register", 0)
        del pg

        # 5a. what the host link allows: pinned H2D and D2H copies running at once on every rank (the e2e path is bound by
        #     this, not by the kernels).  Each direction repeats its buffer for ~the same duration and is timed with CUDA
        #     events on its own stream, so both rates are measured under bidirectional load.
        def link_rates():
            nin = B * n * 6; nout = B * 3 * n                     # doubles: the pinned input buffer, the pinned Reconst buffer
            d_i = torch.empty(nin, dtype=torch.float64, device=dev); d_o = torch.ones(nout, dtype=torch.float64, device=dev)
            hin = torch.from_numpy(h_in.reshape(-1)); hout = torch.from_numpy(h_rec.reshape(-1))
            s1, s2 = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            def once(reps_in, reps_out):
                with torch.cuda.stream(s1):
                    ev[0].record(s1)
                    for _ in range(reps_in):
                        d_i.copy_(hin, non_blocking=True)
                    ev[1].record(s1)
                with torch.cuda.stream(s2):
                    ev[2].record(s2)
                    for _ in range(reps_out):
                        hout.copy_(d_o, non_blocking=True)
                    ev[3].record(s2)
                s1.synchronize(); s2.synchronize()
                t_in = ev[0].elapsed_time(ev[1]) * 1e-3 if reps_in else 1.0
                t_out = ev[2].elapsed_time(ev[3]) * 1e-3 if reps_out else 1.0
                return reps_in * nin * 8 / t_in / 1e9, reps_out * nout * 8 / t_out / 1e9
            out = []
            for reps in ((3, 6), (3, 0), (0, 6)):                 # both directions at once, H2D alone, D2H alone
                once(*reps); barrier()
                r = torch.tensor(once(*reps), dtype=torch.float64, device=dev)
                barrier()
                if world > 1:
                    dist.all_reduce(r, op=dist.ReduceOp.MIN)      # the slowest rank's link
                out.append((float(r[0].item()), float(r[1].item())))
            return out
        (h2d_both, d2h_both), (h2d_alone, _), (_, d2h_alone) = link_rates()
        link = {"h2d_gbs_per_gpu": h2d_both, "d2h_gbs_per_gpu": d2h_both, "aggregate_bidirectional_gbs": world * (h2d_both + d2h_both),
                "h2d_alone_gbs_per_gpu": h2d_alone, "d2h_alone_gbs_per_gpu": d2h_alone,
                "note": "pinned host memory, all ranks at once, CUDA events per stream, minimum over ranks; first pair: H2D and D2H "
                        "streams busy at the same time"}
        # time the link needs for one step's volumes -> ceiling of the e2e figures: neither direction faster than alone, and the
        # sum of both not faster than the bidirectional aggregate
        for k_, v_ in e2e_variants.items():
            bi, bo = v_["h2d_bytes_per_step"], v_["d2h_bytes_per_step"]
            t_need = max(bi / (h2d_alone * 1e9), bo / (d2h_alone * 1e9), (bi + bo) / ((h2d_both + d2h_both) * 1e9))
            v_["link_ceiling"] = world * B / t_need
            v_["frac_of_link_ceiling"] = v_["value"] / v_["link_ceiling"]
        for p in (p0, p1, p2, p3, p4, p5, p6):
            lib.tvf_host_free(C.c_void_p(p))

        # 5c. N > 1: shards == single device, checked on the hardware.  Rank 0 re-solves the first K trials of rank 1's
        #     shard on its own GPU and compares them bit for bit with what rank 1 computed.
        if world > 1:
            Kc = min(B, 65536)
            step_tft(); h.call("tvf_synchronize"); torch.cuda.synchronize(dev)      # the output buffers hold the other legs' results
            mine = torch.cat([d_Rt2[:Kc].reshape(-1), d_Rt3[:Kc].reshape(-1), d_T[:Kc].reshape(-1), d_rep[:Kc]]).clone()
            gathered = [torch.empty_like(mine) for _ in range(world)] if rank == 0 else None
            dist.gather(mine, gathered, dst=0)
            if rank == 0:
                tmp_c = torch.empty((Kc, n, 6), dtype=torch.float64, device=dev)
                scene.sweep_batch_device(Kc, n, first_trial=1 * B, device=local_rank, out_ptr=tmp_c.data_ptr(), meta=False)
                r2 = torch.empty((Kc, 12), dtype=torch.float64, device=dev); r3 = torch.empty_like(r2)
                tT = torch.empty((Kc, 27), dtype=torch.float64, device=dev); tr = torch.empty((Kc,), dtype=torch.float64, device=dev)
                ts = torch.zeros((Kc,), dtype=torch.int32, device=dev)
                h.call("tvf_linear_tft_pose_dev", ptr(tmp_c), ptr(d_calm), 0, n, Kc, ptr(r2), ptr(r3), None, ptr(tT), ptr(tr), ptr(ts))
                h.call("tvf_synchronize"); torch.cuda.synchronize(dev)
                ref = torch.cat([r2.reshape(-1), r3.reshape(-1), tT.reshape(-1), tr])
                shard_check = {"trials": int(Kc), "of_rank": 1, "recomputed_on_rank": 0,
                               "bitwise_equal": bool(torch.equal(ref.view(torch.int64), gathered[1].view(torch.int64)))}

        # 5b. the whole inner loop of experiments.m device-resident (generate + solve + per-level reduction; only a
        #     13 x 5 table crosses the bus): tvf_sweep_run
        K_, Ps_, Rt0_ = scene.scene_cameras(50, 0)
        lv = np.ascontiguousarray(np.arange(0.0, 3.0 + 1e-9, 0.25)); Pm = np.ascontiguousarray(np.stack(Ps_))
        g2 = np.ascontiguousarray(Rt0_[0].T); g3 = np.ascontiguousarray(Rt0_[1].T); table = np.zeros((lv.size, 5))

        def step_sweep():
            h.call("tvf_sweep_run", 1, rank * B, B, n, dp(lv), lv.size, dp(Pm), 1800.0, 1200.0, dp(h_calm), dp(g2), dp(g3), dp(table))

        step_sweep()
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            step_sweep()
        dt_sweep = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt_sweep], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt_sweep = float(t.item())
        sweep_value = world * B * 3 / dt_sweep

    # 5d. BASELINE config 5 inside the default line: 8 192 scenes x n = 10 000 (3.9 GB of input), single GPU
    large_n_block = None
    if full and rank == 0 and world == 1 and args.large_n_scenes > 0:
        try:
            large_n_block = large_n_measure(h, lib, local_rank, args.large_n_scenes, 10000, 3, 1)
        except Exception as e:                                      # never lose the headline over the extra block
            large_n_block = {"error": repr(e)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # 6. rooflines
    peaks = measured_peaks()
    hbm_peak = peaks["hbm_gbs"] if peaks else 6650.0
    hbm_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
    kf = kernel_flops(n)
    per_kernel = {}
    dom, dom_ms = None, -1.0
    tot_kernel_ms = sum(v[0] for v in prof.values())
    for name, (tms, cnt) in prof.items():
        per_kernel[name] = {"ms_total": tms, "launches": int(cnt), "share": tms / tot_kernel_ms if tot_kernel_ms else None}
        if tms > dom_ms:
            dom, dom_ms = name, tms
    units_per_launch = B * args.steps / prof[dom][1]                      # problems one launch of the dominant kernel handles
    avg_launch_s = dom_ms * 1e-3 / prof[dom][1]
    fp64_src = "measured on this device by tvf_fp64_peak_tflops (register-resident DFMA loop)"
    if not (fp64_peak and fp64_peak > 1.0):
        fp64_peak, fp64_src = 37.2, "nominal 148 SM x 64 FMA/clk x 1.965 GHz"
    ncu = ncu_counters()
    traffic = None
    if dom in ncu and ncu[dom].get("dram_bytes_per_launch"):
        traffic = ncu[dom]["dram_bytes_per_launch"] * units_per_launch / ncu[dom]["problems_per_launch"]
    # executed FP64 work per problem and kernel, from the committed ncu captures: 2*DFMA + DMUL + DADD thread instructions
    exec_flop_step = 0.0
    exec_known = True
    for name, c in ncu.items():
        if name in per_kernel and c.get("dram_bytes_per_launch") is not None:
            fl = c.get("fp64_flop_per_launch")
            per_kernel[name]["ncu"] = {"fp64_pipe_active_pct": c["fp64_pipe_active_pct"], "issue_active_pct": c["issue_active_pct"],
                                       "dram_bytes_per_problem": c["dram_bytes_per_launch"] / c["problems_per_launch"],
                                       "warp_instr_per_problem": c["warp_instructions"] / c["problems_per_launch"],
                                       "executed_fp64_flop_per_problem": (fl / c["problems_per_launch"] if fl else None),
                                       "registers": c["registers"], "from": c["file"]}
            if fl:
                ms_k, n_k = prof[name]
                tf = fl / c["problems_per_launch"] * (B * args.steps) / (ms_k * 1e-3) / 1e12      # live time, captured flop count
                per_kernel[name]["executed_tflops"] = tf
                per_kernel[name]["frac_executed"] = tf / fp64_peak
    for name in per_kernel:
        fl = per_kernel[name].get("ncu", {}).get("executed_fp64_flop_per_problem")
        if fl is None:
            exec_known = False
        else:
            exec_flop_step += fl
    step_s = ms * 1e-3 / args.steps
    dom_exec = per_kernel[dom].get("executed_tflops")
    alg_tf = kf[dom] * units_per_launch / avg_launch_s / 1e12
    roofline = {"bound": "fp64", "kernel": dom,
                "achieved": dom_exec, "peak": fp64_peak, "unit": "TFLOP/s", "frac": (dom_exec / fp64_peak if dom_exec else None),
                "frac_executed": (dom_exec / fp64_peak if dom_exec else None),
                "fp64_pipe_active_pct": (ncu[dom]["fp64_pipe_active_pct"] if dom in ncu else None),
                "traffic": traffic,
                "traffic_note": "dram__bytes_read+write of this kernel from the committed ncu --set full capture, scaled to this launch size",
                "peak_source": fp64_src,
                "work_model": "achieved = EXECUTED FP64 flop (2*DFMA + DMUL + DADD thread instructions of this kernel, ncu capture in "
                              "profiles/*_counters.json: %s flop per solve) x %.0f solves per launch / live CUDA-event launch time"
                              % (("%.0f" % per_kernel[dom]["ncu"]["executed_fp64_flop_per_problem"]) if dom_exec else "n/a", units_per_launch),
                "algorithmic_speedup_vs_peak": {
                    "value": alg_tf / fp64_peak, "achieved_algorithmic_tflops": alg_tf,
                    "note": "SURVEY.md 8(d) figure: the REFERENCE's operation count for this kernel's share (%d flop per solve, SVD-based) / "
                            "time / peak.  The GPU route (Gram + inverse + power iteration) executes ~10x fewer flops, so this exceeds 1; "
                            "it measures the algorithmic advantage, not hardware efficiency" % kf[dom]}}
    exec_step_tf = exec_flop_step * B / step_s / 1e12 if exec_known else None
    roofline_step = {"bound": "fp64", "achieved": exec_step_tf, "peak": fp64_peak, "unit": "TFLOP/s",
                     "frac": (exec_step_tf / fp64_peak if exec_step_tf else None),
                     "executed_fp64_flop_per_solve": (exec_flop_step if exec_known else None),
                     "fp64_pipe_active_pct_time_weighted": (sum(per_kernel[k]["ncu"]["fp64_pipe_active_pct"] * per_kernel[k]["ms_total"] for k in per_kernel
                                                                if "ncu" in per_kernel[k]) / tot_kernel_ms if exec_known else None),
                     "algorithmic_speedup_vs_peak": tft_flops(n) * B / step_s / 1e12 / fp64_peak,
                     "note": "whole step: executed FP64 flop of all kernels (ncu) / step time / measured DFMA peak; the algorithmic figure "
                             "(%d reference flop per solve, SURVEY.md 8d) is kept beside it" % tft_flops(n)}
    roofline_hbm = {"bound": "hbm", "achieved": pose_bytes(n) * B / step_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                    "frac": pose_bytes(n) * B / step_s / 1e9 / hbm_peak, "peak_source": hbm_src,
                    "note": "%d algorithmic bytes/solve; this path is FP64-bound at n=20, not HBM-bound" % pose_bytes(n)}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic (generateSyntheticScene + experiments.m sub-sampling, generated on the device)",
        "config": {"workload": "experiments.m noise sweep (13 levels 0:0.25:3), n=%d points, %d trials per GPU "
                               "(BASELINE config 3%s)" % (n, B, "" if world == 1 else "/4 sharded"),
                   "method": "LinearTFTPoseEstimation", "n_points": n, "trials_per_gpu": B, "global_trials": B * world,
                   "parallelism": "independent trial ranges per GPU, no collective",
                   "cache": "inputs+outputs per step (%.2f GB) exceed L2; no flush needed" % ((h2d + d2h) / 1e9)},
        "roofline": roofline, "roofline_step": roofline_step, "roofline_hbm": roofline_hbm,
        "kernels": per_kernel,
        "cpu_baseline": cpu_baseline,
        "e2e": ({"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                 "steps": e2e_steps, "max_abs_diff_vs_device_path": e2e_check,
                 "api": "tvf_linear_tft_pose (host pointers, pinned; chunked H2D/compute/D2H over 3 streams)",
                 "link_ceiling": e2e_variants["pinned_all_outputs"]["link_ceiling"],
                 "frac_of_link_ceiling": e2e_variants["pinned_all_outputs"]["frac_of_link_ceiling"]} if full else None),
        "e2e_variants": e2e_variants, "host_link": link, "e2e_pageable_max_abs_diff_vs_device_path": e2e_pageable_check,
        "shard_check": shard_check,
        "gpu_launches": int(launches),
        "clocks": clocks,
        "f_method": ({"metric": "3-view linear F pose solves/sec (LinearFPoseEstimation + ReprError)", "value": f_value,
                      "unit": UNIT, "ms_per_step": ms_f / max(3, args.steps // 2),
                      "roofline_step_frac_fp64": f_flops(n) * B / (ms_f * 1e-3 / max(3, args.steps // 2)) / 1e12 / fp64_peak}
                     if full else None),
        "optimf_method": ({"metric": "3-view optimal-F pose solves/sec (OptimFPoseEstimation + ReprError)", "value": optf_value,
                           "unit": UNIT, "ms_per_step": ms_o / optf_steps, "mean_gauss_helmert_iterations_per_solve": optf_iters,
                           "optimf_gh_kernel_share": gh_ms[0] / ms_o if ms_o > 0 else None} if full else None),
        "device_resident_sweep": ({"api": "tvf_sweep_run: trials generated, solved and reduced per noise level on the device",
                                   "value": sweep_value, "unit": UNIT, "d2h_bytes_per_step": int(table.nbytes),
                                   "mean_repr_err_px_by_level": (table[:, 0] / np.maximum(table[:, 3], 1)).round(4).tolist()}
                                  if full else None),
        "flagged_problems": flagged, "flagged_detail": flagged_detail,
        "large_n": large_n_block,
        "input_generation": {"where": "device (tvf_generate_sweep_dev, TVF scene RNG v2)", "seconds": t_gen, "seconds_warm": t_gen2, "trials_per_s_warm": B / t_gen2, "check": gen_check},
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


DUMP_MAX_TRIALS = 32768
DUMP_MAX_BYTES = 60 * 10 ** 6


def dump_outputs(out_dir, B, n, outputs):
    """Write what the last timed step handed its caller (`outputs`: name -> device tensor with one row per trial) as
    out_dir/<name>.npy in float64, for a fixed sample of trials drawn with a fixed seed (`trial.npy`: their indices),
    so that two builds run with the same arguments can be compared output for output.  At most DUMP_MAX_BYTES."""
    import torch
    per_trial = 8 * (sum(t[0].numel() for t in outputs.values()) + 1)
    S = min(B, DUMP_MAX_TRIALS, DUMP_MAX_BYTES // per_trial)
    idx = np.sort(np.random.default_rng(0).choice(B, size=S, replace=False))
    sel = torch.from_numpy(idx).to(next(iter(outputs.values())).device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "trial.npy"), idx.astype(np.float64))
    for name, t in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.index_select(0, sel).cpu().numpy().astype(np.float64))
    print("bench: wrote %d of %d trials' outputs (n = %d) to %s" % (S, B, n, out_dir), file=sys.stderr)


# ---- BASELINE config 5: large-n triplets (HBM-oriented Gram formation) ------------------------------
def large_n_scenes(B, n, dev, seed=1):
    """B scenes of generateSyntheticScene's geometry (f = 50, angle = 0), n points each, 1 px Gaussian noise, generated on
    the device with torch.  Points whose noisy projections leave the 1800 x 1200 image in any view are re-drawn until every
    point is inside (generateSyntheticScene.m:80-111 fills with fresh points in the same way; the random stream is
    torch's, not the reference generator's -- labelled in `data`)."""
    import torch
    from tft_vs_fund_b200 import scene
    K, Ps, R_t0 = scene.scene_cameras(50, 0)
    g = torch.Generator(device=dev); g.manual_seed(seed)
    Pt = [torch.from_numpy(P).to(dev) for P in Ps]
    hi = torch.tensor([36 * scene.PIX, 24 * scene.PIX] * 3, dtype=torch.float64, device=dev)
    out = torch.empty((B, n, 6), dtype=torch.float64, device=dev)
    step = max(1, (1 << 25) // n)
    for lo in range(0, B, step):
        hi_b = min(B, lo + step)
        chunk = out[lo:hi_b].view(-1, 6)
        todo = torch.arange(chunk.shape[0], device=dev)
        while todo.numel() > 0:
            X = torch.rand((todo.numel(), 3), dtype=torch.float64, device=dev, generator=g) * 400 - 200
            c = torch.empty((todo.numel(), 6), dtype=torch.float64, device=dev)
            for v in range(3):
                x = X @ Pt[v][:, :3].T + Pt[v][:, 3]
                c[:, 2 * v:2 * v + 2] = x[:, :2] / x[:, 2:3] + torch.randn((todo.numel(), 2), dtype=torch.float64, device=dev, generator=g)
            ok = ((c >= 0) & (c <= hi)).all(dim=1)
            chunk[todo[ok]] = c[ok]
            todo = todo[~ok]
    return out, np.tile(K, (3, 1))


def large_n_measure(h, lib, local_rank, B, n, steps, warmup):
    """Times LinearTFTPoseEstimation on B scenes of n points (device-resident) and returns the config-5 block: Gram
    formation (tft_moments_large_kernel) against the HBM and FP64 roofs, and the full pipeline."""
    import torch
    from tft_vs_fund_b200 import _lib
    dev = torch.device("cuda", local_rank)
    d_corresp, CalM = large_n_scenes(B, n, dev)
    stream = torch.cuda.Stream(device=dev)
    h.call("tvf_set_stream", C.c_void_p(stream.cuda_stream))
    d_calm = torch.from_numpy(np.ascontiguousarray(CalM.T)).to(dev)
    d_Rt2 = torch.empty((B, 12), dtype=torch.float64, device=dev); d_Rt3 = torch.empty_like(d_Rt2)
    d_rec = torch.empty((B, 3 * n), dtype=torch.float64, device=dev)
    d_T = torch.empty((B, 27), dtype=torch.float64, device=dev)
    d_rep = torch.empty((B,), dtype=torch.float64, device=dev); d_st = torch.zeros((B,), dtype=torch.int32, device=dev)
    ptr = lambda t: C.c_void_p(t.data_ptr())

    def step_fn():
        h.call("tvf_linear_tft_pose_dev", ptr(d_corresp), ptr(d_calm), 0, n, B, ptr(d_Rt2), ptr(d_Rt3), ptr(d_rec),
               ptr(d_T), ptr(d_rep), ptr(d_st))

    for _ in range(max(1, warmup)):
        step_fn()
    torch.cuda.synchronize(dev)
    h.call("tvf_profile_reset"); h.call("tvf_profile_enable", 1)
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        e0.record(stream)
        for _ in range(steps):
            step_fn()
        e1.record(stream)
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    tot = (C.c_double * _lib.NUM_KERNELS)(); cnt = (C.c_int64 * _lib.NUM_KERNELS)()
    h.call("tvf_profile_read", tot, cnt); h.call("tvf_profile_enable", 0)
    prof = {lib.tvf_kernel_name(i).decode(): (tot[i], cnt[i]) for i in range(_lib.NUM_KERNELS) if cnt[i]}
    peaks = measured_peaks()
    hbm_peak = peaks["hbm_gbs"] if peaks else 6650.0
    fp64_peak = lib.tvf_fp64_peak_tflops(h._h)
    gram_ms, gram_n = prof.get("tft_moments_large_kernel", (float("nan"), 1))
    gram_s = gram_ms * 1e-3 / max(1, gram_n)                       # one launch = all B scenes of the step (or a chunk)
    scenes_per_launch = B * steps / max(1, gram_n)
    gram_bytes = (48 * n + 216) * scenes_per_launch
    c5 = ncu_counters().get("tft_moments_large_kernel")
    gram_traffic = (c5["dram_bytes_per_launch"] * scenes_per_launch / c5["problems_per_launch"]
                    if c5 and c5.get("dram_bytes_per_launch") and n == 10000 else None)
    flop_exec = (c5["fp64_flop_per_launch"] / c5["problems_per_launch"]) if c5 and c5.get("fp64_flop_per_launch") and n == 10000 else None
    block = {
        "metric": "large-n linearTFT Gram formation (normalisation + 96 moments), scenes/s", "unit": "scenes/s",
        "value": scenes_per_launch / gram_s, "steps": steps, "ms_per_step": ms / steps,
        "data": "synthetic (device-generated scenes of generateSyntheticScene's geometry, 1 px noise, out-of-image points re-drawn; torch RNG)",
        "config": {"workload": "large-n triplets: %d correspondences per scene x %d scenes (BASELINE config 5%s)"
                               % (n, B, "" if B >= 65536 else "; 65536 scenes with --workload large-n --trials 65536"),
                   "n_points": n, "scenes": B, "cache": "%.1f GB of input per step, far beyond L2" % (B * n * 48 / 1e9)},
        "roofline": {"bound": "hbm", "kernel": "tft_moments_large_kernel", "achieved": gram_bytes / gram_s / 1e9,
                     "peak": hbm_peak, "unit": "GB/s", "frac": gram_bytes / gram_s / 1e9 / hbm_peak, "traffic": gram_traffic,
                     "traffic_note": "dram__bytes_read+write of this kernel from the committed ncu --set full capture (n = 10000), scaled to this launch size",
                     "fp64_pipe_active_pct_ncu": (c5["fp64_pipe_active_pct"] if c5 else None),
                     "work_model": "48*n+216 algorithmic bytes per scene (SURVEY.md 8d)"},
        "roofline_fp64": {"bound": "fp64", "peak": fp64_peak, "unit": "TFLOP/s",
                          "achieved_executed": (flop_exec * scenes_per_launch / gram_s / 1e12 if flop_exec else None),
                          "frac_executed": (flop_exec * scenes_per_launch / gram_s / 1e12 / fp64_peak if flop_exec else None),
                          "algorithmic": 624.0 * n * scenes_per_launch / gram_s / 1e12,
                          "algorithmic_vs_peak": 624.0 * n * scenes_per_launch / gram_s / 1e12 / fp64_peak,
                          "work_model": "executed = DFMA*2 + DMUL + DADD thread instructions of the ncu capture; algorithmic = 624*n flop per scene "
                                        "(12-nnz rows, symmetric half; SURVEY.md B.3)"},
        "full_pipeline": {"metric": "LinearTFTPoseEstimation + ReprError solves/s at n=%d" % n, "value": B * steps / (ms * 1e-3),
                          "unit": "solves/s"},
        "kernels": {k: {"ms_total": v[0], "launches": int(v[1])} for k, v in prof.items()},
        "flagged_problems": int(torch.count_nonzero(d_st).item()),
        "gpu_launches": int(sum(v[1] for v in prof.values())),
    }
    del d_corresp, d_rec
    torch.cuda.empty_cache()
    return block


def run_large_n(args, local_rank):
    """65 536 scenes x n = 10 000 correspondences as its own bench line (`--workload large-n --n 10000 --trials 65536`);
    the default run carries the same measurement on 8 192 scenes in its `large_n` block."""
    import torch
    from tft_vs_fund_b200 import _lib
    torch.cuda.set_device(local_rank)
    h = _lib.Handle(local_rank)
    sampler = ClockSampler(local_rank)
    blk = large_n_measure(h, h.lib, local_rank, args.trials, args.n, args.steps, max(1, args.warmup))
    clocks = sampler.stop()
    line = {"metric": blk["metric"], "unit": blk["unit"], "value": blk["value"], "n_gpus": 1, "steps": blk["steps"],
            "warmup": max(1, args.warmup), "ms_per_step": blk["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "clocks": clocks}
    line.update({k: v for k, v in blk.items() if k not in line})
    emit(line)


_JSON_OUT = None


def claim_stdout():
    """stdout carries exactly ONE line, the JSON result.  Libraries print there too (NCCL writes its version line to
    stdout when the box exports NCCL_DEBUG=VERSION), so the real stdout is set aside for emit() and file descriptor 1
    is pointed at stderr for everything else (this process and the libraries it loads)."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--trials", type=int, default=1000000, help="trials per GPU and step (BASELINE config 3: 1M)")
    ap.add_argument("--n", type=int, default=20)
    ap.add_argument("--cpu-sample", type=int, default=0, help="trials in the CPU-baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--chunk", type=int, default=0, help="problems per launch (0 = the library's default)")
    ap.add_argument("--legs", default="all", choices=["all", "headline"],
                    help="headline = only the device-resident TFT step (what `value` times): used for the ncu launch list, so "
                         "that the list holds the kernels of the step and nothing else")
    ap.add_argument("--large-n-scenes", type=int, default=8192,
                    help="scenes of the config-5 block inside the default line (n = 10000; 0 = skip; N = 1 only)")
    ap.add_argument("--workload", default="sweep", choices=["sweep", "large-n"],
                    help="sweep = BASELINE config 3/4 (headline); large-n = config 5 (use with --n 10000 --trials 65536)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a fixed, seeded sample of the last step's outputs as DIR/<name>.npy "
                         "(sweep workload of the CUDA path, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "sweep"):
        ap.error("--dump-outputs applies to the sweep workload of the CUDA path (--impl b200 --workload sweep)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif args.workload == "large-n":
        if rank == 0:
            run_large_n(args, local_rank)
    else:
        run_gpu(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
