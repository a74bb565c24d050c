"""Throughput of tvf_ransac_pose_refined_dev on one GPU, device-resident, where its time goes, and the packed small-n
adjustment (bundle_adjust_small_kernel) against bundle_adjust_kernel on the same problems.

Configurations as tools/bench_ransac.py: synthetic sweep scenes (n = 100, noise 1 px) with a share f of their columns
replaced by uniform image pixels, H = ceil(log(1e-3) / log(1 - (1 - f)^s)), threshold 2 px; and the EPFL fountain triplet
(n = 1400 raw matches, H = 1024, 1 px).  8 LO rounds.  --distinct host-generated scenes are tiled on the device.  CUDA
events time whole calls; a separate torch.profiler pass splits one call's kernels into hypotheses (sample and pose
kernels), adjustment (bundle_adjust_small_kernel), consensus (the hypotheses' scoring) and LO (everything after the
selection: the winner's consensus, the LO rounds and the result).

Packed against one-warp adjustment: the minimal problems of the n = 100, f = 0.3 configuration (the samples of the
refined call's hypotheses with their linear poses, rebuilt on the host) go through tvf_bundle_adjust_dev
(bundle_adjust_kernel); the refined call on the same problems runs them through bundle_adjust_small_kernel.  Both
kernels are timed by torch.profiler, --repeats passes each, alternating; reported as adjustments per second (median).

    python tools/bench_ransac_refined.py [--out profiles/r06_ransac_refined.json]
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
from bench_bundle_adjust import gpu_info  # noqa: E402

LO_ROUNDS = 8


def kernel_events(fn, stream):
    """(name, microseconds) of the CUDA kernels of one fn() in start order."""
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn(); stream.synchronize()
    ev = sorted(((e.name, e.time_range.start, e.time_range.elapsed_us()) for e in prof.events()
                 if e.device_type.name == "CUDA" and "emcpy" not in e.name and "emset" not in e.name), key=lambda x: x[1])
    return [(nme, dur) for nme, _, dur in ev]


def split_phases(events):
    """seconds of hypotheses, adjustment, consensus and LO (from each chunk's selection to its end)."""
    phase, t = "hyp", {"hyp": 0.0, "adjust": 0.0, "consensus": 0.0, "lo": 0.0}
    for name, dur in events:
        if "ransac_sample_kernel" in name:                 # a chunk starts
            phase = "hyp"
        if "ransac_select_kernel" in name:
            phase = "lo"
        if phase == "lo":
            t["lo"] += dur
        elif "bundle_adjust_small_kernel" in name:
            t["adjust"] += dur
        elif "ransac_consensus_kernel" in name or "ransac_flag_kernel" in name:
            t["consensus"] += dur
        else:
            t["hyp"] += dur
    return {k: v * 1e-6 for k, v in t.items()}


class Refined:
    """tvf_ransac_pose_refined_dev on B problems tiled from Cr (distinct, 6 x n each) on the device."""

    def __init__(self, Cr, CalM, method, H, th, B, device):
        import torch
        from tft_vs_fund_b200 import _lib
        self.dev = torch.device("cuda", device)
        self.h = _lib.handle(device)
        self.method, self.H, self.th, self.B, self.n = method, H, th, B, Cr.shape[2]
        src = torch.from_numpy(np.ascontiguousarray(Cr.transpose(0, 2, 1))).to(self.dev)
        self.c = src.repeat((B + Cr.shape[0] - 1) // Cr.shape[0], 1, 1)[:B].contiguous()
        self.calm = torch.from_numpy(np.ascontiguousarray(CalM.T)).to(self.dev)
        self.seeds = torch.arange(B, dtype=torch.int64, device=self.dev)
        s = 7 if method == 1 else 8
        self.r2 = torch.empty((B, 12), dtype=torch.float64, device=self.dev); self.r3 = torch.empty_like(self.r2)
        self.mk = torch.empty((B, self.n), dtype=torch.uint8, device=self.dev)
        self.cnt, self.smp, self.lo, self.st = (torch.empty(x, dtype=torch.int32, device=self.dev)
                                                for x in ((B,), (B, s), (B,), (B,)))

    def __call__(self):
        p = lambda t: C.c_void_p(t.data_ptr())
        self.h.call("tvf_ransac_pose_refined_dev", self.method, p(self.c), p(self.calm), 0, self.n, self.B, self.H,
                    self.th, p(self.seeds), LO_ROUNDS, p(self.r2), p(self.r3), p(self.mk), p(self.cnt), p(self.smp),
                    p(self.lo), p(self.st))


def with_stream(h, stream, fn):
    h.call("tvf_set_stream", C.c_void_p(stream.cuda_stream))
    try:
        return fn()
    finally:
        h.call("tvf_use_own_stream")


def run(label, Cr, CalM, method, H, th, B, seconds, device):
    import torch
    r = Refined(Cr, CalM, method, H, th, B, device)
    stream = torch.cuda.Stream(device=r.dev)

    def measure():
        r(); stream.synchronize()                                          # warm-up
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ms, calls = 0.0, 0
        while ms < 1e3 * seconds:
            a.record(stream); r(); b.record(stream); b.synchronize()
            ms += a.elapsed_time(b); calls += 1
        return ms, calls, split_phases(kernel_events(r, stream))
    ms, calls, phases = with_stream(r.h, stream, measure)
    per_call = ms / 1e3 / calls
    tot = sum(phases.values())
    lo = r.lo.cpu().numpy(); cv = r.cnt.cpu().numpy(); st = r.st.cpu().numpy()
    return {"config": label, "method": method, "n": r.n, "H": H, "threshold": th, "lo_rounds": LO_ROUNDS, "batch": B,
            "calls": calls, "seconds_per_call": per_call, "problems_per_s": B / per_call,
            "share_hypotheses": phases["hyp"] / tot, "share_adjustment": phases["adjust"] / tot,
            "share_consensus": phases["consensus"] / tot, "share_lo": phases["lo"] / tot, "profiled_kernel_seconds": tot,
            "adjustments_per_s_in_call": B * H / phases["adjust"], "failed_fraction": float(np.mean(st != 0)),
            "median_n_inliers": float(np.median(cv)), "mean_lo_done": float(np.mean(lo))}


def packed_vs_warp(Cr, CalM, method, H, B, repeats, device):
    """adjustments/s of bundle_adjust_small_kernel (inside the refined call) and bundle_adjust_kernel
    (tvf_bundle_adjust_dev) on the same B H minimal problems."""
    import torch
    import ransac_oracle as ro
    from tft_vs_fund_b200 import api
    s = 7 if method == 1 else 8
    n = Cr.shape[2]
    Ct = np.concatenate([Cr] * ((B + Cr.shape[0] - 1) // Cr.shape[0]))[:B]
    S = np.concatenate([Ct[b][:, ro.sample(b, np.arange(H), n, s)].transpose(1, 0, 2) for b in range(B)])   # (B H, 6, s)
    pose = (api.LinearTFTPoseEstimation if method == 1 else api.LinearFPoseEstimation)(S, CalM, device=device)
    r = Refined(Cr, CalM, method, H, 2.0, B, device)
    Q = B * H
    dev = r.dev
    d_S = torch.from_numpy(np.ascontiguousarray(S.transpose(0, 2, 1))).to(dev)
    d_r2 = torch.from_numpy(api._cm(pose[0], 2)[0].copy()).to(dev)
    d_r3 = torch.from_numpy(api._cm(pose[1], 2)[0].copy()).to(dev)
    o2, o3 = torch.empty((Q, 12), dtype=torch.float64, device=dev), torch.empty((Q, 12), dtype=torch.float64, device=dev)
    X = torch.empty((Q, 3 * s), dtype=torch.float64, device=dev)
    st = torch.empty(Q, dtype=torch.int32, device=dev)
    p = lambda t: C.c_void_p(t.data_ptr())

    def warp():
        r.h.call("tvf_bundle_adjust_dev", p(d_S), p(r.calm), 0, s, Q, p(d_r2), p(d_r3), None, p(o2), p(o3), p(X), None,
                 None, p(st))
    stream = torch.cuda.Stream(device=dev)

    def measure():
        warp(); r(); stream.synchronize()
        packed, one = [], []
        for _ in range(repeats):
            packed.append(sum(d for nme, d in kernel_events(r, stream) if "bundle_adjust_small_kernel" in nme))
            one.append(sum(d for nme, d in kernel_events(warp, stream) if "bundle_adjust_kernel" in nme))
        return packed, one
    packed, one = with_stream(r.h, stream, measure)
    return {"method": method, "n": s, "adjustments": Q, "repeats": repeats,
            "packed_adjustments_per_s": Q / (np.median(packed) * 1e-6),
            "warp_adjustments_per_s": Q / (np.median(one) * 1e-6),
            "packed_kernel_seconds": [x * 1e-6 for x in packed], "warp_kernel_seconds": [x * 1e-6 for x in one],
            "speedup": float(np.median(one) / np.median(packed)),
            "noconv_fraction": float(np.mean(st.cpu().numpy() & 32 != 0))}


def main():
    import ransac_oracle as ro
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--batch", type=int, default=4000, help="problems per call at 30 %% outliers (a tenth at 50 %%)")
    ap.add_argument("--epfl-batch", type=int, default=32)
    ap.add_argument("--compare-batch", type=int, default=2000)
    ap.add_argument("--distinct", type=int, default=256)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--seconds", type=float, default=2.0)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_ransac_refined.json"))
    a = ap.parse_args()
    info = gpu_info(a.device)
    res = {"what": "tvf_ransac_pose_refined_dev, CUDA events around whole calls; phase shares and the two adjustment "
                   "kernels from torch.profiler passes", **info, "packed_vs_warp": [], "configs": []}
    Cr, CalM, _, _ = ro.outlier_scenes(0.3, a.distinct, 7)
    for method in (1, 7):
        r = packed_vs_warp(Cr, CalM, method, ro.hypotheses_for(0.3, 7 if method == 1 else 8), a.compare_batch,
                           a.repeats, a.device)
        print(json.dumps(r), flush=True)
        res["packed_vs_warp"].append(r)
    for f, B in ((0.3, a.batch), (0.5, max(1, a.batch // 10))):
        Cr, CalM, _, _ = ro.outlier_scenes(f, a.distinct, 7)
        for method in (1, 7):
            H = ro.hypotheses_for(f, 7 if method == 1 else 8)
            r = run("synthetic n=100 f=%.1f" % f, Cr, CalM, method, H, 2.0, B, a.seconds, a.device)
            print(json.dumps(r), flush=True)
            res["configs"].append(r)
    g = np.load(os.path.join(ROOT, "tests", "golden", "epfl_full_triplet.npz"))
    for method in (1, 7):
        r = run("EPFL fountain triplet n=1400", g["Corresp"][None], g["CalM"], method, 1024, 1.0, a.epfl_batch,
                a.seconds, a.device)
        print(json.dumps(r), flush=True)
        res["configs"].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "configs"}))


if __name__ == "__main__":
    main()
