"""Throughput of tvf_ransac_pose_dev on one GPU, device-resident, and where its time goes.

Configurations: synthetic sweep scenes (n = 100, noise 1 px) with a share f of their columns replaced by uniform image
pixels and H = ceil(log(1e-3) / log(1 - (1 - f)^s)), and the EPFL fountain triplet (n = 1400 raw matches, H = 1024).
Problems are --distinct host-generated scenes tiled on the device (the estimator has no cache, so repeats cost the
same as distinct problems).  CUDA events time whole calls; a separate torch.profiler pass splits one call's kernels into
sample + hypotheses (each chunk's sample kernel and pose kernels), consensus (ransac_consensus_kernel) and refit (the
rest of each chunk after its selection).
The consensus kernel's FP64 rate uses OPS_PER_PAIR against tvf_fp64_peak_tflops.

    python tools/bench_ransac.py [--out profiles/r05_ransac.json]
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

# FP64 operations (an FMA counts 2) of one (hypothesis, match) pair of ransac_inlier, counted from csrc/tvf_ransac.cuh:
# the cameras K2 [R2|t2], K3 [R3|t3] (2 x 12 entries x 3 FMA = 144), the DLT rows (3 views x 2 rows x 4 FMA = 48), the
# Householder QR of the 6 x 4 system (~220) and inverse iteration (~55 per step, 4 steps typical = 220), the
# dehomogenisation (3) and three projections with their divisions and residual tests (3 x (24 + 2 + 6) = 96).
OPS_PER_PAIR = 144 + 48 + 220 + 220 + 3 + 96


def split_phases(events):
    """kernel events of one call in start order -> seconds of sample + hypotheses (from each chunk's sample kernel to its
    selection), consensus and refit (the rest of the chunk)."""
    phase, t = "hyp", {"hyp": 0.0, "consensus": 0.0, "refit": 0.0}
    for name, dur in events:
        if "ransac_sample_kernel" in name:                 # a chunk starts
            phase = "hyp"
        if "ransac_consensus_kernel" in name:
            t["consensus"] += dur
        elif "ransac_select_kernel" in name:
            phase = "refit"
            t["refit"] += dur
        else:
            t[phase] += dur
    return {k: v * 1e-6 for k, v in t.items()}


def run(label, Cr, CalM, method, H, B, seconds, device, peak):
    import torch
    from tft_vs_fund_b200 import _lib
    dev = torch.device("cuda", device)
    h = _lib.handle(device)
    p = lambda t: C.c_void_p(t.data_ptr())
    n = Cr.shape[2]
    src = torch.from_numpy(np.ascontiguousarray(Cr.transpose(0, 2, 1))).to(dev)
    d_c = src.repeat((B + Cr.shape[0] - 1) // Cr.shape[0], 1, 1)[:B].contiguous()
    calm = torch.from_numpy(np.ascontiguousarray(CalM.T)).to(dev)
    seeds = torch.arange(B, dtype=torch.int64, device=dev)
    s = 7 if method == 1 else 8
    r2 = torch.empty((B, 12), dtype=torch.float64, device=dev); r3 = torch.empty_like(r2)
    mk = torch.empty((B, n), dtype=torch.uint8, device=dev)
    cnt, smp, st = (torch.empty(x, dtype=torch.int32, device=dev) for x in ((B,), (B, s), (B,)))

    def call():
        h.call("tvf_ransac_pose_dev", method, p(d_c), p(calm), 0, n, B, H, 3.0 if label.startswith("synthetic") else 1.0,
               p(seeds), p(r2), p(r3), p(mk), p(cnt), p(smp), p(st))

    stream = torch.cuda.Stream(device=dev)
    h.call("tvf_set_stream", C.c_void_p(stream.cuda_stream))
    try:
        call(); stream.synchronize()                                       # warm-up
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ms, calls = 0.0, 0
        while ms < 1e3 * seconds:
            a.record(stream); call(); b.record(stream); b.synchronize()
            ms += a.elapsed_time(b); calls += 1
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call(); stream.synchronize()
        ev = sorted(((e.name, e.time_range.start, e.time_range.elapsed_us()) for e in prof.events()
                     if e.device_type.name == "CUDA" and "emcpy" not in e.name and "emset" not in e.name), key=lambda x: x[1])
        phases = split_phases([(nme, dur) for nme, _, dur in ev])
    finally:
        h.call("tvf_use_own_stream")
    per_call = ms / 1e3 / calls
    tot = sum(phases.values())
    pairs = B * H * n
    stv = st.cpu().numpy(); cv = cnt.cpu().numpy()
    return {"config": label, "method": method, "n": n, "H": H, "batch": B, "calls": calls,
            "seconds_per_call": per_call, "problems_per_s": B / per_call,
            "share_sample_hypotheses": phases["hyp"] / tot, "share_consensus": phases["consensus"] / tot,
            "share_refit": phases["refit"] / tot, "profiled_kernel_seconds": tot,
            "consensus_pairs_per_s": pairs / phases["consensus"],
            "consensus_fp64_tflops": pairs * OPS_PER_PAIR / phases["consensus"] / 1e12,
            "consensus_fraction_of_fp64_peak": pairs * OPS_PER_PAIR / phases["consensus"] / 1e12 / peak,
            "failed_fraction": float(np.mean(stv != 0)), "median_n_inliers": float(np.median(cv))}


def main():
    import ransac_oracle as ro
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--batch", type=int, default=100000, help="problems per call of the synthetic configurations")
    ap.add_argument("--epfl-batch", type=int, default=128)
    ap.add_argument("--distinct", type=int, default=512)
    ap.add_argument("--seconds", type=float, default=2.0)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_ransac.json"))
    a = ap.parse_args()
    from tft_vs_fund_b200 import _lib
    info = gpu_info(a.device)
    peak = _lib.handle(a.device).lib.tvf_fp64_peak_tflops(_lib.handle(a.device)._h)
    res = {"what": "tvf_ransac_pose_dev, CUDA events around whole calls; phase shares from one torch.profiler pass",
           **info, "fp64_peak_tflops_measured": peak, "ops_per_consensus_pair": OPS_PER_PAIR, "configs": []}
    for f in (0.3, 0.5):
        Cr, CalM, _, _ = ro.outlier_scenes(f, a.distinct, 7)
        for method in (1, 7):
            H = ro.hypotheses_for(f, 7 if method == 1 else 8)
            r = run("synthetic n=100 f=%.1f" % f, Cr, CalM, method, H, a.batch, a.seconds, a.device, peak)
            print(json.dumps(r), flush=True)
            res["configs"].append(r)
    g = np.load(os.path.join(ROOT, "tests", "golden", "epfl_full_triplet.npz"))
    for method in (1, 7):
        r = run("EPFL fountain triplet n=1400", g["Corresp"][None], g["CalM"], method, 1024, a.epfl_batch, a.seconds,
                a.device, peak)
        print(json.dumps(r), flush=True)
        res["configs"].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "configs"}))


if __name__ == "__main__":
    main()
