"""The calibrated five-point minimal pose (tvf_five_point_pose, RANSAC method 9) on one GPU, against methods 1 and 7.

1. Solver: B minimal problems (5 matches of tests/distinct_k.py scenes at 1 px, tiled on the device) through
   tvf_five_point_pose_dev, and the same scenes' first 7 / 8 matches through tvf_pose_dev (methods 1 / 7).  CUDA events
   around whole _dev calls, median of --repeats after a warm-up; a separate torch.profiler pass gives the kernel time.
2. Plain RANSAC: methods 1, 7, 9 at their own 0.999-confidence H on ro.outlier_scenes (n = 100, f = 0.3 / 0.5, 2 px) and
   on the EPFL fountain triplet (1 024 hypotheses, 1 px): problems per second of the host call (it ends in a
   synchronise), recall, precision and median rotation error.
3. All 120 EPFL triplets, raw matches, one ragged call each: plain and refined method 9 against refined methods 1 and 7.

    python tools/bench_five_point.py [--out profiles/r09_five_point.json]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
from bench_bundle_adjust import gpu_info  # noqa: E402


def rot_err(R_t0, R2, R3):
    import oracle as o
    if not np.all(np.isfinite(R2)):
        return np.inf
    return (o.AngError(R_t0[0], R2)[0] + o.AngError(R_t0[1], R3)[0]) / 2


def stats(res, truths, R_t0s, seconds, B):
    rec = [np.sum(res[2][b] & t) / max(1, t.sum()) for b, t in enumerate(truths)]
    prec = [np.sum(res[2][b] & t) / max(1, res[2][b].sum()) for b, t in enumerate(truths)]
    rot = [rot_err(R_t0s[b], res[0][b], res[1][b]) for b in range(B)]
    return dict(seconds=seconds, problems_per_s=B / seconds, recall_median=float(np.median(rec)),
                recall_mean=float(np.mean(rec)), precision_median=float(np.median(prec)),
                median_rot_err_deg=float(np.median(rot)))


def timed(fn, repeats):
    fn()
    ts = []
    for _ in range(repeats):
        t0 = time.perf_counter(); r = fn(); ts.append(time.perf_counter() - t0)
    return r, float(np.median(ts))


def solver(B, repeats):
    import torch
    import distinct_k as dk
    from tft_vs_fund_b200 import _lib
    dev = torch.device("cuda", 0)
    h = _lib.handle(0)
    Cr, CalM, _, _ = dk.batch(8, 1.0, range(256))
    calm = torch.from_numpy(np.ascontiguousarray(CalM.transpose(0, 2, 1))).to(dev).repeat(B // 256, 1, 1).contiguous()
    out = {}
    for name, n in (("five_point", 5), ("method1_n7", 7), ("method7_n8", 8)):
        c = torch.from_numpy(np.ascontiguousarray(Cr[:, :, :n].transpose(0, 2, 1))).to(dev).repeat(B // 256, 1, 1).contiguous()
        r2 = torch.empty((B, 12), dtype=torch.float64, device=dev); r3 = torch.empty_like(r2)
        st = torch.empty(B, dtype=torch.int32, device=dev)
        p = lambda t: C.c_void_p(t.data_ptr())
        if n == 5:
            call = lambda: h.call("tvf_five_point_pose_dev", p(c), p(calm), 1, B, p(r2), p(r3), None, None, p(st))
        else:
            po = _lib.PoseOut(p(r2), p(r3), None, None, None, None, None, None, None, p(st))
            call = lambda: h.call("tvf_pose_dev", 1 if n == 7 else 7, p(c), p(calm), 1, n, B, C.byref(po))
        torch.cuda.synchronize(); call(); h.call("tvf_synchronize")
        ts = []
        for _ in range(repeats):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(); a.record(); call(); h.call("tvf_synchronize"); b.record(); b.synchronize()
            ts.append(a.elapsed_time(b) * 1e-3)
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call(); h.call("tvf_synchronize"); torch.cuda.synchronize()
        kt = sum(e.device_time_total for e in prof.key_averages() if "emcpy" not in e.key and "emset" not in e.key) * 1e-6
        out[name] = dict(B=B, seconds_median=float(np.median(ts)), solves_per_s=B / float(np.median(ts)),
                         kernel_seconds=kt, flagged=int((st != 0).sum().item()))
        print(name, out[name], flush=True)
    return out


def plain(repeats):
    import ransac_oracle as ro
    import tft_vs_fund_b200 as tvf
    from test_gpu_ransac import epfl_triplets
    out = {}
    for f in (0.3, 0.5):
        Cr, CalM, R_t0, outl = ro.outlier_scenes(f, 256, 91)
        for m in (1, 7, 9):
            H = ro.hypotheses_for(f, {1: 7, 7: 8, 9: 5}[m])
            res, sec = timed(lambda: tvf.ransac_pose(Cr, CalM, method=m, hypotheses=H, threshold=2.0, seed=1), repeats)
            out["synthetic_f%.1f_m%d" % (f, m)] = dict(H=H, **stats(res, list(~outl), [R_t0] * 256, sec, 256))
            print("f", f, "m", m, out["synthetic_f%.1f_m%d" % (f, m)], flush=True)
    Cm, CalMm, R_t0m, truth = epfl_triplets(1)[0]
    for m in (1, 7, 9):
        res, sec = timed(lambda: tvf.ransac_pose(Cm[None], CalMm, method=m, hypotheses=1024, threshold=1.0, seed=1), repeats)
        out["epfl_fountain_m%d" % m] = dict(H=1024, n=int(Cm.shape[1]), **stats(res, [truth], [R_t0m], sec, 1))
        print("fountain m", m, out["epfl_fountain_m%d" % m], flush=True)
    return out


def headline(repeats):
    import tft_vs_fund_b200 as tvf
    from test_gpu_ransac import epfl_triplets
    trips = epfl_triplets()
    Cs, CalM = [t[0] for t in trips], np.stack([t[1] for t in trips])
    seeds = np.arange(1, len(trips) + 1, dtype=np.uint64)
    out = {}
    for label, m, refine in (("plain_m9", 9, False), ("refined_m9", 9, True), ("refined_m1", 1, True),
                             ("refined_m7", 7, True), ("plain_m1", 1, False), ("plain_m7", 7, False)):
        res, sec = timed(lambda: tvf.ransac_pose(Cs, CalM, method=m, hypotheses=1024, threshold=1.0, seed=seeds,
                                                 refine=refine), repeats)
        out[label] = stats(res, [t[3] for t in trips], [t[2] for t in trips], sec, len(trips))
        out[label]["ms"] = sec * 1e3
        print(label, out[label], flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_five_point.json"))
    ap.add_argument("--B", type=int, default=1 << 20)
    ap.add_argument("--repeats", type=int, default=5)
    a = ap.parse_args()
    res = dict(gpu=gpu_info(0), solver=solver(a.B, a.repeats), plain=plain(a.repeats), epfl_120=headline(a.repeats))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
