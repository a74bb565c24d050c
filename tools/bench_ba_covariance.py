"""Cost of tvf_ba_covariance_dev next to the bundle adjustment it follows, device-resident on one GPU.

Per configuration: trials -> tvf_pose_dev (method 1, linear TFT) -> the timed step, alternating three variants in
rounds until each has >= --seconds of device time:
    ba        tvf_bundle_adjust_dev alone;
    ba+cov    tvf_bundle_adjust_dev, then tvf_ba_covariance_dev at its result (cov_cam, sigma2, status);
    ba+cov+p  the same with cov_pts as well.
CUDA events bracket each call, so the covariance's own time is read in the same round as the adjustment's.  n <= 60
uses tvf_generate_sweep_dev trials; larger n tile --distinct host-generated sweep trials on the device (the solvers
have no cache, so repeated problems cost the same as distinct ones).

    python tools/bench_ba_covariance.py [--n 12,20,100] [--out profiles/r04_ba_covariance.json]
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
from bench_bundle_adjust import gpu_info  # noqa: E402


def run(n, B, distinct, seconds, device):
    import torch
    from tft_vs_fund_b200 import _lib, scene
    dev = torch.device("cuda", device)
    h = _lib.handle(device)
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    d_c = torch.empty((B, n, 6), dtype=torch.float64, device=dev)
    if n <= 60:
        d = scene.sweep_batch_device(B, n, device=device, out_ptr=d_c.data_ptr(), meta=False)
        source = "tvf_generate_sweep_dev, %d trials" % B
    else:
        d = scene.sweep_batch(distinct, n)
        src = torch.from_numpy(np.ascontiguousarray(d["Corresp"].transpose(0, 2, 1))).to(dev)
        d_c.copy_(src.repeat((B + distinct - 1) // distinct, 1, 1)[:B])
        source = "%d host-generated sweep trials tiled to %d" % (distinct, B)
    calm = torch.from_numpy(np.ascontiguousarray(d["CalM"].T)).to(dev)
    f64 = lambda *s: torch.empty(s, dtype=torch.float64, device=dev)
    i32 = lambda *s: torch.zeros(s, dtype=torch.int32, device=dev)
    s_r2, s_r3, s_x, s_rep, s_st = f64(B, 12), f64(B, 12), f64(B, 3 * n), f64(B), i32(B)
    out = _lib.PoseOut(p(s_r2), p(s_r3), p(s_x), None, p(s_rep), None, None, None, None, p(s_st))
    torch.cuda.synchronize(dev)
    h.call("tvf_pose_dev", 1, p(d_c), p(calm), 0, n, B, C.byref(out))
    h.call("tvf_synchronize")
    r2, r3, x, rep, it, st = f64(B, 12), f64(B, 12), f64(B, 3 * n), f64(B), i32(B), i32(B)
    cc, cp, s2, cst = f64(B, 144), f64(B, 9 * n), f64(B), i32(B)

    def adjust():
        h.call("tvf_bundle_adjust_dev", p(d_c), p(calm), 0, n, B, p(s_r2), p(s_r3), p(s_x), p(r2), p(r3), p(x), p(rep),
               p(it), p(st))

    def covariance(points):
        h.call("tvf_ba_covariance_dev", p(d_c), p(calm), 0, n, B, p(r2), p(r3), p(x), p(cc), p(cp) if points else None,
               p(s2), p(cst))

    stream = torch.cuda.Stream(device=dev)
    h.call("tvf_set_stream", C.c_void_p(stream.cuda_stream))
    variants = ("ba", "ba+cov", "ba+cov+p")
    ms = {v: [0.0, 0.0] for v in variants}              # [adjustment, covariance] device ms
    calls = {v: 0 for v in variants}
    try:
        adjust(); covariance(False); covariance(True); stream.synchronize()          # warm-up
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        while min(sum(ms[v]) for v in variants) < 1e3 * seconds:
            for v in variants:
                ev[0].record(stream); adjust(); ev[1].record(stream)
                if v != "ba":
                    covariance(v == "ba+cov+p")
                ev[2].record(stream); ev[2].synchronize()
                ms[v][0] += ev[0].elapsed_time(ev[1]); ms[v][1] += ev[1].elapsed_time(ev[2])
                calls[v] += 1
    finally:
        h.call("tvf_use_own_stream")
    stv = st.cpu().numpy(); cstv = cst.cpu().numpy()
    res = {"n": n, "batch": B, "inputs": source,
           "ba_status_nonzero_fraction": float(np.mean(stv != 0)),
           "cov_status": {str(k): int(np.sum(cstv == k)) for k in np.unique(cstv)},
           "sigma2_median": float(np.nanmedian(s2.cpu().numpy()))}
    for v in variants:
        ba_s = ms[v][0] / 1e3 / calls[v]; cov_s = ms[v][1] / 1e3 / calls[v]
        r = {"calls": calls[v], "ba_seconds_per_call": ba_s, "adjustments_per_s": B / ba_s}
        if v != "ba":
            r.update({"cov_seconds_per_call": cov_s, "covariances_per_s": B / cov_s,
                      "cov_share_of_ba_plus_cov": cov_s / (ba_s + cov_s)})
        res[v] = r
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--n", default="12,20,100")
    ap.add_argument("--batch", default="1000000,1000000,200000", help="problems per call, one per --n")
    ap.add_argument("--distinct", type=int, default=4096, help="host-generated trials tiled for n > 60")
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_ba_covariance.json"))
    a = ap.parse_args()
    res = {"what": "tvf_ba_covariance_dev after tvf_bundle_adjust_dev from tvf_pose_dev (method 1) starts; CUDA events "
                   "around each call, the three variants alternating", **gpu_info(a.device), "configs": []}
    for n, B in zip((int(v) for v in a.n.split(",")), (int(v) for v in a.batch.split(","))):
        r = run(n, B, a.distinct, a.seconds, a.device)
        print(json.dumps(r), flush=True)
        res["configs"].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "configs"}))


if __name__ == "__main__":
    main()
