"""Throughput of tvf_bundle_adjust_dev, device-resident: trials -> tvf_pose_dev (method 1, linear TFT) ->
tvf_bundle_adjust_dev, all on one GPU, timed with CUDA events over >= --seconds of adjustment after a warm-up call.

n = 20: 1 M trials from tvf_generate_sweep_dev (the sweep of experiments.m).  The device generator stops at n = 60, so
larger n use --distinct host-generated sweep trials (scene.sweep_batch) tiled on the device up to the batch size; the
batch is sized to keep n * B at 2e7 points.  Repeated problems cost the same as distinct ones (the solver has no cache).

    python tools/bench_bundle_adjust.py [--n 20,100,1000] [--out profiles/r03_bench_bundle_adjust.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info(device):
    import torch
    info = {"gpu": torch.cuda.get_device_name(device)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = "unavailable: %s" % e
    return info


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
        reps = (B + distinct - 1) // distinct
        d_c.copy_(src.repeat(reps, 1, 1)[:B])
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

    def adjust():
        h.call("tvf_bundle_adjust_dev", p(d_c), p(calm), 0, n, B, p(s_r2), p(s_r3), p(s_x), p(r2), p(r3), p(x), p(rep),
               p(it), p(st))

    stream = torch.cuda.Stream(device=dev)                                # the _dev calls run on this stream
    h.call("tvf_set_stream", C.c_void_p(stream.cuda_stream))
    try:
        adjust(); stream.synchronize()                                    # warm-up (module load, arena allocation)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        calls, ms, wall = 0, 0.0, time.perf_counter()
        while ms < 1e3 * seconds:
            e0.record(stream); adjust(); e1.record(stream); e1.synchronize()
            ms += e0.elapsed_time(e1)
            calls += 1
        wall = time.perf_counter() - wall
    finally:
        h.call("tvf_use_own_stream")
    itv = it.cpu().numpy(); stv = st.cpu().numpy()
    start_rep = s_rep.cpu().numpy(); end_rep = rep.cpu().numpy()
    ok = (stv & _lib.ST_NONFINITE) == 0
    return {
        "n": n, "batch": B, "inputs": source, "calls_timed": calls, "seconds_timed_events": ms / 1e3, "seconds_wall": wall,
        "adjustments_per_s": B * calls / (ms / 1e3),
        "iter_mean": float(itv.mean()), "iter_max": int(itv.max()),
        "flagged_fraction": float(np.mean(stv != 0)),
        "nonfinite_fraction": float(np.mean(~ok)),
        "noconv_fraction": float(np.mean((stv & _lib.ST_BA_NOCONV) != 0)),
        "repr_err_start_mean_px": float(np.mean(start_rep[ok])), "repr_err_end_mean_px": float(np.mean(end_rep[ok])),
        "repr_err_never_rose": bool(np.all(end_rep[ok] <= start_rep[ok] * (1 + 1e-12))),
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--n", default="20,100,1000")
    ap.add_argument("--points", type=float, default=2e7, help="n * B per configuration")
    ap.add_argument("--distinct", type=int, default=4096, help="host-generated trials tiled for n > 60")
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_bench_bundle_adjust.json"))
    a = ap.parse_args()
    res = {"what": "tvf_bundle_adjust_dev throughput from tvf_pose_dev (method 1) starts; CUDA events around each call",
           **gpu_info(a.device), "configs": []}
    for n in (int(v) for v in a.n.split(",")):
        B = int(a.points // n)
        r = run(n, B, a.distinct, a.seconds, a.device)
        print(json.dumps(r), flush=True)
        res["configs"].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "configs"}))


if __name__ == "__main__":
    main()
