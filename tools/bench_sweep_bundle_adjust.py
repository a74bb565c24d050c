"""Cost of the after-adjustment columns: tvf_sweep_run_levels against tvf_sweep_run_levels_ba on the same trials, timed
alternately with a host clock around each call (both synchronise before they return), after a warm-up of each.

Two workloads:
  * the noise sweep of experiments.m (13 levels, n = 20) over --trials trials;
  * experiments.m's four options at its default N = 12 ('points' sweeps N itself), with n_sim scaled from the warm-up so
    that a call without adjustment lasts about --seconds.
A window that would be shorter than --seconds repeats the call.  Mean iterations come from the table (column 10 over
column 8); the fraction of counted trials ending with TVF_ST_BA_NOCONV, which the table does not carry, comes from a
separate tvf_pose_dev + tvf_bundle_adjust_dev run on one chunk per workload.  Then tools/bench_bundle_adjust.py --n 12,20
gives the stand-alone adjustment rate.  The device name, power limit and max SM clock are queried, nothing is set.

    python tools/bench_sweep_bundle_adjust.py [--trials 1048576] [--out profiles/r03_sweep_bundle_adjust.json]
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_bundle_adjust import gpu_info  # noqa: E402


def _call(h, name, method, B, levels, L):
    from tft_vs_fund_b200 import _lib, scene
    t = np.zeros((L, 11 if name.endswith("_ba") else 5))
    h.call(name, int(method), 0, int(B), levels, L, 36 * scene.PIX, 24 * scene.PIX, t.ctypes.data_as(_lib.c_double_p))
    return t


def _timed(h, name, method, B, levels, L, reps):
    t0 = time.perf_counter()
    for _ in range(reps):
        table = _call(h, name, method, B, levels, L)
    return time.perf_counter() - t0, table


def noconv_chunk(params, method, per_level, device):
    """One chunk of per_level trials per level through tvf_pose_dev and tvf_bundle_adjust_dev: (counted trials,
    those ending with TVF_ST_BA_NOCONV, mean iter over the counted)."""
    import torch
    from tft_vs_fund_b200 import _lib, scene
    h = _lib.handle(device)
    dev = torch.device("cuda", device)
    p = lambda t: C.c_void_p(t.data_ptr())
    counted = noconv = iters = 0
    for q in params:
        n = q["N"]
        if (method > 6 and n < 8) or n < 7:
            continue
        d_c = torch.empty((per_level, n, 6), dtype=torch.float64, device=dev)
        d = scene.sweep_batch_device(per_level, n, noise_levels=[q["noise"]], focalL=q["f"], angle=q["angle"], device=device,
                                     out_ptr=d_c.data_ptr(), meta=False)
        calm = torch.from_numpy(np.ascontiguousarray(d["CalM"].T)).to(dev)
        f64 = lambda *s: torch.empty(s, dtype=torch.float64, device=dev)
        i32 = lambda *s: torch.zeros(s, dtype=torch.int32, device=dev)
        s_r2, s_r3, s_x, s_st = f64(per_level, 12), f64(per_level, 12), f64(per_level, 3 * n), i32(per_level)
        out = _lib.PoseOut(p(s_r2), p(s_r3), p(s_x), None, None, None, None, None, None, p(s_st))
        torch.cuda.synchronize(dev)
        h.call("tvf_pose_dev", int(method), p(d_c), p(calm), 0, n, per_level, C.byref(out))
        r2, r3, x, rep, it, st = f64(per_level, 12), f64(per_level, 12), f64(per_level, 3 * n), f64(per_level), i32(per_level), i32(per_level)
        h.call("tvf_bundle_adjust_dev", p(d_c), p(calm), 0, n, per_level, p(s_r2), p(s_r3), p(s_x), p(r2), p(r3), p(x), p(rep),
               p(it), p(st))
        h.call("tvf_synchronize")
        pose_st, ba_st, itv = s_st.cpu().numpy(), st.cpu().numpy(), it.cpu().numpy()
        ok = ((pose_st & (_lib.ST_NO_POSE_2 | _lib.ST_NO_POSE_3 | _lib.ST_NONFINITE)) == 0) & ((ba_st & _lib.ST_NONFINITE) == 0)
        counted += int(ok.sum()); noconv += int(((ba_st & _lib.ST_BA_NOCONV) != 0)[ok].sum()); iters += int(itv[ok].sum())
    return counted, noconv, (iters / counted if counted else float("nan"))


def measure(label, params, method, B, windows, seconds, device, noconv_per_level):
    from tft_vs_fund_b200 import _lib, experiments
    h = _lib.handle(device)
    levels, L = experiments._sweep_levels(params), len(params)
    names = ("tvf_sweep_run_levels", "tvf_sweep_run_levels_ba")
    reps = {}
    for name in names:                                     # warm-up: module load, arenas, scratch
        dt, _ = _timed(h, name, method, B, levels, L, 1)
        reps[name] = max(1, math.ceil(seconds / dt))
    times = {name: [] for name in names}
    tables = {}
    for _ in range(windows):
        for name in names:
            dt, tables[name] = _timed(h, name, method, B, levels, L, reps[name])
            times[name].append(dt / reps[name])
    t_plain, t_ba = float(np.median(times[names[0]])), float(np.median(times[names[1]]))
    tb = tables[names[1]]
    fin = np.isfinite(tb[:, 0])
    counted = float(tb[fin, 8].sum())
    c, nc, it_chunk = noconv_chunk(params, method, noconv_per_level, device)
    r = {
        "workload": label, "method": int(method), "levels": L, "trials": int(B),
        "windows": windows, "calls_per_window": reps, "seconds_per_call": times,
        "trials_per_s_without_ba": B / t_plain, "trials_per_s_with_ba": B / t_ba,
        "ba_share_of_step": (t_ba - t_plain) / t_ba,
        "method_columns_equal_plain_table": bool(np.array_equal(tb[:, :5], tables[names[0]], equal_nan=True)),
        "ba_iter_mean": float(tb[fin, 10].sum() / counted) if counted else float("nan"),
        "skipped_after_ba": int(tb[fin, 9].sum()),
        "noconv_chunk": {"trials_per_level": noconv_per_level, "counted": c, "ba_noconv": nc,
                         "ba_noconv_fraction": nc / c if c else float("nan"), "iter_mean": it_chunk},
    }
    print(json.dumps(r), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--trials", type=int, default=1 << 20, help="trials of the n = 20 noise sweep")
    ap.add_argument("--methods", default="1,7,8", help="methods timed on the noise sweep")
    ap.add_argument("--option-methods", default="1", help="methods timed on the four options at N = 12")
    ap.add_argument("--seconds", type=float, default=1.0, help="least length of a timed window")
    ap.add_argument("--windows", type=int, default=3, help="timed windows per entry point")
    ap.add_argument("--noconv-trials", type=int, default=65536, help="trials per level of the NOCONV chunk (split over levels)")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_sweep_bundle_adjust.json"))
    ap.add_argument("--ba-out", default=None, help="--out of tools/bench_bundle_adjust.py (default: a temporary file)")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU and has no CPU fallback")
    from tft_vs_fund_b200 import experiments
    res = {"what": "tvf_sweep_run_levels vs tvf_sweep_run_levels_ba on the same trials; host clock around calls that "
                   "synchronise; median of the windows", **gpu_info(a.device), "configs": []}
    noise = [dict(N=20, noise=float(v), f=50, angle=0) for v in experiments.NOISE_LEVELS]
    for m in (int(v) for v in a.methods.split(",")):
        res["configs"].append(measure("noise sweep, n = 20", noise, m, a.trials, a.windows, a.seconds, a.device,
                                      a.noconv_trials // len(noise)))
    for option in ("noise", "focal", "points", "angle"):
        _, params = experiments.experiment_levels(option)
        L = len(params)
        for m in (int(v) for v in a.option_methods.split(",")):
            from tft_vs_fund_b200 import _lib
            h = _lib.handle(a.device)
            levels = experiments._sweep_levels(params)
            n_sim = 8192
            _call(h, "tvf_sweep_run_levels", m, L * n_sim, levels, L)
            dt, _ = _timed(h, "tvf_sweep_run_levels", m, L * n_sim, levels, L, 1)
            n_sim = int(math.ceil(n_sim * 1.2 * a.seconds / dt))
            r = measure("experiments.m option '%s', N = 12, n_sim = %d" % (option, n_sim), params, m, L * n_sim, a.windows,
                        a.seconds, a.device, max(1, a.noconv_trials // L))
            r["n_sim"] = n_sim
            res["configs"].append(r)
    import tempfile
    ba_out = a.ba_out or os.path.join(tempfile.mkdtemp(), "bench_bundle_adjust.json")
    subprocess.check_call([sys.executable, os.path.join(ROOT, "tools", "bench_bundle_adjust.py"), "--n", "12,20",
                           "--device", str(a.device), "--out", ba_out])
    with open(ba_out) as f:
        res["standalone_bundle_adjust"] = json.load(f)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k not in ("configs", "standalone_bundle_adjust")}))


if __name__ == "__main__":
    main()
