"""Robust-loss bundle adjustment on the GPU (tvf_bundle_adjust_robust), timed with CUDA events around whole _dev calls
(inputs already on the device), the median of --reps calls after one warm-up, variants alternated:

  1. cost of robustness: adjustments/s of each loss against the plain adjustment at n = 20 and n = 100 (B = 65 536,
     sweep scenes at 1 px from the true poses, points triangulated), clean and with 20 % of the matches replaced by
     uniform pixels;
  2. the 120 EPFL triplets with all raw matches, three pipelines, wall time and median rotation / t-direction error
     against epfl.relative_poses:
       a. plain ragged RANSAC (method 1, 1 024 hypotheses, 1 px), then one ragged robust adjustment (Cauchy, c = 2 px)
          over all raw matches from its pose;
       b. the same RANSAC, then the plain ragged adjustment on its consensus (the gather of the consensus columns on
          the host is not timed);
       c. refined RANSAC (8 LO rounds);
     and the recall / precision against epfl.inlier_filter (1 px) of the matches whose Cauchy weight is >= 1/2 (s_i <= c^2).

    python tools/bench_ba_robust.py [--reps 5] [--out profiles/r08_ba_robust.json]
"""
import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

LOSSES = {"huber": 1, "soft_l1": 2, "cauchy": 3}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def ptxas_robust():
    """registers, stack and spills of the *robust* kernels and bundle_adjust_kernel from the build log"""
    path = os.path.join(ROOT, "tft_vs_fund_b200", "build.log")
    if not os.path.exists(path):
        return None
    log = open(path).read().splitlines()
    out = {}
    for i, line in enumerate(log):
        m = re.search(r"Compiling entry function '\S*?\d+(bundle_adjust\w*?_kernel)\w*'", line)
        if not m or m.group(1) in out:
            continue
        block = "\n".join(log[i + 1:i + 4])
        sp = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", block)
        rg = re.search(r"Used (\d+) registers", block)
        out[m.group(1)] = dict(registers=int(rg.group(1)), stack_bytes=int(sp.group(1)), spill_stores=int(sp.group(2)),
                               spill_loads=int(sp.group(3)))
    return out


def timed(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--B", type=int, default=65536)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_ba_robust.json"))
    args = ap.parse_args()
    import torch
    import oracle as o
    from tft_vs_fund_b200 import _lib, api, epfl, scene
    h = _lib.handle(0)
    dev = torch.device("cuda", 0)
    h.call("tvf_set_stream", C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))    # the events' stream
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    f64 = lambda *s: torch.empty(s, dtype=torch.float64, device=dev)
    i32 = lambda *s: torch.zeros(s, dtype=torch.int32, device=dev)
    out = dict(gpu=gpu_info(), reps=args.reps, ptxas=ptxas_robust(),
               note="CUDA events around whole _dev calls; median of reps, variants alternated")

    # ---- 1. cost of robustness ---------------------------------------------------------------------------------------
    B = args.B
    rows = []
    for n in (20, 100):
        for frac in (0.0, 0.2):
            sb = scene.sweep_batch(B, n=n, noise_levels=[1.0])
            Cr = sb["Corresp"].copy()
            if frac:
                rs = np.random.RandomState(n)
                k = int(round(frac * n))
                cols = np.argsort(rs.rand(B, n), axis=1)[:, :k]
                bi = np.repeat(np.arange(B), k)
                for v in range(3):
                    Cr[bi, 2 * v, cols.ravel()] = rs.uniform(0, 36 * scene.PIX, B * k)
                    Cr[bi, 2 * v + 1, cols.ravel()] = rs.uniform(0, 24 * scene.PIX, B * k)
            d_c, d_k = d(api._cm(Cr, 2)[0]), d(sb["CalM"].T)
            r2, r3 = api._pose_pair(sb["R_t0"][0], sb["R_t0"][1], B, True)
            d_r2, d_r3 = d(r2), d(r3)
            o2, o3, oX, orep, ocost, ow, oit, ost = f64(B, 12), f64(B, 12), f64(B, 3 * n), f64(B), f64(B), f64(B, n), \
                i32(B), i32(B)
            plain = lambda: h.call("tvf_bundle_adjust_dev", p(d_c), p(d_k), 0, n, B, p(d_r2), p(d_r3), None, p(o2), p(o3),
                                   p(oX), p(orep), p(oit), p(ost))

            def robust(lid):
                return lambda: h.call("tvf_bundle_adjust_robust_dev", p(d_c), p(d_k), 0, n, B, lid, C.c_double(2.0),
                                      p(d_r2), p(d_r3), None, p(o2), p(o3), p(oX), p(orep), p(ocost), p(ow), p(oit), p(ost))
            ms = {k: [] for k in ["plain"] + list(LOSSES)}
            iters = {}
            for _ in range(3):                            # alternate the variants
                ms["plain"].append(timed(plain, args.reps))
                iters["plain"] = float(oit.float().mean())
                for name, lid in LOSSES.items():
                    ms[name].append(timed(robust(lid), args.reps))
                    iters[name] = float(oit.float().mean())
            row = dict(n=n, B=B, outliers=frac, scale_px=2.0,
                       adjustments_per_s={k: B / (np.median(v) * 1e-3) for k, v in ms.items()},
                       ms={k: v for k, v in ms.items()}, mean_iter=iters)
            rows.append(row)
            print(json.dumps(row), flush=True)
    out["cost_of_robustness"] = rows

    # ---- 2. EPFL, all raw matches --------------------------------------------------------------------------------------
    inp = np.load(os.path.join(ROOT, "tests", "golden", "epfl_inputs.npz"))
    Cs, Ks, R0, truth = [], [], [], []
    for key in ("fountain_P11", "Herz_Jesu_P8"):
        data = epfl.dataset_from_arrays(inp[key + "_indexes_sorted"], inp[key + "_matches"], inp[key + "_offsets"],
                                        inp[key + "_K"], inp[key + "_R"], inp[key + "_t"])
        for it in range(1, data.indexes_sorted.shape[0] + 1):
            im = [int(v) for v in data.indexes_sorted[it - 1, 0:3]]
            Cr = data.corresp(*im).T.copy()
            K, Rt = epfl.relative_poses([data.camera(i) for i in im])
            Cs.append(Cr); Ks.append(K); R0.append(Rt)
            truth.append(np.asarray(epfl.inlier_filter(Cr, K, Rt, 1.0)[1], dtype=bool))
    Bq = len(Cs)
    Ks = np.stack(Ks)
    c, offs = api._pack(Cs, 6)
    M = int(offs[-1])
    op = offs.ctypes.data_as(C.c_void_p)
    d_c, d_k, d_s = d(c), d(api._calm(Ks, Bq)[0]), d(np.arange(1, Bq + 1, dtype=np.uint64).view(np.int64))
    q2, q3, qm, qc, qs, qst, qlo = f64(Bq, 12), f64(Bq, 12), torch.zeros(M, dtype=torch.uint8, device=dev), i32(Bq), \
        i32(Bq, 7), i32(Bq), i32(Bq)
    b2, b3, bX, brep, bcost, bw, bit, bst = f64(Bq, 12), f64(Bq, 12), f64(3 * M), f64(Bq), f64(Bq), f64(M), i32(Bq), i32(Bq)
    ransac = lambda: h.call("tvf_ransac_pose_ragged_dev", 1, p(d_c), p(d_k), 1, op, Bq, 1024, 1.0, p(d_s), p(q2), p(q3),
                            p(qm), p(qc), p(qs), p(qst))
    robust = lambda: h.call("tvf_bundle_adjust_robust_ragged_dev", p(d_c), p(d_k), 1, op, Bq, 3, C.c_double(2.0), p(q2),
                            p(q3), None, p(b2), p(b3), p(bX), p(brep), p(bcost), p(bw), p(bit), p(bst))

    def a_pipeline():
        ransac(); robust()
    ransac(); torch.cuda.synchronize()
    mask = qm.cpu().numpy().astype(bool)
    sub = [Cs[b][:, mask[offs[b]:offs[b + 1]]] for b in range(Bq)]
    cc, coffs = api._pack(sub, 6)
    Mc = int(coffs[-1])
    cop = coffs.ctypes.data_as(C.c_void_p)
    d_cc = d(cc)
    p2, p3, pX, prep, pit, pst = f64(Bq, 12), f64(Bq, 12), f64(3 * max(Mc, 1)), f64(Bq), i32(Bq), i32(Bq)
    plain = lambda: h.call("tvf_bundle_adjust_ragged_dev", p(d_cc), p(d_k), 1, cop, Bq, p(q2), p(q3), None, p(p2), p(p3),
                           p(pX), p(prep), p(pit), p(pst))

    def b_pipeline():
        ransac(); plain()
    f2, f3, fm, fc, fs, flo, fst = f64(Bq, 12), f64(Bq, 12), torch.zeros(M, dtype=torch.uint8, device=dev), i32(Bq), \
        i32(Bq, 7), i32(Bq), i32(Bq)
    refined = lambda: h.call("tvf_ransac_pose_refined_ragged_dev", 1, p(d_c), p(d_k), 1, op, Bq, 1024, 1.0, p(d_s), 8,
                             p(f2), p(f3), p(fm), p(fc), p(fs), p(flo), p(fst))
    t = {"a_ransac_then_robust_all": [], "b_ransac_then_plain_on_consensus": [], "c_refined_ransac": []}
    for _ in range(3):
        t["a_ransac_then_robust_all"].append(timed(a_pipeline, args.reps))
        t["b_ransac_then_plain_on_consensus"].append(timed(b_pipeline, args.reps))
        t["c_refined_ransac"].append(timed(refined, args.reps))
    torch.cuda.synchronize()

    def errs(R2s, R3s):
        rot, tr = [], []
        for b in range(Bq):
            if not np.all(np.isfinite(R2s[b])):
                rot.append(np.inf); tr.append(np.inf); continue
            e2 = o.AngError(R0[b][0], R2s[b]); e3 = o.AngError(R0[b][1], R3s[b])
            rot.append((e2[0] + e3[0]) / 2); tr.append((e2[1] + e3[1]) / 2)
        return dict(median_rot_err_deg=float(np.median(rot)), median_t_err_deg=float(np.median(tr)))
    back = lambda x: api._from_cm(x.cpu().numpy().ravel(), Bq, (3, 4), True)
    w = bw.cpu().numpy()
    rec, prec = [], []
    for b in range(Bq):
        sel = w[offs[b]:offs[b + 1]] >= 0.5
        tp = np.sum(sel & truth[b])
        rec.append(tp / max(1, truth[b].sum())); prec.append(tp / max(1, sel.sum()))
    out["epfl"] = dict(
        triplets=Bq, matches=M, hypotheses=1024, threshold_px=1.0, cauchy_scale_px=2.0, lo_rounds=8,
        ms={k: float(np.median(v)) for k, v in t.items()}, ms_runs=t,
        plain_ransac=errs(back(q2), back(q3)),
        a_ransac_then_robust_all=dict(errs(back(b2), back(b3)), statuses=np.bincount(bst.cpu().numpy()).tolist(),
                                      weight_half_recall_mean=float(np.mean(rec)), weight_half_recall_median=float(np.median(rec)),
                                      weight_half_precision_mean=float(np.mean(prec))),
        b_ransac_then_plain_on_consensus=errs(back(p2), back(p3)),
        c_refined_ransac=errs(back(f2), back(f3)))
    print(json.dumps(out["epfl"]), flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
