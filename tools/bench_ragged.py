"""Ragged batches on the GPU (include/tvf.h), timed with CUDA events around whole _dev calls (inputs already on the device):

  1. RANSAC (plain and refined, methods 1 and 7, 1024 hypotheses, 1 px) over the 120 EPFL triplets with all raw matches:
     one ragged call, uniform calls grouped by exact n (108 distinct n among the 120 triplets: one batched call per
     group), and one uniform call per triplet in the fixture's order;
  2. ragged against uniform on equal n (synthetic, 30 % outliers): what the offset lookup costs in the consensus kernel
     (plain RANSAC, whose time is mostly the consensus) and in the adjustment;
  3. the ragged adjustment plus covariance over the 120 EPFL consensus sets, against one call per triplet.

    python tools/bench_ragged.py [--reps 5] [--out profiles/r07_ragged.json]

Each figure is the median of --reps timed calls after one warm-up call; the spread (min, max) is kept beside it.  The
`ptxas` registers and spills of the ragged kernels are read from the build's log (tft_vs_fund_b200/build.log)."""
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


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def ptxas_ragged():
    """registers, stack and spills of every *_ragged_kernel from the -Xptxas=-v output in the build log"""
    path = os.path.join(ROOT, "tft_vs_fund_b200", "build.log")
    if not os.path.exists(path):
        return None
    log = open(path).read().splitlines()
    out = {}
    for i, line in enumerate(log):
        m = re.search(r"Compiling entry function '\S*?\d+([a-z_]+_ragged_kernel)\w*'", line)
        if not m:
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
    return dict(ms=float(np.median(ts)), min_ms=float(min(ts)), max_ms=float(max(ts)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_ragged.json"))
    args = ap.parse_args()
    import torch
    import ransac_oracle as ro
    from test_gpu_ragged import epfl_problems
    from tft_vs_fund_b200 import _lib, api, scene
    h = _lib.handle(0)
    dev = torch.device("cuda", 0)
    h.call("tvf_set_stream", C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))    # the events' stream
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    Cs, Ks = epfl_problems()
    B = len(Cs)
    out = dict(gpu=gpu_info(), reps=args.reps, note="CUDA events around whole _dev calls; median (min, max) of reps")

    def ransac_runner(Clist, K, seeds, method, refine, H):
        """ragged _dev call over Clist, and per-problem uniform _dev calls in `order`"""
        s = ro.SAMPLE_SIZE[method]
        c, offs = api._pack(Clist, 6)
        Bn, M = len(Clist), int(offs[-1])
        d_c, d_k, d_s = d(c), d(api._calm(K, Bn)[0]), d(np.asarray(seeds, dtype=np.uint64).view(np.int64))
        o2 = torch.empty((Bn, 12), dtype=torch.float64, device=dev); o3 = torch.empty_like(o2)
        om = torch.zeros(M, dtype=torch.uint8, device=dev); oc = torch.zeros(Bn, dtype=torch.int32, device=dev)
        osm = torch.zeros((Bn, s), dtype=torch.int32, device=dev); ost = torch.zeros(Bn, dtype=torch.int32, device=dev)
        olo = torch.zeros(Bn, dtype=torch.int32, device=dev)
        op = offs.ctypes.data_as(C.c_void_p)
        cb = d_c.data_ptr(); kb = d_k.data_ptr(); sb = d_s.data_ptr()

        def ragged():
            if refine:
                h.call("tvf_ransac_pose_refined_ragged_dev", method, p(d_c), p(d_k), 1, op, Bn, H, 1.0, p(d_s), 8, p(o2),
                       p(o3), p(om), p(oc), p(osm), p(olo), p(ost))
            else:
                h.call("tvf_ransac_pose_ragged_dev", method, p(d_c), p(d_k), 1, op, Bn, H, 1.0, p(d_s), p(o2), p(o3), p(om),
                       p(oc), p(osm), p(ost))

        def uniform(order):
            def run():
                for b in order:
                    n = int(offs[b + 1] - offs[b])
                    args = (C.c_void_p(cb + 48 * int(offs[b])), C.c_void_p(kb + 216 * b), 1, n, 1, H, 1.0,
                            C.c_void_p(sb + 8 * b))
                    outs = (C.c_void_p(o2.data_ptr() + 96 * b), C.c_void_p(o3.data_ptr() + 96 * b),
                            C.c_void_p(om.data_ptr() + int(offs[b])), C.c_void_p(oc.data_ptr() + 4 * b),
                            C.c_void_p(osm.data_ptr() + 4 * s * b))
                    if refine:
                        h.call("tvf_ransac_pose_refined_dev", method, *args[:8], 8, *outs, C.c_void_p(olo.data_ptr() + 4 * b),
                               C.c_void_p(ost.data_ptr() + 4 * b))
                    else:
                        h.call("tvf_ransac_pose_dev", method, *args, *outs, C.c_void_p(ost.data_ptr() + 4 * b))
            return run

        def grouped():
            """one uniform call per group of equal n, on copies gathered beforehand"""
            calls = []
            for n_g in sorted(set(np.diff(offs).tolist())):
                idx = [b for b in range(Bn) if offs[b + 1] - offs[b] == n_g]
                k = len(idx)
                g_in = (d(np.concatenate([c[offs[b]:offs[b + 1]] for b in idx])), d(api._calm(K[idx], k)[0]),
                        d(np.asarray(seeds, dtype=np.uint64)[idx].view(np.int64)))
                g_out = [torch.empty((k, 12), dtype=torch.float64, device=dev) for _ in range(2)] + \
                    [torch.zeros(k * n_g, dtype=torch.uint8, device=dev)] + \
                    [torch.zeros(k * w, dtype=torch.int32, device=dev) for w in (1, s, 1, 1)]
                calls.append((int(n_g), k, g_in, g_out))

            def run():
                for n_g, k, (gc, gk, gs), (r2, r3, m, cnt, smp, lo, st) in calls:
                    if refine:
                        h.call("tvf_ransac_pose_refined_dev", method, p(gc), p(gk), 1, n_g, k, H, 1.0, p(gs), 8, p(r2),
                               p(r3), p(m), p(cnt), p(smp), p(lo), p(st))
                    else:
                        h.call("tvf_ransac_pose_dev", method, p(gc), p(gk), 1, n_g, k, H, 1.0, p(gs), p(r2), p(r3), p(m),
                               p(cnt), p(smp), p(st))
            return run, len(calls)

        def snapshot():
            torch.cuda.synchronize()
            return [t.cpu().numpy().copy() for t in (o2, o3, om, oc, osm, ost, olo)]
        return ragged, uniform, grouped, snapshot

    # ---- 1. EPFL RANSAC -------------------------------------------------------------------------------------------
    sizes = np.array([C_.shape[1] for C_ in Cs])
    res1 = {}
    for refine in (False, True):
        for method in (1, 7):
            ragged, uniform, grouped, snap = ransac_runner(Cs, Ks, np.arange(1, B + 1), method, refine, 1024)
            r = timed(ragged, args.reps); got = snap()
            run_g, n_groups = grouped()
            g = timed(run_g, args.reps)
            t = timed(uniform(range(B)), args.reps); want = snap()
            same = all(np.array_equal(x, y, equal_nan=True) for x, y in zip(got, want))
            res1["%s_method%d" % ("refined" if refine else "plain", method)] = dict(
                ragged_one_call=r, uniform_grouped_by_n=dict(g, calls=n_groups),
                uniform_per_triplet=dict(t, calls=B), ragged_equals_uniform=bool(same),
                speedup_vs_grouped=g["ms"] / r["ms"])
            print(json.dumps({k: res1[k] for k in list(res1)[-1:]}), flush=True)
    out["epfl_ransac"] = dict(triplets=B, matches=int(sizes.sum()), n_min=int(sizes.min()), n_max=int(sizes.max()),
                              hypotheses=1024, threshold_px=1.0, lo_rounds=8, results=res1)

    # ---- 2. equal n: ragged against uniform -------------------------------------------------------------------------
    Bq, n = 512, 100
    Cr, CalM, _, _ = ro.outlier_scenes(0.3, Bq, 71)
    Kb = np.broadcast_to(CalM, (Bq, 9, 3)).copy()
    ragged, _, _, snap = ransac_runner(list(Cr), Kb, np.arange(Bq), 1, False, 1024)
    d_c, d_k = d(api._cm(Cr, 2)[0]), d(api._calm(Kb, Bq)[0])
    d_s = d(np.arange(Bq, dtype=np.uint64).view(np.int64))
    u = [torch.empty((Bq, 12), dtype=torch.float64, device=dev) for _ in range(2)] + \
        [torch.zeros((Bq, n), dtype=torch.uint8, device=dev), torch.zeros(Bq, dtype=torch.int32, device=dev),
         torch.zeros((Bq, 7), dtype=torch.int32, device=dev), torch.zeros(Bq, dtype=torch.int32, device=dev)]
    unif = lambda: h.call("tvf_ransac_pose_dev", 1, p(d_c), p(d_k), 1, n, Bq, 1024, 1.0, p(d_s), *[p(t) for t in u])
    rows = []
    for _ in range(3):                                         # alternate the two forms
        rows.append((timed(unif, args.reps)["ms"], timed(ragged, args.reps)["ms"]))
    got = snap()
    same = np.array_equal(got[3], u[3].cpu().numpy()) and np.array_equal(got[0], u[0].cpu().numpy())
    eq = dict(ransac_plain=dict(B=Bq, n=n, hypotheses=1024, consensus_pairs=Bq * n * 1024,
                                uniform_ms=[r[0] for r in rows], ragged_ms=[r[1] for r in rows], equal_results=bool(same)))
    Bb = 65536
    sb = scene.sweep_batch(Bb, n=n, noise_levels=[1.0])
    c, offs = api._pack(list(sb["Corresp"]), 6)
    d_c, d_k = d(c), d(sb["CalM"].T)
    r2, r3 = api._pose_pair(sb["R_t0"][0], sb["R_t0"][1], Bb, True)
    d_r2, d_r3 = d(r2), d(r3)
    o = [torch.empty((Bb, 12), dtype=torch.float64, device=dev) for _ in range(2)] + \
        [torch.empty(3 * Bb * n, dtype=torch.float64, device=dev), torch.empty(Bb, dtype=torch.float64, device=dev),
         torch.zeros(Bb, dtype=torch.int32, device=dev), torch.zeros(Bb, dtype=torch.int32, device=dev)]
    op = offs.ctypes.data_as(C.c_void_p)
    ba_u = lambda: h.call("tvf_bundle_adjust_dev", p(d_c), p(d_k), 0, n, Bb, p(d_r2), p(d_r3), None, *[p(t) for t in o])
    ba_r = lambda: h.call("tvf_bundle_adjust_ragged_dev", p(d_c), p(d_k), 0, op, Bb, p(d_r2), p(d_r3), None, *[p(t) for t in o])
    rows = []
    for _ in range(3):
        tu = timed(ba_u, args.reps)["ms"]; ru = o[0].cpu().numpy().copy()
        tr = timed(ba_r, args.reps)["ms"]; rr = o[0].cpu().numpy().copy()
        rows.append((tu, tr))
    eq["bundle_adjust"] = dict(B=Bb, n=n, start="ground truth, 1 px noise", uniform_ms=[r[0] for r in rows],
                               ragged_ms=[r[1] for r in rows], equal_results=bool(np.array_equal(ru, rr)))
    out["equal_n"] = eq
    print(json.dumps(eq), flush=True)

    # ---- 3. adjustment + covariance over the EPFL consensus sets ---------------------------------------------------
    res = api.ransac_pose(Cs, Ks, method=1, hypotheses=1024, threshold=1.0, seed=np.arange(1, B + 1, dtype=np.uint64),
                          refine=True)
    Cm = [Cs[b][:, res[2][b]] for b in range(B)]
    c, offs = api._pack(Cm, 6)
    M = int(offs[-1])
    d_c, d_k = d(c), d(api._calm(Ks, B)[0])
    r2, r3 = api._pose_pair(res[0], res[1], B, True)
    d_r2, d_r3 = d(r2), d(r3)
    b2 = torch.empty((B, 12), dtype=torch.float64, device=dev); b3 = torch.empty_like(b2)
    bX = torch.empty(3 * M, dtype=torch.float64, device=dev); brep = torch.empty(B, dtype=torch.float64, device=dev)
    bit = torch.zeros(B, dtype=torch.int32, device=dev); bst = torch.zeros(B, dtype=torch.int32, device=dev)
    cc = torch.empty((B, 144), dtype=torch.float64, device=dev); cp = torch.empty(9 * M, dtype=torch.float64, device=dev)
    cs2 = torch.empty(B, dtype=torch.float64, device=dev); cst = torch.zeros(B, dtype=torch.int32, device=dev)
    op = offs.ctypes.data_as(C.c_void_p)

    def rag():
        h.call("tvf_bundle_adjust_ragged_dev", p(d_c), p(d_k), 1, op, B, p(d_r2), p(d_r3), None, p(b2), p(b3), p(bX),
               p(brep), p(bit), p(bst))
        h.call("tvf_ba_covariance_ragged_dev", p(d_c), p(d_k), 1, op, B, p(b2), p(b3), p(bX), p(cc), p(cp), p(cs2), p(cst))

    def loop():
        for b in range(B):
            n_b = int(offs[b + 1] - offs[b])
            if n_b < 4:
                continue
            a = lambda t, k, off=0: C.c_void_p(t.data_ptr() + k * off)
            h.call("tvf_bundle_adjust_dev", a(d_c, 48, int(offs[b])), a(d_k, 216, b), 1, n_b, 1, a(d_r2, 96, b),
                   a(d_r3, 96, b), None, a(b2, 96, b), a(b3, 96, b), a(bX, 24, int(offs[b])), a(brep, 8, b), a(bit, 4, b),
                   a(bst, 4, b))
            h.call("tvf_ba_covariance_dev", a(d_c, 48, int(offs[b])), a(d_k, 216, b), 1, n_b, 1, a(b2, 96, b),
                   a(b3, 96, b), a(bX, 24, int(offs[b])), a(cc, 1152, b), a(cp, 72, int(offs[b])), a(cs2, 8, b),
                   a(cst, 4, b))
    tr = timed(rag, args.reps); got = [t.cpu().numpy().copy() for t in (b2, bX, cc, cs2)]
    tl = timed(loop, args.reps); want = [t.cpu().numpy().copy() for t in (b2, bX, cc, cs2)]
    out["epfl_ba_covariance"] = dict(problems=B, matches=M, consensus_min=int(np.diff(offs).min()),
                                     consensus_max=int(np.diff(offs).max()), ragged_two_calls=tr, uniform_per_triplet=tl,
                                     equal_results=all(np.array_equal(x, y, equal_nan=True) for x, y in zip(got, want)))
    print(json.dumps(out["epfl_ba_covariance"]), flush=True)
    out["gpu_after"] = gpu_info()
    out["ptxas_sm_100a"] = ptxas_ragged()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
