"""Generate the committed golden vectors under tests/golden/ (run in the build container, where
/root/reference is mounted):   python tests/golden/make_golden.py

Inputs come from the documented scene generator / the reference's EPFL data files.  Expected outputs:
  tft_*/f_*          from the oracle (oracle/reference_port.py, the NumPy restatement);
  ref_tft_*/ref_f_*  from the reference's OWN unmodified .m files under /root/reference, executed by
                     oracle/mini_matlab.py (NumPy/LAPACK built-ins) -- these pin the restatement.  The GPU box has no /root/reference, so the `-m gpu`
tests read only these .npz files (plus the live oracle on the same seeded inputs)."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
import oracle as o  # noqa: E402

REFERENCE = "/root/reference"


_interp = None


def reference_run(C, CalM):
    """The reference's own .m files (unmodified, from /root/reference) executed by oracle/mini_matlab.py."""
    global _interp
    if not os.path.isdir(REFERENCE):
        return None
    from oracle.mini_matlab import reference_interpreter, Cell
    if _interp is None:
        _interp = reference_interpreter(REFERENCE, rng_factory=o.SceneRNG)
    K = [CalM[0:3], CalM[3:6], CalM[6:9]]
    out = {}
    for m, fn in (("tft", "LinearTFTPoseEstimation"), ("f", "LinearFPoseEstimation")):
        R2, R3, Rec, T, it = _interp.call(fn, [C.copy(), CalM.copy()], 5)
        assert float(np.asarray(it).item()) == 0.0
        rep = _interp.call("ReprError", [Cell([K[0] @ np.eye(3, 4), K[1] @ R2, K[2] @ R3]), C.copy(), Rec], 1)[0]
        out[m] = (R2, R3, Rec, T, float(np.asarray(rep).item()))
    return out


def run_both(C, CalM):
    K = [CalM[0:3], CalM[3:6], CalM[6:9]]
    out = {}
    ref = reference_run(C, CalM)
    if ref is not None:
        out["ref_tft"], out["ref_f"] = ref["tft"], ref["f"]
    R2, R3, Rec, T, _ = o.LinearTFTPoseEstimation(C, CalM)
    out["tft"] = (R2, R3, Rec, T, o.ReprError([K[0] @ np.eye(3, 4), K[1] @ R2, K[2] @ R3], C, Rec))
    R2, R3, Rec, T, _, F21, F31 = o.LinearFPoseEstimation(C, CalM, return_F=True)
    out["f"] = (R2, R3, Rec, T, o.ReprError([K[0] @ np.eye(3, 4), K[1] @ R2, K[2] @ R3], C, Rec), F21, F31)
    return out


def pack(cases):
    """cases: list of dict(Corresp, CalM, res=run_both(...)) with equal n -> arrays with a leading case axis."""
    d = dict(Corresp=np.stack([c["Corresp"] for c in cases]), CalM=np.stack([c["CalM"] for c in cases]))
    for m in ("tft", "f", "ref_tft", "ref_f"):
        if m not in cases[0]["res"]:
            continue
        names = ["Rt2", "Rt3", "Reconst", "T", "repr"] + (["F21", "F31"] if m == "f" else [])
        for k, name in enumerate(names):
            d["%s_%s" % (m, name)] = np.stack([np.asarray(c["res"][m][k]) for c in cases])
    for key in cases[0]:
        if key not in ("Corresp", "CalM", "res"):
            d[key] = np.stack([np.asarray(c[key]) for c in cases])
    return d


def sweep():
    """experiments.m defaults at the benchmark shape: 13 noise levels x n_sim=20 seeds, n=20."""
    cases = []
    for j in range(13 * 20):
        noise, seed = 0.25 * (j % 13), j // 13 + 1
        CalM, R_t0, C, _ = o.experiments_subsample(20, noise, seed)
        cases.append(dict(Corresp=C, CalM=CalM, res=run_both(C, CalM), noise=noise, seed=seed,
                          Rt0_2=R_t0[0], Rt0_3=R_t0[1]))
    d = pack(cases)
    # the ref_* arrays go to a companion file, which keeps each file under 1 MB
    np.savez_compressed(os.path.join(HERE, "sweep_n20.npz"), **{k: v for k, v in d.items() if not k.startswith("ref_")})
    np.savez_compressed(os.path.join(HERE, "sweep_n20_ref.npz"), **{k: v for k, v in d.items() if k.startswith("ref_")})


def example():
    """example.m:22-28: N=100, noise=1, seed=1, f=50, angle=0."""
    CalM, R_t0, C, _ = o.generateSyntheticScene(100, 1, 1, 50, 0)
    np.savez_compressed(os.path.join(HERE, "example_n100.npz"),
                        **pack([dict(Corresp=C, CalM=CalM, res=run_both(C, CalM), Rt0_2=R_t0[0], Rt0_3=R_t0[1])]))


def epfl(ntrip=6):
    """experiments_real.m:78-109 on the first triplets of both datasets (100 sampled inliers each)."""
    cases = []
    for ds in ("fountain-P11", "Herz-Jesu-P8"):
        path = os.path.join(REFERENCE, "Data", ds)
        idx, cor, names = o.load_corresp_triplets(path)
        for it in range(1, ntrip + 1):
            d = o.epfl_triplet(path, idx, cor, names, it)
            inl = d["Corresp_inliers"]
            sample = o.SceneRNG(it).randsample(inl.shape[1], min(100, inl.shape[1]))
            C = inl[:, sample]
            cases.append(dict(Corresp=C, CalM=d["CalM"], res=run_both(C, d["CalM"]), Rt0_2=d["R_t0"][0],
                              Rt0_3=d["R_t0"][1], n_inliers=inl.shape[1], gt_repr=d["REr"],
                              triplet=np.array(d["triplet"])))
    np.savez_compressed(os.path.join(HERE, "epfl_triplets.npz"), **pack(cases))


def optimf():
    """SURVEY 8 f4: OptimFPoseEstimation / optimF (Gauss-Helmert refinement of F) on the first 13 x 8 trials of the
    sweep (n = 20) and on N = 12 points (experiments.m's default N).  optf_* from the oracle port
    (oracle/gauss_helmert_port.py), ref_optf_* from the reference's unmodified .m files run by mini_matlab."""
    have_ref = os.path.isdir(REFERENCE)
    if have_ref:
        from oracle.mini_matlab import reference_interpreter
        interp = reference_interpreter(REFERENCE, rng_factory=o.SceneRNG)
    for name, n, ntr in (("optimf_n20.npz", 20, 13 * 8), ("optimf_n12.npz", 12, 13 * 3)):
        d = {}
        def put(k, v):
            d.setdefault(k, []).append(np.asarray(v))
        for j in range(ntr):
            noise, seed = 0.25 * (j % 13), j // 13 + 1
            CalM, R_t0, C, _ = o.experiments_subsample(n, noise, seed)
            K = CalM[:3]
            R2, R3, Rec, T, it, F21, F31 = o.OptimFPoseEstimation(C, CalM, return_F=True)
            rep = o.ReprError([K @ np.eye(3, 4), K @ R2, K @ R3], C, Rec)
            F, it1 = o.optimF(C[0:2], C[2:4])
            for k, v in (("Corresp", C), ("CalM", CalM), ("noise", noise), ("seed", seed), ("optf_Rt2", R2), ("optf_Rt3", R3),
                         ("optf_Reconst", Rec), ("optf_T", T), ("optf_iter", it), ("optf_F21", F21), ("optf_F31", F31),
                         ("optf_repr", rep), ("optf_F_single", F), ("optf_iter_single", it1)):
                put(k, v)
            if have_ref:
                r = interp.call("OptimFPoseEstimation", [C.copy(), CalM.copy()], 5)
                rF, rit = interp.call("optimF", [C[0:2].copy(), C[2:4].copy()], 2)
                for k, v in (("ref_optf_Rt2", r[0]), ("ref_optf_Rt3", r[1]), ("ref_optf_Reconst", r[2]), ("ref_optf_T", r[3]),
                             ("ref_optf_iter", float(np.asarray(r[4]).item())), ("ref_optf_F_single", rF),
                             ("ref_optf_iter_single", float(np.asarray(rit).item()))):
                    put(k, v)
        np.savez_compressed(os.path.join(HERE, name), **{k: np.stack(v) for k, v in d.items()})


def large_n(n=10000, seeds=(1, 2)):
    """BASELINE config 5 shape: n = 10 000 correspondences per scene, 1 px noise.  The oracle needs ~90 s per
    scene, so its outputs are stored; the inputs are regenerated from the seed by the test (the first points are
    stored as a generator check) and Reconst is stored for every 50th point only."""
    d = {k: [] for k in ("seed", "Corresp_head", "CalM", "Rt2", "Rt3", "T", "repr", "Reconst_sub")}
    for seed in seeds:
        CalM, R_t0, C, _ = o.generateSyntheticScene(n, 1.0, seed, 50, 0)
        K = CalM[:3]
        R2, R3, Rec, T, _ = o.LinearTFTPoseEstimation(C, CalM)
        rep = o.ReprError([K @ np.eye(3, 4), K @ R2, K @ R3], C, Rec)
        for k, v in (("seed", seed), ("Corresp_head", C[:, :8]), ("CalM", CalM), ("Rt2", R2), ("Rt3", R3), ("T", T),
                     ("repr", rep), ("Reconst_sub", Rec[:, ::50])):
            d[k].append(np.asarray(v))
    np.savez_compressed(os.path.join(HERE, "large_n10000.npz"), **{k: np.stack(v) for k, v in d.items()})


def oracle_votes(C, CalM):
    """The 4 + 4 cheirality votes of recover_R_t for both methods (R_t_from_TFT.m:91-104 with the tensor of
    LinearTFTPoseEstimation; LinearFPoseEstimation.m:94-107 with its two F), as the oracle computes them:
    candidate order (R,t),(R,-t),(Rp,-t),(Rp,t) per pair.  NaN sums are stored as NaN."""
    K1, K2, K3 = CalM[0:3], CalM[3:6], CalM[6:9]
    T = o.LinearTFTPoseEstimation(C, CalM)[3]
    _, _, v2, v3 = o.R_t_from_TFT(T, CalM, C, return_votes=True)
    F21, F31 = o.LinearFPoseEstimation(C, CalM, return_F=True)[5:7]
    f2 = o.recover_R_t_F(K1, K2, F21, C[0:2], C[2:4], return_votes=True)[2]
    f3 = o.recover_R_t_F(K1, K3, F31, C[0:2], C[4:6], return_votes=True)[2]
    return np.array(list(v2) + list(v3), dtype=np.float64), np.array(list(f2) + list(f3), dtype=np.float64)


def add_votes(name):
    """Add tft_votes / f_votes (cases x 8) to an existing golden file (VERDICT r1: votes were never compared)."""
    path = os.path.join(HERE, name)
    d = dict(np.load(path))
    tv, fv = [], []
    for b in range(d["Corresp"].shape[0]):
        a, c = oracle_votes(d["Corresp"][b], d["CalM"][b])
        tv.append(a); fv.append(c)
    d["tft_votes"] = np.stack(tv); d["f_votes"] = np.stack(fv)
    np.savez_compressed(path, **d)


DATASETS = (("fountain-P11", 70), ("Herz-Jesu-P8", 50))        # experiments_real.m:31-36


def epfl_inputs():
    """The raw inputs of experiments_real.m for every tested triplet (70 + 50): the match lists of
    Corresp_triplets.mat, the calibration/orientation of every image and indexes_sorted -- data, not code; the GPU
    box has no /root/reference, and tests/test_gpu_parity.py runs epfl.run_real on exactly these."""
    d = {}
    for ds, ntrip in DATASETS:
        path = os.path.join(REFERENCE, "Data", ds)
        idx, cor, names = o.load_corresp_triplets(path)
        key = ds.replace("-", "_")
        d[key + "_indexes_sorted"] = idx[:ntrip]
        cams = [o.readCalibrationOrientation_EPFL(path, nm) for nm in names]
        d[key + "_K"] = np.stack([c[0] for c in cams]); d[key + "_R"] = np.stack([c[1] for c in cams])
        d[key + "_t"] = np.stack([c[2] for c in cams])
        rows, offs = [], [0]
        for it in range(1, ntrip + 1):
            im = [int(v) for v in idx[it - 1, 0:3]]
            rows.append(np.asarray(cor[im[0] - 1, im[1] - 1, im[2] - 1], dtype=np.float64))
            offs.append(offs[-1] + rows[-1].shape[0])
        d[key + "_matches"] = np.concatenate(rows); d[key + "_offsets"] = np.array(offs, dtype=np.int64)
    np.savez_compressed(os.path.join(HERE, "epfl_inputs.npz"), **d)


def epfl_all():
    """experiments_real.m:75-138 for methods 1 and 7 on ALL tested triplets (70 of fountain-P11, 50 of Herz-Jesu-P8):
    per triplet the sample (seeded with the loop index, :103), the poses, T, the cheirality votes, and the row
    [ReprError over all inliers (:130-131), rot_err, t_err (:133-136)].  real_* from the oracle port, ref_real_* from
    the reference's unmodified .m files run by oracle/mini_matlab.py."""
    from oracle.mini_matlab import reference_interpreter, Cell
    interp = reference_interpreter(REFERENCE, rng_factory=o.SceneRNG)
    d = {}
    def put(k, v):
        d.setdefault(k, []).append(np.asarray(v))
    for dsi, (ds, ntrip) in enumerate(DATASETS):
        path = os.path.join(REFERENCE, "Data", ds)
        idx, cor, names = o.load_corresp_triplets(path)
        for it in range(1, ntrip + 1):
            t = o.epfl_triplet(path, idx, cor, names, it)
            inl, CalM, R_t0 = t["Corresp_inliers"], t["CalM"], t["R_t0"]
            N = inl.shape[1]
            sample = o.SceneRNG(it).randsample(N, min(100, N))
            C = inl[:, sample]
            Cpad = np.full((6, 100), np.nan); Cpad[:, :C.shape[1]] = C
            K = [CalM[0:3], CalM[3:6], CalM[6:9]]
            for k, v in (("dataset", dsi), ("it", it), ("triplet", t["triplet"]), ("n_inliers", N), ("n_sample", C.shape[1]),
                         ("gt_repr", t["REr"]), ("Corresp", Cpad), ("CalM", CalM), ("Rt0_2", R_t0[0]), ("Rt0_3", R_t0[1]),
                         ("sample", np.pad(sample, (0, 100 - sample.size), constant_values=-1))):
                put(k, v)
            tv, fv = oracle_votes(C, CalM)
            put("tft_votes", tv); put("f_votes", fv)
            for m, fn, mname in (("tft", o.LinearTFTPoseEstimation, "LinearTFTPoseEstimation"),
                                 ("f", o.LinearFPoseEstimation, "LinearFPoseEstimation")):
                R2, R3, _, T, _ = fn(C, CalM)
                rep = o.ReprError([K[0] @ np.eye(3, 4), K[1] @ R2, K[2] @ R3], inl)
                r2, t2 = o.AngError(R_t0[0], R2); r3, t3 = o.AngError(R_t0[1], R3)
                put(m + "_Rt2", R2); put(m + "_Rt3", R3); put(m + "_T", T)
                put("real_" + m, [rep, (r2 + r3) / 2, (t2 + t3) / 2])
                q2, q3, _, qT, _ = interp.call(mname, [C.copy(), CalM.copy()], 5)
                rrep = interp.call("ReprError", [Cell([K[0] @ np.eye(3, 4), K[1] @ q2, K[2] @ q3]), inl.copy()], 1)[0]
                a2 = interp.call("AngError", [R_t0[0].copy(), q2], 2); a3 = interp.call("AngError", [R_t0[1].copy(), q3], 2)
                put("ref_" + m + "_T", qT)
                put("ref_real_" + m, [float(np.asarray(rrep).item()),
                                      (float(np.asarray(a2[0]).item()) + float(np.asarray(a3[0]).item())) / 2,
                                      (float(np.asarray(a2[1]).item()) + float(np.asarray(a3[1]).item())) / 2])
            print(ds, it, N, flush=True)
    np.savez_compressed(os.path.join(HERE, "epfl_all_triplets.npz"), **{k: np.stack(v) for k, v in d.items()})


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "votes":
        for nm in ("sweep_n20.npz", "example_n100.npz", "epfl_triplets.npz"):
            add_votes(nm)
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "epfl_all":
        epfl_inputs(); epfl_all(); sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "large":
        large_n(); sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "optimf":
        optimf(); sys.exit(0)
    sweep(); example(); large_n(); optimf()
    if os.path.isdir(REFERENCE):
        epfl()
    print("golden vectors written to", HERE)
