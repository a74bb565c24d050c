"""The synthetic sweep of experiments.m, batched: every (noise level, seed) trial of
experiments.m:74-144 for the two linear methods in one (sharded) call.

experiments.m loops `interval` x `n_sim` x methods, calling `methods{m}(Corresp,CalM)` once per trial
(:107-109) and accumulating ReprError / AngError means per noise level (:112-124).  Here the trial
loop collapses into one batched call per method and rank; the accumulation is a per-level sum that is
gathered and added in rank order (tft_vs_fund_b200.sharding)."""
import numpy as np

from . import _lib, api, scene, sharding

NOISE_LEVELS = np.arange(0.0, 3.0 + 1e-9, 0.25)          # experiments.m:40  interval=0:0.25:3
METHODS = {1: ("Linear TFT", api.LinearTFTPoseEstimation), 7: ("Linear F", api.LinearFPoseEstimation),
           8: ("Optimal F", api.OptimFPoseEstimation)}          # numbering of experiments.m:51-59


def evaluate(res, R_t0, device=None):
    """Per-trial errors as experiments.m:112-120: (repr_err, rot_err, t_err) with the two views averaged."""
    B = res[0].shape[0]
    r2, t2 = api.AngError(R_t0[0], res[0], device=device)
    r3, t3 = api.AngError(R_t0[1], res[1], device=device)
    return np.asarray(res.repr_err).reshape(B), (r2 + r3) / 2.0, (t2 + t3) / 2.0


def level_sums(level_idx, n_levels, *columns, bad=None):
    """Sum each per-trial column per level -> (n_levels, len(columns)+2): sums, trials counted, trials skipped.
    `bad` (bool per trial): trials without a pose (status NO_POSE / NONFINITE) -- the reference would stop there on
    the undefined R_f; both sweep drivers leave them out of the sums and report their number per level (the same
    policy as sweep_eval_accumulate_kernel)."""
    level_idx = np.asarray(level_idx)
    good = np.ones(level_idx.shape, dtype=bool) if bad is None else ~np.asarray(bad, dtype=bool)
    out = np.zeros((n_levels, len(columns) + 2))
    for k, col in enumerate(columns):
        out[:, k] = np.bincount(level_idx[good], weights=np.asarray(col)[good], minlength=n_levels)
    out[:, -2] = np.bincount(level_idx[good], minlength=n_levels)
    out[:, -1] = np.bincount(level_idx[~good], minlength=n_levels)
    return out


def run_sweep(total_trials, n=20, methods=(1, 7), noise_levels=NOISE_LEVELS, focalL=50, angle=0, device=None,
              solver=None, workers=1, bundle_adjust=False):
    """Sharded sweep.  Returns on rank 0 a dict method -> (n_levels, 3) array of mean [repr_err, rot_err,
    t_err] per noise level (the `(:,m,1)` slices of experiments.m:68-70), None on the other ranks.
    `solver(method_id, Corresp, CalM)` may replace the GPU call (used by the CPU plumbing tests).
    bundle_adjust=True: every method's pose is then refined by api.bundle_adjust (what experiments.m:127-141 do with
    the reference's own BundleAdjustment, which this is not: DESIGN.md section 8) and each entry is (n_levels, 6):
    the three means above, then the same three after the adjustment.  Trials without a pose or with a non-finite
    adjustment are left out of the adjusted means."""
    if bundle_adjust and solver is not None:
        raise ValueError("bundle_adjust needs the library's pose methods (solver must be None)")
    rank, size = sharding.world()
    lo, hi = sharding.shard_range(total_trials, rank, size)
    d = scene.sweep_batch(hi - lo, n, first_trial=lo, noise_levels=noise_levels, focalL=focalL, angle=angle,
                          workers=workers)
    L = len(noise_levels)
    level_idx = (np.arange(lo, hi) % L).astype(np.int64)
    out = {}
    skipped = {}
    for m in methods:
        bad = None
        if solver is not None:
            repr_err, rot_err, t_err = solver(m, d["Corresp"], d["CalM"], d["R_t0"])
        else:
            res = METHODS[m][1](d["Corresp"], d["CalM"], device=device)
            repr_err, rot_err, t_err = evaluate(res, d["R_t0"], device=device)
            bad = (np.asarray(res.status) & (_lib.ST_NO_POSE_2 | _lib.ST_NO_POSE_3 | _lib.ST_NONFINITE)) != 0
        total = sharding.sum_in_rank_order(level_sums(level_idx, L, repr_err, rot_err, t_err, bad=bad))
        if bundle_adjust:
            ba = api.bundle_adjust(d["Corresp"], d["CalM"], res[0], res[1], res[2], device=device)
            bad_ba = bad | ((np.asarray(ba.status) & _lib.ST_NONFINITE) != 0)
            total_ba = sharding.sum_in_rank_order(level_sums(level_idx, L, *evaluate(ba, d["R_t0"], device=device), bad=bad_ba))
        if total is not None:
            out[m] = total[:, :3] / total[:, 3:4]
            if bundle_adjust:
                out[m] = np.hstack([out[m], total_ba[:, :3] / total_ba[:, 3:4]])
            skipped[m] = total[:, 4].astype(np.int64)
    if rank == 0:
        run_sweep.last_skipped = skipped        # trials without a pose per (method, level); all zero in the reference's sweeps
    return out if rank == 0 else None


def run_sweep_device(total_trials, n=20, methods=(1, 7), noise_levels=NOISE_LEVELS, focalL=50, angle=0, device=None,
                     bundle_adjust=False):
    """run_sweep with everything on the device (tvf_sweep_run): trials are generated, solved and reduced per
    noise level in HBM; each rank moves one L x 5 table.  Per-rank sums are added in rank order on rank 0.
    bundle_adjust=True: the device-resident twin of run_sweep(bundle_adjust=True) -- the noise levels become L levels of
    tvf_sweep_run_levels_ba with the same n, cameras, CalM and ground truth, and each entry is (n_levels, 6) as there.
    run_sweep_device.last_skipped_ba and .last_ba_iter then hold, per method and level, the trials left out of the
    adjusted means and the mean number of adjustment iterations."""
    if bundle_adjust:
        params = [dict(N=int(n), noise=float(v), f=focalL, angle=angle) for v in np.asarray(noise_levels, dtype=np.float64).ravel()]
        return _run_levels(run_sweep_device, params, total_trials, methods, device, True)
    rank, size = sharding.world()
    lo, hi = sharding.shard_range(total_trials, rank, size)
    noise_levels = np.ascontiguousarray(noise_levels, dtype=np.float64)
    L = noise_levels.size
    K, Ps, R_t0 = scene.scene_cameras(focalL, angle)
    P = np.ascontiguousarray(np.stack(Ps), dtype=np.float64)
    calm = np.ascontiguousarray(np.tile(K, (3, 1)).T)
    g2 = np.ascontiguousarray(R_t0[0].T); g3 = np.ascontiguousarray(R_t0[1].T)
    h = _lib.handle(device)
    dp = lambda a: a.ctypes.data_as(_lib.c_double_p)
    out = {}
    skipped = {}
    for m in methods:
        table = np.zeros((L, 5))
        h.call("tvf_sweep_run", int(m), lo, hi - lo, n, dp(noise_levels), L, dp(P), 36 * scene.PIX, 24 * scene.PIX,
               dp(calm), dp(g2), dp(g3), dp(table))
        total = sharding.sum_in_rank_order(table)
        if total is not None:
            out[m] = total[:, :3] / total[:, 3:4]
            skipped[m] = total[:, 4].astype(np.int64)
    if rank == 0:
        run_sweep_device.last_skipped = skipped
    return out if rank == 0 else None


def _sweep_levels(params):
    """tvf_sweep_level array of the per-level parameters (N, noise, f, angle)."""
    levels = (_lib.SweepLevel * len(params))()
    for lv, p in zip(levels, params):
        K, Ps, R_t0 = scene.scene_cameras(p["f"], p["angle"])
        lv.noise, lv.n = p["noise"], p["N"]
        lv.P[:] = np.ascontiguousarray(np.stack(Ps)).ravel()
        lv.calm[:] = np.tile(K, (3, 1)).T.ravel()
        lv.Rt0_2[:] = R_t0[0].T.ravel(); lv.Rt0_3[:] = R_t0[1].T.ravel()
    return levels


def _run_levels(driver, params, total_trials, methods, device, bundle_adjust):
    """tvf_sweep_run_levels[_ba] over the global trials [0, total_trials), sharded; per-rank tables added in rank order.
    Returns on rank 0 dict method -> (L, 3) means, or (L, 6) with the adjusted means; inf on the levels the reference
    skips.  Sets driver.last_skipped (and with bundle_adjust .last_skipped_ba, .last_ba_iter) on rank 0."""
    L = len(params)
    levels = _sweep_levels(params)
    W, fn = (11, "tvf_sweep_run_levels_ba") if bundle_adjust else (5, "tvf_sweep_run_levels")
    rank, size = sharding.world()
    lo, hi = sharding.shard_range(total_trials, rank, size)
    h = _lib.handle(device)
    out, skipped, skipped_ba, ba_iter = {}, {}, {}, {}
    for m in methods:
        table = np.zeros((L, W))
        h.call(fn, int(m), lo, hi - lo, levels, L, 36 * scene.PIX, 24 * scene.PIX, table.ctypes.data_as(_lib.c_double_p))
        unavailable = np.isinf(table[:, 0])
        table[unavailable, :3] = 0.0
        if bundle_adjust:
            table[unavailable, 5:8] = 0.0
        total = sharding.sum_in_rank_order(table)
        if total is not None:
            with np.errstate(divide="ignore", invalid="ignore"):
                out[m] = total[:, :3] / total[:, 3:4]
                if bundle_adjust:
                    out[m] = np.hstack([out[m], total[:, 5:8] / total[:, 8:9]])
                    ba_iter[m] = total[:, 10] / total[:, 8]
            out[m][unavailable] = np.inf
            skipped[m] = total[:, 4].astype(np.int64)
            if bundle_adjust:
                skipped_ba[m] = total[:, 9].astype(np.int64)
    if rank == 0:
        driver.last_skipped = skipped
        if bundle_adjust:
            driver.last_skipped_ba, driver.last_ba_iter = skipped_ba, ba_iter
    return out if rank == 0 else None


# ---- the four experiments of experiments.m:23-47 -------------------------------------------------------------
INTERVALS = {                                                                     # experiments.m:38-47
    "noise": [0.25 * k for k in range(13)],                                      # 0:0.25:3
    "focal": list(range(20, 301, 20)),                                           # 20:20:300
    "points": [7, 8, 9, 10, 15, 20, 25],                                         # [7:9,10:5:25]
    "angle": [166, 168, 170, 172, 174, 175, 176, 177, 178, 179, 179.5, 180],     # [166:2:174,175:179,179.5,180]
}


def experiment_levels(option, N=12, noise=1.0, f=50, angle=0, interval=None):
    """The per-level parameters (N, noise, f, angle) of experiments.m:74-89 for `option`; defaults are :30-33."""
    interval = INTERVALS[option] if interval is None else list(interval)
    out = []
    for v in interval:
        p = dict(N=int(N), noise=float(noise), f=f, angle=angle)
        p[{"noise": "noise", "focal": "f", "points": "N", "angle": "angle"}[option]] = int(v) if option == "points" else v
        out.append(p)
    return interval, out


def run_experiment(option, n_sim=20, methods=(1, 7), N=12, noise=1.0, f=50, angle=0, interval=None, device=None,
                   bundle_adjust=False):
    """experiments.m for one `option`, device-resident (tvf_sweep_run_levels): level i x seeds 1..n_sim x methods.  Sharded
    like run_sweep (contiguous ranges of the global trial index j = (seed-1)*L + level).  Returns on rank 0
    (interval, dict method -> (L, 3) mean [repr_err, rot_err, t_err]; inf where the reference skips the method for lack
    of matches, experiments.m:99-104), None elsewhere.
    bundle_adjust=True (tvf_sweep_run_levels_ba): every pose is then refined by the library's bundle adjustment (not the
    reference's BundleAdjustment.m, DESIGN.md section 8) on the device, and each entry is (L, 6): the three means, then the
    same three after the adjustment, as run_sweep(bundle_adjust=True).  run_experiment.last_skipped_ba (trials left out of
    the adjusted means: no pose, or a non-finite adjustment) and .last_ba_iter (mean adjustment iterations) are per level."""
    interval, params = experiment_levels(option, N, noise, f, angle, interval)
    out = _run_levels(run_experiment, params, len(params) * n_sim, methods, device, bundle_adjust)
    return (interval, out) if out is not None else None


def run_experiment_host(option, n_sim=20, methods=(1, 7), N=12, noise=1.0, f=50, angle=0, interval=None, device=None,
                        bundle_adjust=False):
    """The same experiment driven from the host (inputs from scene.sweep_batch, one batched solver call per level and
    method, NumPy reduction): the twin the tests hold run_experiment against.  bundle_adjust=True: api.bundle_adjust from
    each method's (R_t_2, R_t_3, Reconst), evaluated as the method; entries (L, 6) and, as for run_experiment,
    run_experiment_host.last_skipped, .last_skipped_ba and .last_ba_iter per method and level."""
    interval, params = experiment_levels(option, N, noise, f, angle, interval)
    L = len(params)
    out = {m: np.zeros((L, 6 if bundle_adjust else 3)) for m in methods}
    skipped = {m: np.zeros(L, dtype=np.int64) for m in methods}
    skipped_ba = {m: np.zeros(L, dtype=np.int64) for m in methods}
    ba_iter = {m: np.full(L, np.nan) for m in methods}
    for i, p in enumerate(params):
        d = scene.sweep_batch(n_sim, p["N"], noise_levels=[p["noise"]], focalL=p["f"], angle=p["angle"])
        lvl = np.zeros(n_sim, dtype=np.int64)
        for m in methods:
            if (m > 6 and p["N"] < 8) or p["N"] < 7:                                                 # experiments.m:99-104
                out[m][i] = np.inf
                continue
            res = METHODS[m][1](d["Corresp"], d["CalM"], device=device)
            repr_err, rot_err, t_err = evaluate(res, d["R_t0"], device=device)
            bad = (np.asarray(res.status) & (_lib.ST_NO_POSE_2 | _lib.ST_NO_POSE_3 | _lib.ST_NONFINITE)) != 0
            sums = level_sums(lvl, 1, repr_err, rot_err, t_err, bad=bad)
            out[m][i, :3] = sums[0, :3] / sums[0, 3]
            skipped[m][i] = int(sums[0, 4])
            if bundle_adjust:
                ba = api.bundle_adjust(d["Corresp"], d["CalM"], res[0], res[1], res[2], device=device)
                bad_ba = bad | ((np.asarray(ba.status) & _lib.ST_NONFINITE) != 0)
                sums = level_sums(lvl, 1, *evaluate(ba, d["R_t0"], device=device), np.asarray(ba[3], dtype=np.float64),
                                  bad=bad_ba)
                with np.errstate(divide="ignore", invalid="ignore"):
                    out[m][i, 3:] = sums[0, :3] / sums[0, 4]
                    ba_iter[m][i] = sums[0, 3] / sums[0, 4]
                skipped_ba[m][i] = int(sums[0, 5])
    run_experiment_host.last_skipped = skipped
    if bundle_adjust:
        run_experiment_host.last_skipped_ba, run_experiment_host.last_ba_iter = skipped_ba, ba_iter
    return interval, out
