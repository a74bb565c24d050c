"""CPU oracle of the RANSAC pose estimator (tvf_ransac_pose, include/tvf.h), for the tests: the same algorithm in NumPy
on the oracle's pose methods (oracle.LinearTFTPoseEstimation / LinearFPoseEstimation per hypothesis) and its
triangulation (oracle.triangulation3D), with the NumPy twin of the counter-based sampler of csrc/tvf_ransac.cuh."""
import numpy as np

import oracle as o

SAMPLE_SIZE = {1: 7, 7: 8}
METHODS = {1: o.LinearTFTPoseEstimation, 7: o.LinearFPoseEstimation}
_GOLD, _M1, _M2 = np.uint64(0x9E3779B97F4A7C15), np.uint64(0xBF58476D1CE4E5B9), np.uint64(0x94D049BB133111EB)


def mix64(z):
    """splitmix64's output function on uint64 arrays (wrapping arithmetic)."""
    z = np.asarray(z, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = z + _GOLD
        z = (z ^ (z >> np.uint64(30))) * _M1
        z = (z ^ (z >> np.uint64(27))) * _M2
    return z ^ (z >> np.uint64(31))


def draw(seed, h, j):
    """r = mix64(seed ^ mix64((h << 8) | j)), elementwise."""
    hj = (np.asarray(h, dtype=np.uint64) << np.uint64(8)) | np.asarray(j, dtype=np.uint64)
    return mix64(np.asarray(seed, dtype=np.uint64) ^ mix64(hj))


def uniform(r, m):
    """((r >> 32) * m) >> 32: a uniform integer in [0, m)."""
    return ((np.asarray(r, dtype=np.uint64) >> np.uint64(32)) * np.asarray(m, dtype=np.uint64)) >> np.uint64(32)


def sample(seed, h, n, s):
    """Floyd's algorithm: the s distinct indices of hypotheses h (array) of key seed, in draw order -> (len(h), s)."""
    h = np.atleast_1d(np.asarray(h, dtype=np.uint64))
    out = np.zeros((h.size, s), dtype=np.int64)
    for j in range(s):
        m = n - s + j + 1
        u = uniform(draw(seed, h, j), m).astype(np.int64)
        taken = np.any(out[:, :j] == u[:, None], axis=1)
        out[:, j] = np.where(taken, m - 1, u)
    return out


def residuals(Corresp, CalM, R_t_2, R_t_3):
    """|re-projection - observation| (6 x N) of every match triangulated with K1[I|0], K2 R_t_2, K3 R_t_3; NaN for a
    match or a pose that is not finite (LAPACK's SVD does not take them)."""
    Ps = [CalM[0:3] @ np.eye(3, 4), CalM[3:6] @ R_t_2, CalM[6:9] @ R_t_3]
    ok = np.all(np.isfinite(Corresp), axis=0) & all(np.all(np.isfinite(P)) for P in Ps)
    r = np.full(Corresp.shape, np.nan)
    with np.errstate(all="ignore"):
        X = o.triangulation3D(Ps, Corresp[:, ok])
        r[:, ok] = np.abs(o.project3Dpoints(X[0:3] / X[3:4], Ps) - Corresp[:, ok])
    return r


def inliers(Corresp, CalM, R_t_2, R_t_3, th):
    """(mask, max residual per match): inlier iff all six residuals are finite and <= th (NaN: outlier)."""
    r = residuals(Corresp, CalM, R_t_2, R_t_3)
    with np.errstate(invalid="ignore"):
        return np.all(r <= th, axis=0), np.max(r, axis=0)


def solve(method, Corresp, CalM):
    """The method's pose, or None where the library flags the problem (no pose, a non-finite result)."""
    try:
        with np.errstate(all="ignore"):
            R2, R3 = METHODS[method](Corresp, CalM)[:2]
    except Exception:
        return None
    if R2 is None or R3 is None or not (np.all(np.isfinite(R2)) and np.all(np.isfinite(R3))):
        return None
    return R2, R3


def ransac(Corresp, CalM, method, H, th, seed):
    """tvf_ransac_pose on one problem.  Returns a dict: Rt2, Rt3, inliers, n_inliers, sample, status (0 or 128),
    counts (H; -1 = flagged), margins (H x N: |max residual - th| per match, NaN for a NaN residual), best, refit
    (whether the refit was returned) and refit_margins (N, or None)."""
    s = SAMPLE_SIZE[method]
    n = Corresp.shape[1]
    idx = sample(seed, np.arange(H), n, s)
    counts = np.full(H, -1, dtype=np.int64)
    margins = np.full((H, n), np.nan)
    poses, masks = [None] * H, [None] * H
    for h in range(H):
        pose = solve(method, Corresp[:, idx[h]], CalM)
        if pose is None:
            continue
        mask, mx = inliers(Corresp, CalM, pose[0], pose[1], th)
        counts[h], margins[h], poses[h], masks[h] = int(mask.sum()), np.abs(mx - th), pose, mask
    best = int(np.argmax(counts))                       # the first of equal counts: the smallest h
    out = dict(counts=counts, margins=margins, best=best, refit=False, refit_margins=None)
    if counts[best] < 0:
        return dict(out, Rt2=np.full((3, 4), np.nan), Rt3=np.full((3, 4), np.nan), inliers=np.zeros(n, bool), n_inliers=0,
                    sample=np.full(s, -1), status=128)
    res = dict(out, Rt2=poses[best][0], Rt3=poses[best][1], inliers=masks[best], n_inliers=int(counts[best]),
               sample=idx[best], status=0)
    if counts[best] >= s:
        pose = solve(method, Corresp[:, masks[best]], CalM)
        if pose is not None:
            mask, mx = inliers(Corresp, CalM, pose[0], pose[1], th)
            res["refit_margins"] = np.abs(mx - th)
            if mask.sum() >= counts[best]:
                res.update(Rt2=pose[0], Rt3=pose[1], inliers=mask, n_inliers=int(mask.sum()), refit=True)
    return res


def near_threshold(res, tol):
    """Whether a match of a hypothesis that could have won (count >= best - 1), or of the refit, lies within tol of the
    threshold: there a rounding difference may change the result."""
    best = res["counts"][res["best"]]
    rows = res["margins"][res["counts"] >= best - 1]
    near = bool(np.any(rows < tol))
    if res["refit_margins"] is not None:
        near = near or bool(np.any(res["refit_margins"] < tol))
    return near


def outlier_scenes(f, count, seed, noise=1.0):
    """`count` sweep scenes (tft_vs_fund_b200.scene.sweep_batch, n = 100, `noise` px) whose columns are replaced, a share f of
    them chosen at random, by uniform pixels of the 1800 x 1200 image in all three views.  Returns
    (Corresp (count, 6, 100), CalM, R_t0, outlier mask (count, 100))."""
    from tft_vs_fund_b200 import scene
    d = scene.sweep_batch(count, n=100, noise_levels=[noise])
    Cr = d["Corresp"].copy()
    rs = np.random.RandomState(seed)
    out = np.zeros((count, 100), dtype=bool)
    for b in range(count):
        cols = rs.choice(100, int(round(f * 100)), replace=False)
        out[b, cols] = True
        Cr[b][0::2, cols] = rs.uniform(0.0, 36 * scene.PIX, size=(3, cols.size))
        Cr[b][1::2, cols] = rs.uniform(0.0, 24 * scene.PIX, size=(3, cols.size))
    return Cr, d["CalM"], d["R_t0"], out


def hypotheses_for(f, s):
    """H = ceil(log(1e-3) / log(1 - (1 - f)^s)): an all-inlier sample with probability 0.999."""
    return int(np.ceil(np.log(1e-3) / np.log(1.0 - (1.0 - f) ** s)))


def robustness_stats(method, Cr, CalM, R_t0, outliers, results):
    """Per-problem rotation error (degrees, mean of views 2 and 3) of `results` (list of (Rt2, Rt3, inliers)), the same
    for the method run on the true inlier columns, and recall / precision of the true inliers."""
    rot, ref, rec, prec = [], [], [], []
    for b, (R2, R3, mask) in enumerate(results):
        truth = ~outliers[b]
        rot.append((o.AngError(R_t0[0], R2)[0] + o.AngError(R_t0[1], R3)[0]) / 2 if np.all(np.isfinite(R2)) else np.inf)
        p = METHODS[method](Cr[b][:, truth], CalM)
        ref.append((o.AngError(R_t0[0], p[0])[0] + o.AngError(R_t0[1], p[1])[0]) / 2)
        tp = np.sum(mask & truth)
        rec.append(tp / truth.sum()); prec.append(tp / max(1, mask.sum()))
    rot, ref = np.array(rot), np.array(ref)
    return dict(share_below_1deg=float(np.mean(rot < 1.0)), median_ratio=float(np.median(rot) / np.median(ref)),
                recall=float(np.mean(rec)), precision=float(np.mean(prec)))
