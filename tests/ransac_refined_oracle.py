"""CPU oracle of the refined RANSAC pose estimator (tvf_ransac_pose_refined, include/tvf.h), for the tests: the rule in
NumPy on tests/ransac_oracle.py (sampler, method solves, inlier test) and oracle/bundle_adjust.py (the adjustment, SciPy's
Levenberg-Marquardt from points triangulated by oracle.triangulation3D)."""
import numpy as np
from scipy.optimize import least_squares

import oracle as o
import ransac_oracle as ro
from oracle import bundle_adjust as oba


# oracle.bundle_adjust.bundle_adjust's minimisation with an evaluation budget: a sample with outliers can take MINPACK
# tens of thousands of evaluations, where the library stops after 400 damped solves (TVF_ST_BA_NOCONV, still scored)
MAX_NFEV = 400


def adjust(Corresp, CalM, R_t_2, R_t_3):
    """tvf_bundle_adjust(reconst0 = NULL) on Corresp from (R_t_2, R_t_3): (R_t_2, R_t_3) adjusted, or None where the
    library reports TVF_ST_NONFINITE (a non-finite input, start point or start cost, or |t2| = 0)."""
    Ps = [CalM[0:3] @ np.eye(3, 4), CalM[3:6] @ R_t_2, CalM[6:9] @ R_t_3]
    if not (np.all(np.isfinite(Corresp)) and all(np.all(np.isfinite(P)) for P in Ps)) or not np.linalg.norm(R_t_2[:, 3]) > 0:
        return None
    with np.errstate(all="ignore"):
        X = o.triangulation3D(Ps, Corresp)
        X = X[0:3] / X[3:4]
        if not np.all(np.isfinite(X)) or not np.isfinite(oba.repr_error([CalM[0:3], CalM[3:6], CalM[6:9]], R_t_2[:, :3],
                                                                         R_t_2[:, 3], R_t_3[:, :3], R_t_3[:, 3], X, Corresp)):
            return None
        Ks = [CalM[0:3], CalM[3:6], CalM[6:9]]
        ch = oba.Chart(*oba.normalise_gauge(R_t_2[:, :3], R_t_2[:, 3], R_t_3[:, :3], R_t_3[:, 3], X))
        sol = least_squares(lambda p: oba.residuals(Ks, *ch.unpack(p), Corresp), np.zeros(11 + 3 * X.shape[1]),
                            jac=lambda p: ch.jacobian(Ks, p, Corresp).toarray(), method="lm", xtol=1e-15, ftol=1e-15,
                            gtol=1e-15, max_nfev=MAX_NFEV)
        R2, t2, R3, t3, _ = ch.unpack(sol.x)
    if not (np.all(np.isfinite(R2)) and np.all(np.isfinite(t2)) and np.all(np.isfinite(R3)) and np.all(np.isfinite(t3))):
        return None
    return np.column_stack([R2, t2]), np.column_stack([R3, t3])


def ransac_refined(Corresp, CalM, method, H, th, seed, lo_rounds=8):
    """tvf_ransac_pose_refined on one problem.  Returns a dict: Rt2, Rt3, inliers, n_inliers, sample, status (0 or 128),
    lo_done, counts (H; -1 = flagged), margins (H x N, as ransac_oracle.ransac), best, lo_counts (the count after the
    selection and after every accepted LO round) and lo_margins (per LO round tried: |max residual - th| per match)."""
    s = ro.SAMPLE_SIZE[method]
    n = Corresp.shape[1]
    idx = ro.sample(seed, np.arange(H), n, s)
    counts = np.full(H, -1, dtype=np.int64)
    margins = np.full((H, n), np.nan)
    poses, masks = [None] * H, [None] * H
    for h in range(H):
        pose = ro.solve(method, Corresp[:, idx[h]], CalM)
        if pose is None:
            continue
        pose = adjust(Corresp[:, idx[h]], CalM, pose[0], pose[1])
        if pose is None:
            continue
        mask, mx = ro.inliers(Corresp, CalM, pose[0], pose[1], th)
        counts[h], margins[h], poses[h], masks[h] = int(mask.sum()), np.abs(mx - th), pose, mask
    best = int(np.argmax(counts))                       # the first of equal counts: the smallest h
    out = dict(counts=counts, margins=margins, best=best, lo_counts=[], lo_margins=[])
    if counts[best] < 0:
        return dict(out, Rt2=np.full((3, 4), np.nan), Rt3=np.full((3, 4), np.nan), inliers=np.zeros(n, bool), n_inliers=0,
                    sample=np.full(s, -1), status=128, lo_done=0)
    pose, mask, cnt = poses[best], masks[best], int(counts[best])
    out["lo_counts"].append(cnt)
    done = 0
    for _ in range(lo_rounds):
        if cnt < 4:
            break
        p = adjust(Corresp[:, mask], CalM, pose[0], pose[1])
        if p is None:
            break
        m, mx = ro.inliers(Corresp, CalM, p[0], p[1], th)
        out["lo_margins"].append(np.abs(mx - th))
        if not m.sum() > cnt:
            break
        pose, mask, cnt, done = p, m, int(m.sum()), done + 1
        out["lo_counts"].append(cnt)
    return dict(out, Rt2=pose[0], Rt3=pose[1], inliers=mask, n_inliers=cnt, sample=idx[best], status=0, lo_done=done)


def near_threshold(res, tol):
    """Whether a match of a hypothesis that could have won (count >= best - 1), or of an LO round, lies within tol of
    the threshold: there a rounding difference may change the result."""
    best = res["counts"][res["best"]]
    near = bool(np.any(res["margins"][res["counts"] >= best - 1] < tol))
    return near or any(bool(np.any(m < tol)) for m in res["lo_margins"])
