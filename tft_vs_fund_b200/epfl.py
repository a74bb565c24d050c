"""Real-data side of the path (SURVEY.md 8 f2): the EPFL fountain-P11 / Herz-Jesu-P8 triplets.

Host-side loaders (`.camera` text files, the MAT-v5 `Corresp_triplets.mat`) and the per-triplet preparation
of experiments_real.m:78-109, with the numerical steps -- triangulation of all N matches with the
ground-truth cameras, re-projection, 1-pixel inlier mask, ReprError without 3-D points -- on the GPU through
the C ABI (tvf_triangulate, tvf_project3d, tvf_repr_error)."""
import os

import numpy as np

from . import api


def _row(line):
    return [float(tok) for tok in line.split()]


def readCalibrationOrientation_EPFL(image_path, image_name):
    """[K,R,t,im_size]=readCalibrationOrientation_EPFL(image_path,image_name)
    (Data/readCalibrationOrientation_EPFL.m:1,5-22): K (3 lines), one skipped line, R' (3 lines), camera
    centre C -> t = -R*C, image size."""
    with open(os.path.join(image_path, image_name + ".camera")) as f:
        ln = f.read().splitlines()
    K = np.array([_row(ln[0]), _row(ln[1]), _row(ln[2])])
    R = np.array([_row(ln[4]), _row(ln[5]), _row(ln[6])]).T
    t = -R @ np.array(_row(ln[7]))
    return K, R, t, np.array(_row(ln[8]))


def load_corresp_triplets(path_to_data):
    """experiments_real.m:45-48: indexes_sorted (K x 4: i, j, k, N by descending N), Corresp cell, im_names."""
    import scipy.io as sio
    m = sio.loadmat(os.path.join(path_to_data, "Corresp_triplets.mat"))
    return (m["indexes_sorted"].astype(np.int64), m["Corresp"], [str(x[0]) for x in m["im_names"].ravel()])


class Dataset:
    """What experiments_real.m:45-48,86-88 reads for one EPFL dataset: `indexes_sorted` (K x 4), the match list of a
    triplet (N x 6, by 1-based image numbers) and the calibration/orientation (K, R, t) of an image."""

    def __init__(self, indexes_sorted, corresp, camera):
        self.indexes_sorted = np.asarray(indexes_sorted, dtype=np.int64)
        self._corresp, self._camera = corresp, camera

    def corresp(self, im1, im2, im3):
        return np.asarray(self._corresp(im1, im2, im3), dtype=np.float64)

    def camera(self, im):
        return self._camera(im)


def load_dataset(path_to_data):
    """Dataset from the reference's files: Corresp_triplets.mat (MAT v5) and the `.camera` text files."""
    idx, cor, names = load_corresp_triplets(path_to_data)
    return Dataset(idx, lambda a, b, c: cor[a - 1, b - 1, c - 1],
                   lambda im: readCalibrationOrientation_EPFL(path_to_data, names[im - 1])[:3])


def dataset_from_arrays(indexes_sorted, matches, offsets, K, R, t):
    """Dataset from packed arrays (the committed fixture tests/golden/epfl_inputs.npz): row r of indexes_sorted owns
    matches[offsets[r]:offsets[r+1]]; K, R, t are stacked per image."""
    idx = np.asarray(indexes_sorted, dtype=np.int64)
    rows = {tuple(int(v) for v in idx[r, :3]): r for r in range(idx.shape[0])}

    def corresp(a, b, c):
        r = rows[(a, b, c)]
        return matches[offsets[r]:offsets[r + 1]]
    return Dataset(idx, corresp, lambda im: (K[im - 1], R[im - 1], t[im - 1]))


def relative_poses(cams):
    """experiments_real.m:89-91: CalM = [K1;K2;K3], R_t0 = {[R2*R1', t2-R2*R1'*t1], [R3*R1', t3-R3*R1'*t1]}."""
    (K1, R1, t1), (K2, R2, t2), (K3, R3, t3) = cams
    CalM = np.vstack([K1, K2, K3])
    R_t0 = [np.column_stack([R2 @ R1.T, t2 - R2 @ R1.T @ t1]), np.column_stack([R3 @ R1.T, t3 - R3 @ R1.T @ t1])]
    return CalM, R_t0


def inlier_filter(Corresp, CalM, R_t0, repr_err_th=1.0, device=None):
    """experiments_real.m:94-100 on the GPU: triangulate every match with the ground-truth cameras, re-project,
    keep the columns whose six residuals are all <= repr_err_th pixels.  Returns (Corresp_inliers, mask, REr)."""
    K1, K2, K3 = CalM[0:3], CalM[3:6], CalM[6:9]
    Ps = [K1 @ np.eye(3, 4), K2 @ R_t0[0], K3 @ R_t0[1]]
    X = api.triangulation3D(Ps, Corresp, device=device)                     # :94
    Reconst0 = X[0:3] / X[3:4]                                              # :95
    Corresp_new = api.project3Dpoints(Reconst0, Ps, device=device)          # :96
    residuals = Corresp_new - Corresp                                       # :97
    mask = np.sum(np.abs(residuals) > repr_err_th, axis=0) == 0             # :98
    inl = Corresp[:, mask]
    REr = api.ReprError(Ps, inl, device=device)                             # :100 (triangulates the inliers itself)
    return inl, mask, REr


def prepare_triplet(data, it, repr_err_th=1.0, device=None):
    """experiments_real.m:78-101 for the 1-based row `it` of indexes_sorted.  data: a Dataset."""
    im = [int(v) for v in data.indexes_sorted[it - 1, 0:3]]
    Corresp = data.corresp(*im).T                                                                       # :80
    cams = [data.camera(i) for i in im]                                                                 # :86-88
    CalM, R_t0 = relative_poses(cams)
    inl, mask, REr = inlier_filter(Corresp, CalM, R_t0, repr_err_th, device)
    return dict(triplet=tuple(im), CalM=CalM, R_t0=R_t0, Corresp=Corresp, Corresp_inliers=inl, inlier_mask=mask, REr=REr)


def consensus_stats(mask, truth):
    """A consensus mask against the ground-truth inlier mask: dict(mask, size, precision, recall)."""
    mask = np.asarray(mask, dtype=bool); truth = np.asarray(truth, dtype=bool)
    tp = int(np.sum(mask & truth))
    size = int(np.sum(mask))
    return dict(mask=mask, size=size, precision=tp / size if size else 0.0,
                recall=tp / int(np.sum(truth)) if np.any(truth) else 0.0)


def run_real(data, triplets_to_test, initial_sample_size=100, methods=(1, 7), device=None, details=None,
             bundle_adjust=False, covariance=False, raw_matches=False):
    """The linear-method part of experiments_real.m:75-138.  `data`: a Dataset or the path of a dataset directory;
    `triplets_to_test`: rows of indexes_sorted (1-based; the reference uses 1:70 / 1:50, :31-36).  Per loop index `it`:
    pre-filter (:94-101), sample min(100, N) inliers with rng(it) (:103-105; documented stand-in for MATLAB's
    randsample: scene.SceneRNG(it).randsample), run methods 1 / 7 on the sample (:126), evaluate ReprError over ALL
    inliers (triangulating them, :130-131) and AngError against the ground truth (:133-136).
    Returns dict method -> array (len(triplets_to_test), 3) of [repr_err, rot_err, t_err]; `details` (a list) receives
    one dict per triplet (inlier count, ground-truth RMS, sample, per-method poses / T / votes).
    bundle_adjust=True: each method's pose is then refined by api.bundle_adjust on the same sample, from the method's
    R_t_2, R_t_3 and Reconst -- the library's three-view adjustment, not the reference's BundleAdjustment.m (DESIGN.md
    section 8) -- and the adjusted cameras are evaluated exactly as the method's.  Each entry is then (T, 6): the three
    errors of the method, then the same three after the adjustment; details[k]["ba"][m] holds the adjusted result.
    covariance=True (with bundle_adjust): api.ba_covariance is also taken at each adjusted pose, and
    details[k]["ba"][m] gets .sigma2 (the a-posteriori pixel noise variance of the sample) and the predicted RMS
    rotation / translation errors .pred_rot_err, .pred_t_err (degrees, api.pose_rms_errors scaled by sigma2, the mean
    of the two views as :133-136).  The returned error columns are unchanged.
    raw_matches=True: the pose comes from api.ransac_pose on ALL N matches of the triplet (1024 hypotheses, threshold
    1 px, seed = it), so the ground truth is not used for estimation; the evaluation is unchanged (ReprError over the
    ground-truth inliers, AngError against the ground truth).  details[k]["consensus"][m] holds the consensus mask, its
    size and its precision and recall against the ground-truth inlier mask; bundle_adjust / covariance run on the
    consensus columns, starting from the RANSAC pose (the points triangulated from it); a consensus of fewer than 4
    matches cannot be adjusted and gets +inf in the adjusted columns."""
    from .scene import SceneRNG
    from .experiments import METHODS
    if not isinstance(data, Dataset):
        data = load_dataset(data)
    out = {m: np.zeros((len(triplets_to_test), 6 if bundle_adjust else 3)) for m in methods}

    def errors(R2, R3, CalM, inl, R_t0):
        Ps = [CalM[0:3] @ np.eye(3, 4), CalM[3:6] @ R2, CalM[6:9] @ R3]
        rep = api.ReprError(Ps, inl, device=device)                                                     # :130-131
        r2, t2 = api.AngError(R_t0[0], R2, device=device)
        r3, t3 = api.AngError(R_t0[1], R3, device=device)
        return [rep, (r2 + r3) / 2, (t2 + t3) / 2]                                                      # :133-136

    for row, trip in enumerate(triplets_to_test):
        it = row + 1                                                                                    # :75 loop index
        d = prepare_triplet(data, trip, device=device)
        inl = d["Corresp_inliers"]
        N = inl.shape[1]
        sample = SceneRNG(it).randsample(N, min(initial_sample_size, N))                               # :103-105
        C0 = inl[:, sample]
        CalM = d["CalM"]
        rec = dict(triplet=d["triplet"], n_inliers=N, REr=d["REr"], sample=sample, res={})
        if bundle_adjust:
            rec["ba"] = {}
        if raw_matches:
            rec["consensus"] = {}
        Nm = d["Corresp"].shape[1] if raw_matches else N
        for m in methods:
            if (m > 6 and Nm < 8) or Nm < 7:                                                            # :117-122
                out[m][row] = np.inf
                continue
            if raw_matches:
                res = api.ransac_pose(d["Corresp"], CalM, method=m, hypotheses=1024, threshold=1.0, seed=it, device=device)
                Cm, X0 = d["Corresp"][:, res[2]], None
                rec["consensus"][m] = consensus_stats(res[2], d["inlier_mask"])
            else:
                res = METHODS[m][1](C0, CalM, device=device)                                            # :126
                Cm, X0 = C0, res[2]
            out[m][row, :3] = errors(res[0], res[1], CalM, inl, d["R_t0"])
            rec["res"][m] = res
            if bundle_adjust and Cm.shape[1] < 4:                                                       # too few to adjust
                out[m][row, 3:] = np.inf
            elif bundle_adjust:
                ba = api.bundle_adjust(Cm, CalM, res[0], res[1], X0, device=device)
                out[m][row, 3:] = errors(ba[0], ba[1], CalM, inl, d["R_t0"])
                if covariance:
                    cov = api.ba_covariance(Cm, CalM, ba[0], ba[1], ba[2], device=device)
                    rot, tdir = api.pose_rms_errors(cov[0], ba[0], ba[1], sigma2=cov[1])
                    ba.sigma2 = cov[1]
                    ba.pred_rot_err, ba.pred_t_err = float(np.mean(rot)), float(np.mean(tdir))
                rec["ba"][m] = ba
        if details is not None:
            details.append(rec)
    return out
