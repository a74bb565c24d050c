"""Scenes whose three views have different intrinsics (TEST INFRASTRUCTURE).

Every calibrated entry point takes CalM = [K1; K2; K3], one 9 x 3 for the batch or one per problem.  The sweep scenes,
the golden files and the EPFL cameras all have K1 = K2 = K3 and one K for every problem, so an index slip that reads
the wrong view's K, or the wrong problem's, changes nothing there.  These scenes draw K1, K2, K3 per problem from a
seeded family around the sweep's K and reproject the sweep's points with them, so the ground truth is known exactly."""
import numpy as np

import oracle as o
from tft_vs_fund_b200 import scene as pscene

IMAGE_W, IMAGE_H = 36 * pscene.PIX, 24 * pscene.PIX        # the sweep's 1800 x 1200 image


def draw_ks(rs, K):
    """K1, K2, K3 around K: focal x 0.7 .. 1.4, fy / fx 0.98 .. 1.03, principal point +-60 px, skew 0 or up to 0.5,
    K[2,2] = 1.  The three focal lengths differ pairwise by at least 0.15 f, so no two views share a K."""
    f = K[0, 0]
    while True:
        scale = rs.uniform(0.7, 1.4, 3)
        if np.min(np.abs(scale[:, None] - scale[None, :]) + np.eye(3)) >= 0.15:
            break
    Ks = []
    for v in range(3):
        fx = f * scale[v]
        skew = 0.0 if rs.rand() < 0.5 else rs.uniform(-0.5, 0.5)
        Ks.append(np.array([[fx, skew, K[0, 2] + rs.uniform(-60.0, 60.0)],
                            [0.0, fx * rs.uniform(0.98, 1.03), K[1, 2] + rs.uniform(-60.0, 60.0)],
                            [0.0, 0.0, 1.0]]))
    return Ks


def scene(n, noise, seed):
    """(Corresp 6 x n, CalM 9 x 3 with three different K, R_t0 [Rt2, Rt3], points 3 x n in camera 1's frame): the
    noise-free sweep scene of experiments_subsample(n, 0, seed), its points triangulated with the true cameras, then
    reprojected with a K per view drawn from (seed, n), plus `noise` px of Gaussian noise."""
    CalM0, R_t0, Cr0, _ = o.experiments_subsample(n, 0.0, seed)
    K = CalM0[:3]
    Xh = o.triangulation3D([K @ np.eye(3, 4), K @ R_t0[0], K @ R_t0[1]], Cr0)
    X = Xh[:3] / Xh[3]
    rs = np.random.RandomState(1000 * seed + n)
    Ks = draw_ks(rs, K)
    Cr = o.project3Dpoints(X, [Ks[0] @ np.eye(3, 4), Ks[1] @ R_t0[0], Ks[2] @ R_t0[1]])
    Cr = Cr + noise * rs.standard_normal(Cr.shape)
    return Cr, np.vstack(Ks), [R_t0[0].copy(), R_t0[1].copy()], X


def batch(n, noise, seeds):
    """scene() for each seed, stacked: Corresp (B, 6, n), CalM (B, 9, 3), R_t0 (B, 2, 3, 4), points (B, 3, n).  `noise`
    is one level or one per seed."""
    noise = np.broadcast_to(np.asarray(noise, dtype=np.float64), (len(seeds),))
    parts = [scene(n, float(nz), int(s)) for nz, s in zip(noise, seeds)]
    return (np.stack([p[0] for p in parts]), np.stack([p[1] for p in parts]), np.stack([np.stack(p[2]) for p in parts]),
            np.stack([p[3] for p in parts]))


def gauge_truth(CalM, R_t0, X):
    """The true state with |t2| = 1, as the bundle adjustment and its covariance state it: (Rt2, Rt3, X)."""
    s = 1.0 / np.linalg.norm(R_t0[0][:, 3])
    return (np.column_stack([R_t0[0][:, :3], R_t0[0][:, 3] * s]), np.column_stack([R_t0[1][:, :3], R_t0[1][:, 3] * s]),
            X * s)


def outlier_scenes(f, count, seed, noise=1.0, n=100):
    """ransac_oracle.outlier_scenes with a K per view and per problem: `count` scenes of n matches (scene(n, noise,
    seed + b)) whose columns are replaced, a share f of them (one share, or one per scene) chosen at random, by uniform
    pixels of the 1800 x 1200 image in all three views.  Returns (Corresp (count, 6, n), CalM (count, 9, 3), R_t0 (count, 2, 3, 4), outlier mask
    (count, n))."""
    Cr, CalM, R_t0, _ = batch(n, noise, [seed + b for b in range(count)])
    rs = np.random.RandomState(seed)
    out = np.zeros((count, n), dtype=bool)
    for b, fb in enumerate(np.broadcast_to(np.asarray(f, dtype=np.float64), (count,))):
        cols = rs.choice(n, int(round(fb * n)), replace=False)
        out[b, cols] = True
        Cr[b][0::2, cols] = rs.uniform(0.0, IMAGE_W, size=(3, cols.size))
        Cr[b][1::2, cols] = rs.uniform(0.0, IMAGE_H, size=(3, cols.size))
    return Cr, CalM, R_t0, out


def wrong_k(CalM):
    """The calibrations an index slip would read instead of CalM (9 x 3, or B x 9 x 3): {name: CalM of the same shape}.
    'K2 and K3 swapped' and 'K1 for every view' always; 'problem 0 for every problem' for a batch."""
    CalM = np.asarray(CalM, dtype=np.float64)
    swapped = CalM.copy()
    swapped[..., 3:6, :], swapped[..., 6:9, :] = CalM[..., 6:9, :], CalM[..., 3:6, :]
    out = {"K2 and K3 swapped": swapped, "K1 for every view": np.concatenate([CalM[..., 0:3, :]] * 3, axis=-2)}
    if CalM.ndim == 3:
        out["problem 0 for every problem"] = np.broadcast_to(CalM[0], CalM.shape).copy()
    return out
