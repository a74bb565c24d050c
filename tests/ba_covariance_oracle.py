"""CPU oracle of the bundle adjustment's covariance (tvf_ba_covariance).  TEST INFRASTRUCTURE ONLY.

Built on oracle/bundle_adjust.py's model and Jacobian, by a route independent of the kernel's: the dense Jacobian of
`Chart.jacobian` at p = 0 (the chart at the gauge-normalised state, with the oracle's own tangent basis `onb`), the
dense inverse of H = J'J with NumPy (after a symmetric diagonal scaling, which changes nothing but the rounding), and
the camera and point blocks read off it.  No Schur complement, and a different basis of t2's tangent plane.
"""
import numpy as np

from oracle import bundle_adjust as oba


def dense_inverse(Corresp, CalM, R_t_2, R_t_3, Reconst, U=None):
    """(inv(J'J), J, r, U) in the local chart at the gauge-normalised state; U: the tangent basis of t2 (default: the
    oracle's onb)."""
    Ks = [CalM[0:3], CalM[3:6], CalM[6:9]]
    R2, t2, R3, t3, X = oba.normalise_gauge(R_t_2[:, :3], R_t_2[:, 3], R_t_3[:, :3], R_t_3[:, 3],
                                            np.asarray(Reconst, float))
    ch = oba.Chart(R2, t2, R3, t3, X, U=U)
    J = ch.jacobian(Ks, np.zeros(11 + 3 * X.shape[1]), Corresp).toarray()
    r = oba.residuals(Ks, R2, t2, R3, t3, X, Corresp)
    H = J.T @ J
    d = 1.0 / np.sqrt(np.diag(H))
    Hi = d[:, None] * np.linalg.inv(d[:, None] * H * d[None, :]) * d[None, :]
    return 0.5 * (Hi + Hi.T), J, r, ch.U


def expansion(U):
    """G = blkdiag(I3, U, I3, I3) (12 x 11)."""
    G = np.zeros((12, 11))
    G[0:3, 0:3] = np.eye(3); G[3:6, 3:5] = U; G[6:9, 5:8] = np.eye(3); G[9:12, 8:11] = np.eye(3)
    return G


def covariance(Corresp, CalM, R_t_2, R_t_3, Reconst):
    """(cov_cam 12 x 12 over [w2, dt2 (ambient), w3, dt3], cov_pts (n, 3, 3), sigma2) at the state, unit pixel noise,
    as tvf_ba_covariance defines them."""
    Hi, J, r, U = dense_inverse(Corresp, CalM, R_t_2, R_t_3, Reconst)
    n = Corresp.shape[1]
    G = expansion(U)
    cov_cam = G @ Hi[:11, :11] @ G.T
    cov_pts = np.stack([Hi[11 + 3 * i:14 + 3 * i, 11 + 3 * i:14 + 3 * i] for i in range(n)])
    return cov_cam, cov_pts, float(r @ r) / (3 * n - 11)


def chart_coordinates(R_t_2, R_t_3, ref2, ref3):
    """[w2, dt2, w3, dt3] of the pose (R_t_2, R_t_3) relative to (ref2, ref3), both with |t2| = 1 (the coordinates
    cov_cam is stated in, to first order): R = exp([w]x) R_ref, dt = t - t_ref."""
    from scipy.spatial.transform import Rotation
    w = lambda R, Rr: Rotation.from_matrix(R @ Rr.T).as_rotvec()
    return np.concatenate([w(R_t_2[:, :3], ref2[:, :3]), R_t_2[:, 3] - ref2[:, 3],
                           w(R_t_3[:, :3], ref3[:, :3]), R_t_3[:, 3] - ref3[:, 3]])
