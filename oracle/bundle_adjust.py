"""CPU oracle of the library's three-view bundle adjustment (tvf_bundle_adjust).  TEST INFRASTRUCTURE ONLY.

Objective: sum over views m = 1..3 and points i of |pi(K_m (R_m X_i + t_m)) - x_{m,i}|^2 in pixels, camera 1 fixed at
K1[I|0], scale gauge |t2| = 1.  Unknowns: R2, t2 on the unit sphere, R3, t3, X_i (11 + 3n degrees of freedom).

Its own route, independent of the kernel's: SciPy's MINPACK Levenberg-Marquardt ('lm') over ONE global chart around
the start, p = [w2 (3), a (2), w3 (3), dt3 (3), dX (3n)] with
    R2 = expm([w2]x) R2_0,   t2 = (t2_0 + U a) / |t2_0 + U a|,   R3 = expm([w3]x) R3_0,   t3 = t3_0 + dt3,   X = X_0 + dX,
rotation vectors through SciPy's Rotation, and the analytic Jacobian in that chart (left Jacobian of SO(3) and the
derivative of the sphere normalisation) assembled as a sparse matrix.  The kernel instead re-linearises at every
iterate in a local chart, solves the reduced camera system and damps with its own schedule; the two agree only
through the minimiser, which is what the tests compare.
"""
import numpy as np
import scipy.sparse as sp
from scipy.optimize import least_squares
from scipy.spatial.transform import Rotation


def skew(v):
    return np.array([[0.0, -v[2], v[1]], [v[2], 0.0, -v[0]], [-v[1], v[0], 0.0]])


def onb(t):
    """An orthonormal basis (3 x 2) of the plane orthogonal to the unit vector t (cross products with the axis of
    t's smallest component)."""
    a = np.eye(3)[np.argmin(np.abs(t))]
    u = np.cross(t, a); u /= np.linalg.norm(u)
    return np.stack([u, np.cross(t, u)], 1)


def left_jacobian(w):
    """J_l(w) with d(expm([w]x) v)/dw = -[expm([w]x) v]x J_l(w)."""
    th = np.linalg.norm(w)
    W = skew(w)
    if th < 1e-6:
        return np.eye(3) + 0.5 * W + W @ W / 6.0
    return np.eye(3) + (1.0 - np.cos(th)) / th ** 2 * W + (th - np.sin(th)) / th ** 3 * (W @ W)


def residuals(Ks, R2, t2, R3, t3, X, C):
    """6n residuals, point-major: (view 1 x, y, view 2 x, y, view 3 x, y) of point 0, then point 1, ..."""
    out = []
    for m, (R, t) in enumerate(((np.eye(3), np.zeros(3)), (R2, t2), (R3, t3))):
        h = Ks[m] @ (R @ X + t[:, None])
        out.append(h[:2] / h[2] - C[2 * m:2 * m + 2])
    return np.stack(out, 0).transpose(2, 0, 1).reshape(-1)


def repr_error(Ks, R2, t2, R3, t3, X, C):
    """ReprError.m:65: sqrt(sum of squares / (3 n))."""
    r = residuals(Ks, R2, t2, R3, t3, X, C)
    return float(np.sqrt(np.sum(r * r) / (3 * X.shape[1])))


class Chart:
    """The global chart p -> (R2, t2, R3, t3, X) around a start state."""

    def __init__(self, R2, t2, R3, t3, X, U=None):
        self.R2, self.t2, self.R3, self.t3, self.X = R2, t2, R3, t3, X
        self.U = onb(t2) if U is None else U
        self.n = X.shape[1]

    def unpack(self, p):
        s = self.t2 + self.U @ p[3:5]
        return (Rotation.from_rotvec(p[0:3]).as_matrix() @ self.R2, s / np.linalg.norm(s),
                Rotation.from_rotvec(p[5:8]).as_matrix() @ self.R3, self.t3 + p[8:11],
                self.X + p[11:].reshape(self.n, 3).T)

    def jacobian(self, Ks, p, C):
        """Analytic d residuals / dp (6n x (11 + 3n)), sparse."""
        R2, t2, R3, t3, X = self.unpack(p)
        n = self.n
        s = self.t2 + self.U @ p[3:5]
        ns = np.linalg.norm(s)
        dt2 = (np.eye(3) - np.outer(t2, t2)) @ self.U / ns                   # d t2 / d a
        Jl2, Jl3 = left_jacobian(p[0:3]), left_jacobian(p[5:8])
        rows, cols, vals = [], [], []
        for i in range(n):
            for m, (R, t) in enumerate(((np.eye(3), np.zeros(3)), (R2, t2), (R3, t3))):
                v = R @ X[:, i]
                h = Ks[m] @ (v + t)
                q = h[:2] / h[2]
                A = (Ks[m][:2] - np.outer(q, Ks[m][2])) / h[2]                   # d pixel / d camera coordinates
                blocks = [(11 + 3 * i, A @ R)]
                if m == 1:
                    blocks += [(0, -A @ skew(v) @ Jl2), (3, A @ dt2)]
                elif m == 2:
                    blocks += [(5, -A @ skew(v) @ Jl3), (8, A)]
                for c0, blk in blocks:
                    for a in range(2):
                        for b in range(blk.shape[1]):
                            rows.append(6 * i + 2 * m + a); cols.append(c0 + b); vals.append(blk[a, b])
        return sp.csr_matrix((vals, (rows, cols)), shape=(6 * n, 11 + 3 * n))


def normalise_gauge(R2, t2, R3, t3, X):
    """Scale t2, t3 and the points by 1/|t2| (the reprojection is unchanged)."""
    s = 1.0 / np.linalg.norm(t2)
    return R2, t2 * s, R3, t3 * s, X * s


def bundle_adjust(Corresp, CalM, R_t_2, R_t_3, Reconst):
    """Minimiser of the pixel reprojection error from the given start.  Returns (R_t_2, R_t_3, Reconst, repr_err)."""
    Ks = [CalM[0:3], CalM[3:6], CalM[6:9]]
    R2, t2, R3, t3, X = normalise_gauge(R_t_2[:, :3], R_t_2[:, 3], R_t_3[:, :3], R_t_3[:, 3], np.asarray(Reconst, float))
    ch = Chart(R2, t2, R3, t3, X)
    f = lambda p: residuals(Ks, *ch.unpack(p), Corresp)
    jac = lambda p: ch.jacobian(Ks, p, Corresp).toarray()
    s = least_squares(f, np.zeros(11 + 3 * X.shape[1]), jac=jac, method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15,
                      max_nfev=20000)
    R2, t2, R3, t3, X = ch.unpack(s.x)
    return np.column_stack([R2, t2]), np.column_stack([R3, t3]), X, repr_error(Ks, R2, t2, R3, t3, X, Corresp)


def gradient(Corresp, CalM, R_t_2, R_t_3, Reconst):
    """Gradient J'r of (1/2) sum r^2 in the local chart at the given state (after gauge normalisation)."""
    Ks = [CalM[0:3], CalM[3:6], CalM[6:9]]
    R2, t2, R3, t3, X = normalise_gauge(R_t_2[:, :3], R_t_2[:, 3], R_t_3[:, :3], R_t_3[:, 3], np.asarray(Reconst, float))
    ch = Chart(R2, t2, R3, t3, X)
    p = np.zeros(11 + 3 * X.shape[1])
    return ch.jacobian(Ks, p, Corresp).T @ residuals(Ks, R2, t2, R3, t3, X, Corresp)


def gradient_batch(Corresp, CalM, R_t_2, R_t_3, Reconst):
    """gradient() for a batch, vectorised: Corresp (B,6,n), CalM (9,3) or (B,9,3), poses (B,3,4), Reconst (B,3,n) ->
    (B, 11 + 3n) in the same unknowns (the oracle's own tangent basis of t2, points point-major)."""
    Corresp = np.asarray(Corresp, float); Reconst = np.asarray(Reconst, float)
    B, _, n = Corresp.shape
    CalM = np.broadcast_to(np.asarray(CalM, float), (B, 9, 3))
    s = 1.0 / np.linalg.norm(R_t_2[:, :, 3], axis=1)
    poses = [(np.broadcast_to(np.eye(3), (B, 3, 3)), np.zeros((B, 3))),
             (R_t_2[:, :, :3], R_t_2[:, :, 3] * s[:, None]), (R_t_3[:, :, :3], R_t_3[:, :, 3] * s[:, None])]
    X = Reconst * s[:, None, None]
    U = np.stack([onb(t) for t in poses[1][1]])                                   # (B,3,2)
    g = np.zeros((B, 11 + 3 * n)); gX = np.zeros((B, n, 3))
    for m, (R, t) in enumerate(poses):
        K = CalM[:, 3 * m:3 * m + 3]
        v = np.einsum("bij,bjn->bni", R, X)                                       # (B,n,3) camera frame, before t
        h = np.einsum("bij,bnj->bni", K, v + t[:, None, :])
        q = h[..., :2] / h[..., 2:3]
        r = q - Corresp[:, 2 * m:2 * m + 2].transpose(0, 2, 1)                    # (B,n,2)
        A = (K[:, None, :2, :] - q[..., :, None] * K[:, None, 2:3, :]) / h[..., 2, None, None]   # (B,n,2,3)
        a = np.einsum("bnk,bnkj->bnj", r, A)                                      # r'A per point (B,n,3)
        gX += np.einsum("bnj,bji->bni", a, R)
        if m == 1:
            g[:, 0:3] = np.cross(v, a).sum(1)
            g[:, 3:5] = np.einsum("bj,bjk->bk", a.sum(1), U)
        elif m == 2:
            g[:, 5:8] = np.cross(v, a).sum(1)
            g[:, 8:11] = a.sum(1)
    g[:, 11:] = gX.reshape(B, -1)
    return g
