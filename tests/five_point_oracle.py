"""CPU oracle of the calibrated five-point minimal pose (tvf_five_point_pose, RANSAC method 9), by routes independent of
the device's: the essential matrices from Stewénius' 10 x 10 action matrix and numpy.linalg.eig (the device: Nistér's
degree-10 polynomial and Sturm sequences), P3P from Grunert's quartic and numpy.roots (the device: Lambda Twist).  The
selection rule is include/tvf.h's."""
import itertools

import numpy as np

import oracle as o
import ransac_oracle as ro

# grevlex: the ten cubics lead, then the basis of the quotient ring [x^2, xy, xz, y^2, yz, z^2, x, y, z, 1]
MONO = [(3, 0, 0), (2, 1, 0), (2, 0, 1), (1, 2, 0), (1, 1, 1), (1, 0, 2), (0, 3, 0), (0, 2, 1), (0, 1, 2), (0, 0, 3),
        (2, 0, 0), (1, 1, 0), (1, 0, 1), (0, 2, 0), (0, 1, 1), (0, 0, 2), (1, 0, 0), (0, 1, 0), (0, 0, 1), (0, 0, 0)]
IDX = {m: i for i, m in enumerate(MONO)}


def _pmul(a, b):
    out = {}
    for (ea, ca), (eb, cb) in itertools.product(a.items(), b.items()):
        e = tuple(x + y for x, y in zip(ea, eb))
        out[e] = out.get(e, 0.0) + ca * cb
    return out


def _padd(*ps, w=None):
    out = {}
    for k, p in enumerate(ps):
        for e, c in p.items():
            out[e] = out.get(e, 0.0) + (1.0 if w is None else w[k]) * c
    return out


def normalise_E(E):
    """unit Frobenius norm, the largest-magnitude entry (first in column-major order) positive"""
    E = E / np.linalg.norm(E)
    f = E.ravel(order="F")
    return E * np.sign(f[np.argmax(np.abs(f))])


def essentials(q1, q2, imag_tol=1e-8):
    """E (k, 3, 3) of the calibrated rays q1, q2 (3 x 5), ordered as found, and the real solutions' count"""
    A = np.stack([np.kron(q1[:, j], q2[:, j]) for j in range(5)])       # E(:) column-major: q2' E q1
    N = np.linalg.svd(A)[2][5:]                                         # X, Y, Z, W
    E = [[{(1, 0, 0): N[0][r + 3 * c], (0, 1, 0): N[1][r + 3 * c], (0, 0, 1): N[2][r + 3 * c],
           (0, 0, 0): N[3][r + 3 * c]} for c in range(3)] for r in range(3)]
    det = _padd(*[_pmul(E[0][c], _padd(_pmul(E[1][(c + 1) % 3], E[2][(c + 2) % 3]),
                                       _pmul(E[1][(c + 2) % 3], E[2][(c + 1) % 3]), w=[1, -1])) for c in range(3)])
    EEt = [[_padd(*[_pmul(E[r][k], E[s][k]) for k in range(3)]) for s in range(3)] for r in range(3)]
    tr = _padd(EEt[0][0], EEt[1][1], EEt[2][2])
    rows = [det]
    for r in range(3):
        for c in range(3):
            rows.append(_padd(_padd(*[_pmul(EEt[r][k], E[k][c]) for k in range(3)], w=[2, 2, 2]), _pmul(tr, E[r][c]),
                              w=[1, -1]))
    M = np.zeros((10, 20))
    for i, p in enumerate(rows):
        for e, c in p.items():
            M[i, IDX[e]] += c
    Cm = np.linalg.solve(M[:, :10], M[:, 10:])
    act = np.zeros((10, 10))                                            # x * basis = act @ basis (mod the ideal)
    for k, m in enumerate(MONO[10:]):
        xm = (m[0] + 1, m[1], m[2])
        i = IDX[xm]
        if i < 10:
            act[k] = -Cm[i]
        else:
            act[k, i - 10] = 1.0
    w, V = np.linalg.eig(act)
    out = []
    for j in range(10):
        v = V[:, j]
        if abs(w[j].imag) > imag_tol * max(1.0, abs(w[j])):
            continue
        v = (v / v[9]).real
        out.append(normalise_E((v[6] * N[0] + v[7] * N[1] + v[8] * N[2] + N[3]).reshape(3, 3, order="F")))
    return np.array(out).reshape(-1, 3, 3), len(out)


def p3p_grunert(X, y):
    """poses (R, t), x_cam = R X + t, of the points X (3 x 3, columns) seen along the unit rays y (3 x 3, columns),
    with positive depths: Grunert's quartic (Haralick et al. 1994) by numpy.roots"""
    a2 = np.sum((X[:, 1] - X[:, 2]) ** 2); b2 = np.sum((X[:, 0] - X[:, 2]) ** 2); c2 = np.sum((X[:, 0] - X[:, 1]) ** 2)
    ca, cb, cg = y[:, 1] @ y[:, 2], y[:, 0] @ y[:, 2], y[:, 0] @ y[:, 1]
    p, q = (a2 - c2) / b2, (a2 + c2) / b2
    A4 = (p - 1) ** 2 - 4 * c2 / b2 * ca ** 2
    A3 = 4 * (p * (1 - p) * cb - (1 - q) * ca * cg + 2 * c2 / b2 * ca ** 2 * cb)
    A2 = 2 * (p ** 2 - 1 + 2 * p ** 2 * cb ** 2 + 2 * (b2 - c2) / b2 * ca ** 2 - 4 * q * ca * cb * cg
              + 2 * (b2 - a2) / b2 * cg ** 2)
    A1 = 4 * (-p * (1 + p) * cb + 2 * a2 / b2 * cg ** 2 * cb - (1 - q) * ca * cg)
    A0 = (1 + p) ** 2 - 4 * a2 / b2 * cg ** 2
    out = []
    for v in np.roots([A4, A3, A2, A1, A0]):
        if abs(v.imag) > 1e-8 * max(1.0, abs(v)):
            continue
        v = v.real
        u = ((p - 1) * v ** 2 - 2 * p * cb * v + 1 + p) / (2 * (cg - v * ca))
        d = 1 + u * u - 2 * u * cg
        if not d > 0:
            continue
        s1 = np.sqrt(c2 / d)
        s = np.array([s1, u * s1, v * s1])
        if not np.all(s > 0):
            continue
        Y = y * s
        Xc, Yc = X - X.mean(1, keepdims=True), Y - Y.mean(1, keepdims=True)     # Kabsch
        U, _, Vt = np.linalg.svd(Yc @ Xc.T)
        R = U @ np.diag([1, 1, np.linalg.det(U @ Vt)]) @ Vt
        out.append((R, Y.mean(1) - R @ X.mean(1)))
    return out


def five_point_pose(Cr, CalM):
    """(Rt2, Rt3, E (k, 3, 3) in eig's order, n_E, status, ambiguity) of one sample Cr (6 x 5): include/tvf.h's
    rule.  ambiguity: the gap between the two smallest view-3 errors of the surviving pairs (inf with one pair)."""
    K = [CalM[3 * v:3 * v + 3] for v in range(3)]
    q = [np.linalg.solve(K[v], np.vstack([Cr[2 * v:2 * v + 2], np.ones(5)])) for v in range(3)]
    nan = np.full((3, 4), np.nan)
    if not np.all(np.isfinite(Cr)):
        return nan, nan, np.zeros((0, 3, 3)), 0, 4, np.inf
    Es, nE = essentials(q[0], q[1])
    P1 = K[0] @ np.eye(3, 4)
    cands, any2 = [], False
    for E in Es:
        U, _, Vt = np.linalg.svd(E)
        W = np.array([[0, -1, 0], [1, 0, 0], [0, 0, 1.0]])
        Ra, Rb = U @ W @ Vt, U @ W.T @ Vt
        Ra, Rb = Ra * np.sign(np.linalg.det(Ra)), Rb * np.sign(np.linalg.det(Rb))
        t = U[:, 2]
        for R, tt in ((Ra, t), (Ra, -t), (Rb, -t), (Rb, t)):
            Xh = o.triangulation3D([P1, K[1] @ np.column_stack([R, tt])], Cr[:4])
            X = Xh[:3] / Xh[3]
            if np.all(X[2] > 0) and np.all((R @ X + tt[:, None])[2] > 0):
                break
        else:
            continue
        any2 = True
        y = q[2][:, :3] / np.linalg.norm(q[2][:, :3], axis=0)
        for R3, t3 in p3p_grunert(X[:, :3], y):
            Xc = R3 @ X + t3[:, None]
            if not np.all(Xc[2] > 0):
                continue
            xp = K[2] @ Xc[:, 3:]
            err = np.max(np.hypot(*(xp[:2] / xp[2] - Cr[4:6, 3:])))
            cands.append((err, np.column_stack([R, tt]), np.column_stack([R3, t3])))
    if not any2:
        return nan, nan, Es, nE, 4, np.inf
    if not cands:
        return nan, nan, Es, nE, 8, np.inf
    errs = sorted(c[0] for c in cands)
    best = min(cands, key=lambda c: c[0])
    return best[1], best[2], Es, nE, 0, (errs[1] - errs[0]) if len(errs) > 1 else np.inf


def ransac(Cr, CalM, H, th, seed):
    """RANSAC method 9 (include/tvf.h) on the oracle's pieces: (Rt2, Rt3, inliers, n_inliers, sample, status)"""
    n = Cr.shape[1]
    idx = ro.sample(seed, np.arange(H), n, 5)
    best, bh = -2, -1
    for h in range(H):
        R2, R3, _, _, st, _ = five_point_pose(Cr[:, idx[h]], CalM)
        c = -1 if st else int(ro.inliers(Cr, CalM, R2, R3, th).sum())
        if c > best:
            best, bh, pose = c, h, (R2, R3)
    if best < 0:
        return np.full((3, 4), np.nan), np.full((3, 4), np.nan), np.zeros(n, bool), 0, np.full(5, -1), 128
    mask = ro.inliers(Cr, CalM, pose[0], pose[1], th)
    res = (pose[0], pose[1], mask, int(mask.sum()), idx[bh], 0)
    if mask.sum() >= 8:
        R2, R3, _, _, _ = o.LinearFPoseEstimation(Cr[:, mask], CalM)
        fm = ro.inliers(Cr, CalM, R2, R3, th)
        if fm.sum() >= mask.sum():
            res = (R2, R3, fm, int(fm.sum()), idx[bh], 0)
    return res
