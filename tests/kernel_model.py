"""NumPy model of the GPU algorithms (TEST HELPER, not product code).

Mirrors, step for step, what the CUDA kernels in tft_vs_fund_b200/csrc do
(96 Kronecker moments -> 27x27 Gram -> Gauss-Jordan sweep inverse + power iteration ->
epipoles by QR + inverse iteration (Jacobi fallback) -> 15-dim projected Gram -> ... -> QR-based DLT),
so the numerical design (tolerances, iteration counts) can be validated
against the oracle on CPU before any GPU time is spent.
"""
import numpy as np

# ---- index tables shared with the CUDA side (csrc/tvf_tables.cuh) ----------
SYM6 = {(0, 0): 0, (0, 1): 1, (1, 0): 1, (0, 2): 2, (2, 0): 2, (1, 1): 3, (1, 2): 4, (2, 1): 4, (2, 2): 5}
# M(x,y) = S S^T = [1 0 -x; 0 1 -y; -x -y x^2+y^2]; features m4 = [1, -x, -y, r2]; -1 marks a structural zero
M4 = {(0, 0): 0, (1, 1): 0, (0, 1): -1, (1, 0): -1, (0, 2): 1, (2, 0): 1, (1, 2): 2, (2, 1): 2, (2, 2): 3}


def normalize_stats(p):
    c = p.mean(axis=1)
    d = np.sqrt(((p - c[:, None]) ** 2).sum(axis=0)).mean()
    s = np.sqrt(2.0) / d
    return c, s


def moments96(x1, x2, x3):
    """x* are normalised 2xn.  moment[a*16+b*4+g] = sum A6[a]*m4(view3)[b]*m4(view2)[g]."""
    n = x1.shape[1]
    A6 = np.stack([x1[0] ** 2, x1[0] * x1[1], x1[0], x1[1] ** 2, x1[1], np.ones(n)])
    m2 = np.stack([np.ones(n), -x2[0], -x2[1], x2[0] ** 2 + x2[1] ** 2])
    m3 = np.stack([np.ones(n), -x3[0], -x3[1], x3[0] ** 2 + x3[1] ** 2])
    mom = np.einsum('an,bn,gn->abg', A6, m3, m2).reshape(96)
    return mom


def gram27_from_moments(mom):
    G = np.zeros((27, 27))
    for r in range(27):
        j, k, i = r % 3, (r // 3) % 3, r // 9
        for c in range(27):
            j2, k2, i2 = c % 3, (c // 3) % 3, c // 9
            g = M4[(j, j2)]; b = M4[(k, k2)]
            if g < 0 or b < 0:
                continue
            G[r, c] = mom[SYM6[(i, i2)] * 16 + b * 4 + g]
    return G


def smallest_eigvec_spd(G, max_iter=80, tol=4e-15):
    """What tvf_warp.cuh::smallest_eigvec_spd does: scale to unit trace, relative diagonal shift 1e-13,
    N Gauss-Jordan sweeps in place (pivot row updated through c_k = d - 1), then power iteration with
    the (negated) inverse."""
    N = G.shape[0]
    A = G / np.trace(G)
    delta = 1e-13 / N
    A = A + delta * np.eye(N)
    floor = 1e-3 * delta
    for k in range(N):
        col = A[:, k].copy()
        d = max(col[k], floor)
        piv = 1.0 / d
        rk = col * piv
        c = col.copy(); c[k] -= 1.0
        newA = A - np.outer(c, rk)
        newA[:, k] = rk; newA[k, k] = -piv
        A = newA
    # pivot-normalised power iteration (tvf_warp.cuh::smallest_eigvec_spd): the iterate is scaled so that its largest component is 1
    # (dividing by the signed pivot also absorbs the sign of -M); one exact 2-norm normalisation at the end
    # start: M (e_0 + e_{N/2} + e_{N-1}), the sum of three columns of the inverse (tvf_warp.cuh::smallest_eigvec_spd_half):
    # a free first application
    x = A[:, 0] + A[:, N // 2] + A[:, N - 1]
    its = 0
    for its in range(1, max_iter + 1):
        z = A @ x
        z = z / z[np.argmax(np.abs(z))]
        d = np.max(np.abs(z - x))
        x = z
        if not d > tol:
            break
    x = x / np.linalg.norm(x)
    return x, its


def jacobi_svd_V(A, sweeps=12):
    """One-sided (Hestenes) Jacobi: returns (V, column norms) with columns sorted by
    descending norm; A is m x k, small."""
    A = np.array(A, dtype=np.float64)
    m, k = A.shape
    V = np.eye(k)
    for _ in range(sweeps):
        rotated = False
        for p in range(k - 1):
            for q in range(p + 1, k):
                alpha = A[:, p] @ A[:, p]; beta = A[:, q] @ A[:, q]; gamma = A[:, p] @ A[:, q]
                if abs(gamma) <= 1e-300 or abs(gamma) <= 2.2e-16 * np.sqrt(alpha * beta):
                    continue
                rotated = True
                zeta = (beta - alpha) / (2.0 * gamma)
                t = np.sign(zeta) / (abs(zeta) + np.sqrt(1.0 + zeta * zeta)) if zeta != 0 else 1.0
                c = 1.0 / np.sqrt(1.0 + t * t); s = c * t
                Ap = A[:, p].copy(); Aq = A[:, q].copy()
                A[:, p] = c * Ap - s * Aq; A[:, q] = s * Ap + c * Aq
                Vp = V[:, p].copy(); Vq = V[:, q].copy()
                V[:, p] = c * Vp - s * Vq; V[:, q] = s * Vp + c * Vq
        if not rotated:
            break
    nrm = np.sqrt((A * A).sum(axis=0))
    order = np.argsort(-nrm, kind='stable')
    return V[:, order], nrm[order], A[:, order]


def null3_qr(Mx, max_iter=12):
    """tvf_math.cuh::null3_qr: Householder QR of the 3x3 + inverse iteration with R (rate (s3/s2)^2); None when it has not
    converged in max_iter steps or the input is not finite -- null3 then takes the Jacobi route, as the kernels do."""
    Mx = np.asarray(Mx, dtype=np.float64)
    if not np.all(np.isfinite(Mx)):
        return None
    R = np.linalg.qr(Mx, mode='r')
    rmax = np.max(np.abs(np.diag(R)))
    if not rmax > 0.0:
        return None
    tiny = 1e-300 + 1e-18 * rmax
    for k in range(3):
        if abs(R[k, k]) < tiny:
            R[k, k] = np.copysign(tiny, R[k, k]) if R[k, k] != 0 else tiny
    x = np.linalg.solve(R, np.array([0.0, 0.0, 1.0]))
    x /= np.linalg.norm(x)
    dprev = 0.0
    for _ in range(max_iter):
        z = np.linalg.solve(R, np.linalg.solve(R.T, x))
        z /= np.linalg.norm(z)
        d2 = float(np.sum((z - x) ** 2)); x = z
        if not d2 > 1e-26 or not d2 * d2 > 1e-28 * dprev:
            return x
        dprev = d2
    return None


def null3(Mx):
    v = null3_qr(Mx)
    if v is not None:
        return v
    V, _, _ = jacobi_svd_V(Mx)
    return V[:, 2]


def epipoles(T):
    """T 3x3x3 -> (e21, e31) unsigned (linearTFT.m:71-79)."""
    v = [null3(T[:, :, i]) for i in range(3)]
    e31 = null3(np.stack(v))
    v = [null3(T[:, :, i].T) for i in range(3)]
    e21 = null3(np.stack(v))
    return e21, e31


def onb(e):
    """Duff et al. branchless orthonormal basis: returns u1, u2 with {e,u1,u2} orthonormal."""
    sgn = 1.0 if e[2] >= 0 else -1.0
    a = -1.0 / (sgn + e[2]); b = e[0] * e[1] * a
    u1 = np.array([1.0 + sgn * e[0] * e[0] * a, sgn * b, -sgn * e[0]])
    u2 = np.array([b, sgn + e[1] * e[1] * a, -e[1]])
    return u1, u2


def constrained_tft(G, e21, e31):
    """linearTFT.m:82-86 without svd(E): orthonormal basis of range(E), projected Gram."""
    u1, u2 = onb(e21); v1, v2 = onb(e31)
    Bs = [np.outer(e21, e31), np.outer(e21, v1), np.outer(e21, v2), np.outer(u1, e31), np.outer(u2, e31)]
    Up = np.zeros((27, 15))
    for i in range(3):
        for a, B in enumerate(Bs):
            Up[9 * i:9 * i + 9, 5 * i + a] = B.reshape(9, order='F')   # index j+3k
    G15 = Up.T @ G @ Up
    tp, its = smallest_eigvec_spd(G15)
    t = Up @ tp
    t /= np.linalg.norm(t)
    T = t.reshape(3, 3, 3, order='F')
    # minimum-norm a = pinv(E) t  (closed form, DESIGN.md)
    A = np.zeros((3, 3)); Bm = np.zeros((3, 3))
    for i in range(3):
        Ti = T[:, :, i]
        tau = e21 @ Ti @ e31
        A[:, i] = Ti @ e31 - 0.5 * tau * e21
        Bm[:, i] = 0.5 * tau * e31 - Ti.T @ e21
    P2 = np.column_stack([A, e21]); P3 = np.column_stack([Bm, e31])
    return T, P2, P3, its


def dlt_null(rows, max_iter=40, tol=1e-15):
    """Smallest right singular vector of rows (m x 4) via Householder QR + inverse iteration on R."""
    R = np.linalg.qr(np.asarray(rows, dtype=np.float64), mode='r')
    scale = np.max(np.abs(np.diag(R)))
    for d in range(4):
        if abs(R[d, d]) < 1e-300 + 1e-18 * scale:
            R[d, d] = 1e-18 * scale if scale > 0 else 1e-300
    x = np.linalg.solve(R, np.array([0, 0, 0, 1.0]))
    x /= np.linalg.norm(x)
    its = 0
    dprev = 0.0
    for its in range(1, max_iter + 1):
        y = np.linalg.solve(R.T, x)
        z = np.linalg.solve(R, y)
        z /= np.linalg.norm(z)
        if z @ x < 0:
            z = -z
        d2 = float(np.sum((z - x) ** 2)); x = z
        # tvf_math.cuh::dlt_null: stop on a change below 1e-13, or as soon as the error LEFT,
        # |z - x| * rate with rate ~ |z - x| / |previous change|, is below 1e-14
        if not d2 > 1e-26 or not d2 * d2 > 1e-28 * dprev:
            break
        dprev = d2
    return x, its


def dlt_rows(Ps, pts):
    rows = []
    for P, (x, y) in zip(Ps, pts):
        rows.append(-P[1] + y * P[2])
        rows.append(P[0] - x * P[2])
    return np.array(rows)


# ---------------------------------------------------------------------------
# pose tail (model of the thread-per-problem / thread-per-point kernels)
# ---------------------------------------------------------------------------
def inv3(M):
    return np.linalg.inv(M)


def transform_inverse(T, M1, M2, M3):
    M2i = inv3(M2); M3i = inv3(M3)
    Tn = np.zeros((3, 3, 3))
    for i in range(3):
        Tn[:, :, i] = M2i @ (M1[0, i] * T[:, :, 0] + M1[1, i] * T[:, :, 1] + M1[2, i] * T[:, :, 2]) @ M3i.T
    return Tn / np.linalg.norm(Tn.ravel())


def svd3_full(E):
    """Full SVD of a 3x3 by one-sided Jacobi: U, s, V with u3 = u1 x u2 (E is ~rank 2)."""
    V, s, AV = jacobi_svd_V(E)
    u1 = AV[:, 0] / s[0]; u2 = AV[:, 1] / s[1]
    u3 = np.cross(u1, u2)
    return np.column_stack([u1, u2, u3]), s, V


def decompose_E(E):
    U, s, V = svd3_full(E)
    W = np.array([[0.0, -1, 0], [1, 0, 0], [0, 0, 1]])
    R = U @ W @ V.T; Rp = U @ W.T @ V.T
    R = R * np.sign(np.linalg.det(R)); Rp = Rp * np.sign(np.linalg.det(Rp))
    return R, Rp, U[:, 2].copy()


def depth_signs_ray(A, r3, tz):
    """tvf_math.cuh::dlt4_depth_signs_ray: the two depth signs of the DLT solution of the 4x4 system A from the 4-D cross
    product Xt of its first three rows (ray of view 1 meets a plane of view 2), certified by
    sin(angle(Xt, v)) <= eta = |A[3].Xt| |B|_F^2 / (2 |Xt|^2)  (B = A[:3]); None when the certificate declines."""
    B = A[:3]
    Xt = np.array([np.linalg.det(B[:, [1, 2, 3]]), -np.linalg.det(B[:, [0, 2, 3]]),
                   np.linalg.det(B[:, [0, 1, 3]]), -np.linalg.det(B[:, [0, 1, 2]])])
    xx = Xt @ Xt; b2 = float(np.sum(B * B)); rb2 = abs(A[3] @ Xt) * b2
    if not rb2 < 0.4 * xx or not xx >= 1e-12 * b2 ** 3:
        return None
    q1 = Xt[2] * Xt[3]; q2 = (r3 @ Xt[:3] + tz * Xt[3]) * Xt[3]
    if not abs(q1) >= 1.0605 * rb2 + 1e-6 * xx or not abs(q2) >= 1.616 * rb2 + 1e-6 * xx:
        return None
    return (1 if q1 > 0 else -1), (1 if q2 > 0 else -1)


def cheirality(R, Rp, t, P1, K2, x1, x2):
    cands = [(R, t), (R, -t), (Rp, -t), (Rp, t)]
    best = 0; sel = None; votes = []
    for (Rc, tc) in cands:
        P2 = K2 @ np.column_stack([Rc, tc])
        v = 0
        for n in range(x1.shape[1]):
            A = dlt_rows([P1, P2], [x1[:, n], x2[:, n]])
            sg = depth_signs_ray(A, Rc[2], tc[2])         # certified shortcut first, as in the kernels
            if sg is not None:
                v += sg[0] + sg[1]
                continue
            X, _ = dlt_null(A)
            X = X / X[3]
            z2 = Rc[2] @ X[:3] + tc[2]
            v += np.sign(X[2]) + np.sign(z2)
        votes.append(v)
        if v >= best:
            best = v; sel = (Rc, tc)
    return sel, votes


def pose_tail(E21, E31, CalM, C):
    K1, K2, K3 = CalM[0:3], CalM[3:6], CalM[6:9]
    P1 = K1 @ np.eye(3, 4)
    (R2, t2), v2 = cheirality(*decompose_E(E21), P1, K2, C[0:2], C[2:4])
    (R3, t3), v3 = cheirality(*decompose_E(E31), P1, K3, C[0:2], C[4:6])
    P2 = K2 @ np.column_stack([R2, t2])
    u3 = K3 @ t3; KR3 = K3 @ R3
    num = 0.0; den = 0.0
    for n in range(C.shape[1]):
        X, _ = dlt_null(dlt_rows([P1, P2], [C[0:2, n], C[2:4, n]]))
        X = X[:3] / X[3]
        p3 = np.array([C[4, n], C[5, n], 1.0])
        c1 = np.cross(p3, KR3 @ X); c2 = np.cross(p3, u3)
        num += c1 @ c2; den += c2 @ c2
    t3 = -num / den * t3
    Rt2 = np.column_stack([R2, t2]); Rt3 = np.column_stack([R3, t3])
    P3 = K3 @ Rt3
    Rec = np.zeros((3, C.shape[1])); sq = 0.0
    for n in range(C.shape[1]):
        X, _ = dlt_null(dlt_rows([P1, P2, P3], [C[0:2, n], C[2:4, n], C[4:6, n]]))
        X = X[:3] / X[3]; Rec[:, n] = X
        for v, P in enumerate((P1, P2, P3)):
            x = P @ np.append(X, 1.0)
            sq += (x[0] / x[2] - C[2 * v, n]) ** 2 + (x[1] / x[2] - C[2 * v + 1, n]) ** 2
    return Rt2, Rt3, Rec, np.sqrt(sq / (3 * C.shape[1])), v2, v3


def tft_pose_model(C, CalM):
    cs = [normalize_stats(C[2 * v:2 * v + 2]) for v in range(3)]
    xs = [s * (C[2 * v:2 * v + 2] - c[:, None]) for v, (c, s) in enumerate(cs)]
    Ns = [np.array([[s, 0, -s * c[0]], [0, s, -s * c[1]], [0, 0, 1.0]]) for (c, s) in cs]
    G = gram27_from_moments(moments96(*xs))
    t, _ = smallest_eigvec_spd(G)
    e21, e31 = epipoles(t.reshape(3, 3, 3, order='F'))
    Tn, _, _, _ = constrained_tft(G, e21, e31)
    T = transform_inverse(Tn, *Ns)
    K1, K2, K3 = CalM[0:3], CalM[3:6], CalM[6:9]
    Tc = transform_inverse(T, K1, K2, K3)
    e21, e31 = epipoles(Tc)
    e21 = e21 * np.sign(e21[2]); e31 = e31 * np.sign(e31[2])
    cx = lambda v: np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])
    E21 = cx(e21) @ np.column_stack([Tc[:, :, i] @ e31 for i in range(3)])
    E31 = -cx(e31) @ np.column_stack([Tc[:, :, i].T @ e21 for i in range(3)])
    return (T,) + pose_tail(E21, E31, CalM, C)


def moments36(x1, x2):
    n = x1.shape[1]
    A6 = np.stack([x1[0] ** 2, x1[0] * x1[1], x1[0], x1[1] ** 2, x1[1], np.ones(n)])
    B6 = np.stack([x2[0] ** 2, x2[0] * x2[1], x2[0], x2[1] ** 2, x2[1], np.ones(n)])
    return np.einsum('an,bn->ab', A6, B6).reshape(36)


def gram9_from_moments(mom):
    G = np.zeros((9, 9))
    for r in range(9):
        a, b = r // 3, r % 3          # column index of linearF.m:51-52: 3*(x1-index)+(x2-index)
        for c in range(9):
            a2, b2 = c // 3, c % 3
            G[r, c] = mom[SYM6[(a, a2)] * 6 + SYM6[(b, b2)]]
    return G


def linearF_model(p1, p2):
    c1, s1 = normalize_stats(p1); c2, s2 = normalize_stats(p2)
    x1 = s1 * (p1 - c1[:, None]); x2 = s2 * (p2 - c2[:, None])
    N1 = np.array([[s1, 0, -s1 * c1[0]], [0, s1, -s1 * c1[1]], [0, 0, 1.0]])
    N2 = np.array([[s2, 0, -s2 * c2[0]], [0, s2, -s2 * c2[1]], [0, 0, 1.0]])
    f, _ = smallest_eigvec_spd(gram9_from_moments(moments36(x1, x2)))
    F = f.reshape(3, 3, order='F')
    F = N2.T @ F @ N1
    U, s, V = svd3_full(F)      # rank-2 projection: drop sigma3 (u3 unused)
    return s[0] * np.outer(U[:, 0], V[:, 0]) + s[1] * np.outer(U[:, 1], V[:, 1])


def f_pose_model(C, CalM):
    cs = [normalize_stats(C[2 * v:2 * v + 2]) for v in range(3)]
    xs = [s * (C[2 * v:2 * v + 2] - c[:, None]) for v, (c, s) in enumerate(cs)]
    Ns = [np.array([[s, 0, -s * c[0]], [0, s, -s * c[1]], [0, 0, 1.0]]) for (c, s) in cs]
    F21 = Ns[1].T @ linearF_model(xs[0], xs[1]) @ Ns[0]
    F31 = Ns[2].T @ linearF_model(xs[0], xs[2]) @ Ns[0]
    K1, K2, K3 = CalM[0:3], CalM[3:6], CalM[6:9]
    return (F21, F31) + pose_tail(K2.T @ F21 @ K1, K3.T @ F31 @ K1, CalM, C)
