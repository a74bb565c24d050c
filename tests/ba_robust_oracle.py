"""CPU oracle of the robust-loss bundle adjustment (tvf_bundle_adjust_robust).  TEST INFRASTRUCTURE ONLY.

Objective: sum_i c^2 rho(s_i / c^2), s_i the six squared pixel residuals of match i, with SciPy least_squares' rho
(huber, soft_l1, cauchy), on the model of oracle/bundle_adjust.py (camera 1 = K1[I|0], |t2| = 1).

It reuses that oracle's global chart and analytic Jacobian but takes its own route to the minimiser: MINPACK 'lm' on
the rescaled residuals r~_i = f(s_i) r_i, f(s) = sqrt(c^2 rho(s / c^2) / s) (f(0) = 1), whose squared norm is exactly the
robust cost, with the Jacobian of r~ by the chain rule on the existing one.  The kernel instead re-weights a Gauss-Newton
model at every linearisation (IRLS); the two agree only through the stationary points, which is what the tests compare.
"""
import numpy as np
from scipy.optimize import least_squares

from oracle import bundle_adjust as oba

LOSSES = ("huber", "soft_l1", "cauchy")


def rho(loss, z):
    """SciPy least_squares' rho(z) (rho[0] of its loss functions), elementwise."""
    z = np.asarray(z, dtype=np.float64)
    if loss == "huber":
        return np.where(z <= 1.0, z, 2.0 * np.sqrt(np.maximum(z, 1.0)) - 1.0)
    if loss == "soft_l1":
        return 2.0 * (np.sqrt(1.0 + z) - 1.0)
    if loss == "cauchy":
        return np.log1p(z)
    raise ValueError(loss)


def drho(loss, z):
    """rho'(z), elementwise: the match weights."""
    z = np.asarray(z, dtype=np.float64)
    if loss == "huber":
        return np.where(z <= 1.0, 1.0, 1.0 / np.sqrt(np.maximum(z, 1.0)))
    if loss == "soft_l1":
        return 1.0 / np.sqrt(1.0 + z)
    if loss == "cauchy":
        return 1.0 / (1.0 + z)
    raise ValueError(loss)


def match_cost(loss, s, c):
    """c^2 rho(s / c^2); Huber's quadratic branch is s itself, as in the kernel."""
    c2 = c * c
    out = c2 * rho(loss, s / c2)
    return np.where(s <= c2, s, out) if loss == "huber" else out


def _factor(loss, s, c):
    """f(s) = sqrt(c^2 rho(s/c^2) / s) and df/ds per match (1 and 0 at s = 0)."""
    c2 = c * c
    g = match_cost(loss, s, c)
    dg = drho(loss, s / c2)
    pos = s > 0.0
    ss = np.where(pos, s, 1.0)
    f = np.where(pos, np.sqrt(g / ss), 1.0)
    dfds = np.where(pos, (dg * ss - g) / (2.0 * ss * ss * f), 0.0)
    return f, dfds


class Problem:
    """One problem in the oracle's global chart around its gauge-normalised start."""

    def __init__(self, Corresp, CalM, R_t_2, R_t_3, Reconst, loss, scale):
        self.C = np.asarray(Corresp, dtype=np.float64)
        self.Ks = [CalM[0:3], CalM[3:6], CalM[6:9]]
        self.loss, self.c = loss, float(scale)
        R2, t2, R3, t3, X = oba.normalise_gauge(R_t_2[:, :3], R_t_2[:, 3], R_t_3[:, :3], R_t_3[:, 3],
                                                np.asarray(Reconst, dtype=np.float64))
        self.ch = oba.Chart(R2, t2, R3, t3, X)
        self.n = X.shape[1]
        self.p0 = np.zeros(11 + 3 * self.n)

    def residuals(self, p):
        return oba.residuals(self.Ks, *self.ch.unpack(p), self.C)

    def s(self, p):
        r = self.residuals(p).reshape(self.n, 6)
        return np.sum(r * r, axis=1)

    def cost(self, p):
        """sum_i c^2 rho(s_i / c^2)"""
        return float(np.sum(match_cost(self.loss, self.s(p), self.c)))

    def scaled(self, p):
        r = self.residuals(p).reshape(self.n, 6)
        f, _ = _factor(self.loss, np.sum(r * r, axis=1), self.c)
        return (r * f[:, None]).ravel()

    def scaled_jacobian(self, p):
        """d r~ / dp = f J + 2 (df/ds) r (r'J), match by match (dense)."""
        J = self.ch.jacobian(self.Ks, p, self.C).toarray()
        r = self.residuals(p).reshape(self.n, 6)
        f, dfds = _factor(self.loss, np.sum(r * r, axis=1), self.c)
        Jm = J.reshape(self.n, 6, -1)
        rJ = np.einsum("ik,ikj->ij", r, Jm)
        return (f[:, None, None] * Jm + 2.0 * (dfds[:, None] * r)[:, :, None] * rJ[:, None, :]).reshape(6 * self.n, -1)

    def gradient(self, p):
        """Analytic gradient of (1/2) cost in the chart: sum_i rho'(s_i / c^2) J_i' r_i (J_i the chain rule of
        oracle/bundle_adjust.py's Jacobian, vectorised over the matches)."""
        R2, t2, R3, t3, X = self.ch.unpack(p)
        s = self.ch.t2 + self.ch.U @ p[3:5]
        dt2 = (np.eye(3) - np.outer(t2, t2)) @ self.ch.U / np.linalg.norm(s)
        w = drho(self.loss, self.s(p) / (self.c * self.c))
        g = np.zeros(p.size); gX = np.zeros((self.n, 3))
        for m, (R, t) in enumerate(((np.eye(3), np.zeros(3)), (R2, t2), (R3, t3))):
            K = self.Ks[m]
            v = (R @ X).T                                                          # (n, 3)
            h = (v + t) @ K.T
            q = h[:, :2] / h[:, 2:3]
            r = q - self.C[2 * m:2 * m + 2].T
            A = (K[None, :2, :] - q[:, :, None] * K[None, 2:3, :]) / h[:, 2, None, None]   # (n, 2, 3)
            a = w[:, None] * np.einsum("nk,nkj->nj", r, A)
            gX += a @ R
            if m == 1:
                g[0:3] = oba.left_jacobian(p[0:3]).T @ np.cross(v, a).sum(0)
                g[3:5] = dt2.T @ a.sum(0)
            elif m == 2:
                g[5:8] = oba.left_jacobian(p[5:8]).T @ np.cross(v, a).sum(0)
                g[8:11] = a.sum(0)
        g[11:] = gX.ravel()
        return g

    def numeric_gradient(self, p, h=1e-7):
        """Central differences of (1/2) cost in the chart (h = 1e-6 already leaves a truncation error of ~1e-8 of a
        perturbed start's gradient at the minimiser of 30 % outliers)."""
        g = np.zeros(p.size)
        for k in range(p.size):
            e = np.zeros(p.size); e[k] = h
            g[k] = (self.cost(p + e) - self.cost(p - e)) / (4.0 * h)
        return g

    def solve(self, newton=2):
        """MINPACK 'lm' on the rescaled residuals, then `newton` Newton steps on (1/2) cost with the Hessian by central
        differences of the analytic gradient.  Gauss-Newton on r~ lacks the second-order term of the matches with large
        residuals (the outliers), so 'lm' converges linearly there and stops on its ftol with a gradient of ~1e-8 of the
        start's; the Newton steps take it to rounding."""
        p = least_squares(self.scaled, self.p0, jac=self.scaled_jacobian, method="lm", xtol=1e-15, ftol=1e-15,
                          gtol=1e-15, max_nfev=20000).x
        for _ in range(newton):
            g = self.gradient(p)
            H = np.zeros((p.size, p.size))
            for k in range(p.size):
                e = np.zeros(p.size); e[k] = 1e-7
                H[:, k] = (self.gradient(p + e) - self.gradient(p - e)) / 2e-7
            try:
                q = p - np.linalg.solve(0.5 * (H + H.T), g)
            except np.linalg.LinAlgError:                  # a flat direction (a point with near-zero weight)
                break
            if not (np.abs(self.gradient(q)).max() < np.abs(g).max() and self.cost(q) <= self.cost(p) * (1 + 1e-14)):
                break
            p = q
        return p


def bundle_adjust_robust(Corresp, CalM, R_t_2, R_t_3, Reconst, loss, scale):
    """The robust minimiser from the given start.  Returns (R_t_2, R_t_3, Reconst, cost, weights, repr_err)."""
    pr = Problem(Corresp, CalM, R_t_2, R_t_3, Reconst, loss, scale)
    p = pr.solve()
    R2, t2, R3, t3, X = pr.ch.unpack(p)
    w = drho(loss, pr.s(p) / (pr.c * pr.c))
    return (np.column_stack([R2, t2]), np.column_stack([R3, t3]), X, pr.cost(p), w,
            oba.repr_error(pr.Ks, R2, t2, R3, t3, X, pr.C))
