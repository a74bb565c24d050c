"""Bundle adjustment on the CPU: the oracle (oracle/bundle_adjust.py) and the per-point algebra of csrc/tvf_ba.cuh
compiled with g++ (the same source the kernel inlines)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

import oracle as o
from oracle import bundle_adjust as oba
from conftest import ROOT, rot_angle, vec_angle

dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
cm = lambda a: np.ascontiguousarray(np.asarray(a, dtype=np.float64).T).ravel()   # 2-D column-major


@pytest.fixture(scope="module")
def bahost(tmp_path_factory):
    """csrc/tvf_ba.cuh built for the host (g++, no FMA contraction) into a temporary directory."""
    inc = os.path.join(ROOT, "tft_vs_fund_b200", "csrc")
    so = str(tmp_path_factory.mktemp("bahost") / "libbahost.so")
    subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-ffp-contract=off", "-I", inc, "-x", "c++",
                           os.path.join(ROOT, "tests", "hostcheck", "ba_hostcheck.cpp"), "-o", so])
    lib = C.CDLL(so)
    lib.hc_ba_cost.restype = C.c_double
    return lib


def normalised_truth(n, seed):
    """A noise-free sweep scene (experiments.m:93-95) with its ground truth in camera 1's frame and the gauge
    |t2| = 1 (the points by triangulation3D with the true cameras: exact up to rounding without noise)."""
    CalM, R_t0, Cr, _ = o.experiments_subsample(n, 0.0, seed)
    K = CalM[:3]
    Xh = o.triangulation3D([K @ np.eye(3, 4), K @ R_t0[0], K @ R_t0[1]], Cr)
    s = 1.0 / np.linalg.norm(R_t0[0][:, 3])
    Rt2 = np.column_stack([R_t0[0][:, :3], R_t0[0][:, 3] * s])
    Rt3 = np.column_stack([R_t0[1][:, :3], R_t0[1][:, 3] * s])
    return CalM, Cr, Rt2, Rt3, Xh[:3] / Xh[3] * s


def perturbed(Rt2, Rt3, X, rs, rot=1e-3, rel=1e-3):
    dR = lambda: Rotation.from_rotvec(rs.standard_normal(3) * rot / np.sqrt(3)).as_matrix()
    t2 = Rt2[:, 3] + rel * rs.standard_normal(3)
    return (np.column_stack([dR() @ Rt2[:, :3], t2 * 2.0]), np.column_stack([dR() @ Rt3[:, :3], (Rt3[:, 3] + rel * rs.standard_normal(3)) * 2.0]),
            (X + rel * rs.standard_normal(X.shape)) * 2.0)


# ---- oracle -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [4, 7, 20, 100])
def test_oracle_returns_ground_truth_of_noise_free_scenes(n):
    rs = np.random.RandomState(n)
    for seed in (1, 2, 3):
        CalM, Cr, Rt2, Rt3, X = normalised_truth(n, seed)
        s2, s3, sX = perturbed(Rt2, Rt3, X, rs)            # includes a factor 2 of scale: the gauge is restored
        g2, g3, gX, rep = oba.bundle_adjust(Cr, CalM, s2, s3, sX)
        assert rep < 1e-9, (n, seed, rep)
        for a, b in ((Rt2, g2), (Rt3, g3)):
            assert rot_angle(a[:, :3], b[:, :3]) < 1e-9 and vec_angle(a[:, 3], b[:, 3]) < 1e-9, (n, seed)
        assert abs(np.linalg.norm(g2[:, 3]) - 1.0) < 1e-14
        assert abs(np.linalg.norm(g3[:, 3]) / np.linalg.norm(Rt3[:, 3]) - 1.0) < 1e-9
        assert np.abs(gX - X).max() < 1e-9 * np.abs(X).max()


def test_oracle_jacobian_matches_central_differences():
    g = np.load(os.path.join(ROOT, "tests", "golden", "sweep_n20.npz"))
    rs = np.random.RandomState(0)
    for b in (3, 77, 200):
        Cr, CalM = g["Corresp"][b], g["CalM"][b]
        Ks = [CalM[0:3], CalM[3:6], CalM[6:9]]
        ch = oba.Chart(g["tft_Rt2"][b][:, :3], g["tft_Rt2"][b][:, 3], g["tft_Rt3"][b][:, :3], g["tft_Rt3"][b][:, 3],
                       g["tft_Reconst"][b])
        p = rs.standard_normal(71) * 1e-2
        J = ch.jacobian(Ks, p, Cr).toarray()
        Jn = np.zeros_like(J)
        for k in range(71):
            e = np.zeros(71); e[k] = 1e-6
            Jn[:, k] = (oba.residuals(Ks, *ch.unpack(p + e), Cr) - oba.residuals(Ks, *ch.unpack(p - e), Cr)) / 2e-6
        assert np.abs(J - Jn).max() < 1e-8 * np.abs(J).max(), b


def test_oracle_never_raises_repr_error_on_the_sweep_goldens():
    g = np.load(os.path.join(ROOT, "tests", "golden", "sweep_n20.npz"))
    worst = 0.0
    for key in ("tft", "f"):
        for b in range(g["Corresp"].shape[0]):
            Cr, CalM = g["Corresp"][b], g["CalM"][b]
            Ks = [CalM[0:3], CalM[3:6], CalM[6:9]]
            R2, R3, X = g[key + "_Rt2"][b], g[key + "_Rt3"][b], g[key + "_Reconst"][b]
            r0 = oba.repr_error(Ks, R2[:, :3], R2[:, 3], R3[:, :3], R3[:, 3], X, Cr)
            rep = oba.bundle_adjust(Cr, CalM, R2, R3, X)[3]
            assert rep <= r0 * (1 + 1e-12), (key, b, r0, rep)
            worst = max(worst, rep / max(r0, 1e-300))
    print("largest ReprError ratio after / before over 520 starts: %.3f" % worst)


# ---- host build of tvf_ba.cuh -------------------------------------------------------------------------------------
def _problem(b, key="tft"):
    g = np.load(os.path.join(ROOT, "tests", "golden", "sweep_n20.npz"))
    R2, t2, R3, t3, X = oba.normalise_gauge(g[key + "_Rt2"][b][:, :3], g[key + "_Rt2"][b][:, 3], g[key + "_Rt3"][b][:, :3],
                                            g[key + "_Rt3"][b][:, 3], g[key + "_Reconst"][b])
    return g["Corresp"][b], g["CalM"][b], np.column_stack([R2, t2]), np.column_stack([R3, t3]), X


def test_header_jacobian_matches_central_differences(bahost):
    for b in (5, 60, 140):
        Cr, CalM, Rt2, Rt3, X = _problem(b)
        calm = cm(CalM)
        for i in (0, 7, 19):
            x6 = np.ascontiguousarray(Cr[:, i]); Xi = np.ascontiguousarray(X[:, i])
            r = np.zeros(6); Jp = np.zeros(18); Jc = np.zeros(66)
            bahost.hc_ba_jac(dp(calm), dp(cm(Rt2)), dp(cm(Rt3)), dp(Xi), dp(x6), dp(r), dp(Jp), dp(Jc))
            Jp = Jp.reshape(6, 3); Jc = Jc.reshape(6, 11)

            def resid(dc, dX):
                a2 = cm(Rt2); a3 = cm(Rt3)
                bahost.hc_ba_update(dp(calm), dp(a2), dp(a3), dp(np.ascontiguousarray(dc)))
                rr = np.zeros(6); j1 = np.zeros(18); j2 = np.zeros(66)
                bahost.hc_ba_jac(dp(calm), dp(a2), dp(a3), dp(np.ascontiguousarray(Xi + dX)), dp(x6), dp(rr), dp(j1), dp(j2))
                return rr
            assert np.abs(resid(np.zeros(11), np.zeros(3)) - r).max() <= 1e-12 * max(1.0, np.abs(r).max())   # t2 renormalised
            for k in range(11):
                e = np.zeros(11); e[k] = 1e-7
                num = (resid(e, np.zeros(3)) - resid(-e, np.zeros(3))) / 2e-7
                assert np.abs(num - Jc[:, k]).max() < 1e-6 * max(1.0, np.abs(Jc).max()), (b, i, k)
            for k in range(3):
                e = np.zeros(3); e[k] = 1e-7
                num = (resid(np.zeros(11), e) - resid(np.zeros(11), -e)) / 2e-7
                assert np.abs(num - Jp[:, k]).max() < 1e-6 * max(1.0, np.abs(Jp).max()), (b, i, k)
            cost = bahost.hc_ba_cost(dp(calm), dp(cm(Rt2)), dp(cm(Rt3)), dp(Xi), dp(x6))
            assert cost == np.sum(r * r) or abs(cost - np.sum(r * r)) <= 1e-15 * cost


def test_rodrigues_update_stays_orthonormal(bahost):
    """exp([w]x) itself is orthonormal to 1e-15 at every angle, and R <- exp([w]x) R adds no more than that to R's own
    departure from orthonormality."""
    rs = np.random.RandomState(3)
    orth = lambda M: np.abs(M.T @ M - np.eye(3)).max()
    for trial in range(300):
        R = Rotation.from_rotvec(rs.standard_normal(3)).as_matrix()
        mag = 10.0 ** rs.uniform(-14, 0.5) if trial % 10 else [0.0, 1e-8, 1e-4][trial // 10 % 3]
        w = rs.standard_normal(3); w *= mag / np.linalg.norm(w)
        E = cm(np.eye(3))
        bahost.hc_ba_rotate(dp(w), dp(E))
        E = E.reshape(3, 3).T
        assert orth(E) <= 1e-15 and abs(np.linalg.det(E) - 1.0) <= 1e-15, (trial, mag)
        assert np.abs(E - Rotation.from_rotvec(w).as_matrix()).max() <= 1e-15, (trial, mag)
        Rm = cm(R)
        bahost.hc_ba_rotate(dp(w), dp(Rm))
        Rn = Rm.reshape(3, 3).T
        assert orth(Rn) <= orth(R) + 1e-15, (trial, mag)
        assert np.abs(Rn - E @ R).max() <= 1e-15, (trial, mag)


@pytest.mark.parametrize("mu", [0.0, 1e-3, 10.0])
def test_reduced_system_equals_the_dense_schur_complement(bahost, mu):
    """The 11 x 11 system summed from the header's point functions == the Schur complement of the oracle's dense
    normal equations (same chart: the oracle's Jacobian at p = 0 with the header's tangent basis), and the back-
    substituted steps == the dense damped solve."""
    for key, b in (("tft", 9), ("f", 44), ("tft", 201)):
        Cr, CalM, Rt2, Rt3, X = _problem(b, key)
        n = Cr.shape[1]
        Ks = [CalM[0:3], CalM[3:6], CalM[6:9]]
        u1 = np.zeros(3); u2 = np.zeros(3)
        bahost.hc_ba_basis(dp(cm(CalM)), dp(cm(Rt2)), dp(cm(Rt3)), dp(u1), dp(u2))
        ch = oba.Chart(Rt2[:, :3], Rt2[:, 3], Rt3[:, :3], Rt3[:, 3], X, U=np.column_stack([u1, u2]))
        J = ch.jacobian(Ks, np.zeros(11 + 3 * n), Cr).toarray()
        r = oba.residuals(Ks, Rt2[:, :3], Rt2[:, 3], Rt3[:, :3], Rt3[:, 3], X, Cr)
        H = J.T @ J; g = J.T @ r
        Hd = H + mu * np.diag(np.diag(H))
        Hcc, Hcp, Hpp = Hd[:11, :11], Hd[:11, 11:], Hd[11:, 11:]
        S = Hcc - Hcp @ np.linalg.solve(Hpp, Hcp.T)
        rhs = g[:11] - Hcp @ np.linalg.solve(Hpp, g[11:])
        sums = np.zeros(99); dc = np.zeros(11); dX = np.zeros(3 * n)
        ok = bahost.hc_ba_system(dp(cm(CalM)), dp(cm(Rt2)), dp(cm(Rt3)), dp(cm(X)), dp(cm(Cr)), n, C.c_double(mu),
                                 dp(sums), dp(dc), dp(dX))
        assert ok == 1
        iu = np.triu_indices(11)
        Su = (S - mu * np.diag(np.diag(H[:11, :11])))[iu]       # the sums carry the damping of the point blocks only
        assert np.abs(sums[:66] - Su).max() <= 1e-12 * np.abs(S).max(), (key, b)
        assert np.abs(sums[66:77] - rhs).max() <= 1e-12 * np.abs(rhs).max(), (key, b)
        assert np.abs(sums[77:88] - np.diag(H)[:11]).max() <= 1e-12 * np.abs(np.diag(H)[:11]).max()
        assert np.abs(sums[88:99] - g[:11]).max() <= 1e-12 * np.abs(g).max()
        step = np.linalg.solve(Hd, -g)
        assert np.abs(dc - step[:11]).max() <= 1e-9 * np.abs(step).max(), (key, b, mu)
        assert np.abs(dX - step[11:]).max() <= 1e-9 * np.abs(step).max(), (key, b, mu)
