"""Robust-loss bundle adjustment on the CPU: the loss functions and the weighted per-point algebra of csrc/tvf_ba.cuh
compiled with g++ (the same source the kernel inlines), and the oracle (tests/ba_robust_oracle.py)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import ba_robust_oracle as bro
from oracle import bundle_adjust as oba
from conftest import ROOT, rot_angle, vec_angle
from test_bundle_adjust_cpu import normalised_truth, perturbed

dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
cm = lambda a: np.ascontiguousarray(np.asarray(a, dtype=np.float64).T).ravel()   # 2-D column-major
LOSS_ID = {"huber": 1, "soft_l1": 2, "cauchy": 3}


@pytest.fixture(scope="module")
def rhost(tmp_path_factory):
    """tests/hostcheck/ba_robust_hostcheck.cpp built for the host (g++, no FMA contraction) into a temporary directory."""
    inc = os.path.join(ROOT, "tft_vs_fund_b200", "csrc")
    so = str(tmp_path_factory.mktemp("barobust") / "libbarobust.so")
    subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-ffp-contract=off", "-I", inc, "-x", "c++",
                           os.path.join(ROOT, "tests", "hostcheck", "ba_robust_hostcheck.cpp"), "-o", so])
    lib = C.CDLL(so)
    for f in ("hc_ba_loss_cost", "hc_ba_loss_weight", "hc_ba_robust_cost"):
        getattr(lib, f).restype = C.c_double
    lib.hc_ba_loss_cost.argtypes = lib.hc_ba_loss_weight.argtypes = [C.c_int, C.c_double, C.c_double]
    return lib


def outlier_problem(b, frac=0.25, key="tft"):
    """A sweep golden (n = 20) at its pose method's result, gauge-normalised, with a share of its matches replaced by
    uniform pixels of the image, so the weights of a small c spread over (0, 1]."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "sweep_n20.npz"))
    R2, t2, R3, t3, X = oba.normalise_gauge(g[key + "_Rt2"][b][:, :3], g[key + "_Rt2"][b][:, 3], g[key + "_Rt3"][b][:, :3],
                                            g[key + "_Rt3"][b][:, 3], g[key + "_Reconst"][b])
    Cr = g["Corresp"][b].copy()
    rs = np.random.RandomState(b)
    cols = rs.choice(Cr.shape[1], int(round(frac * Cr.shape[1])), replace=False)
    Cr[0::2, cols] = rs.uniform(0, 1800, (3, cols.size))
    Cr[1::2, cols] = rs.uniform(0, 1200, (3, cols.size))
    return Cr, g["CalM"][b], np.column_stack([R2, t2]), np.column_stack([R3, t3]), X


# ---- the losses ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("loss", bro.LOSSES)
def test_header_losses_match_numpy(rhost, loss):
    z = np.concatenate([10.0 ** np.linspace(-12, 12, 241), [0.0, 1.0, np.nextafter(1.0, 0), np.nextafter(1.0, 2)]])
    for c2 in (1.0, 9.0, 0.25):
        s = z * c2
        cost = np.array([rhost.hc_ba_loss_cost(LOSS_ID[loss], x, c2) for x in s])
        w = np.array([rhost.hc_ba_loss_weight(LOSS_ID[loss], x, c2) for x in s])
        ref_cost = bro.match_cost(loss, s, np.sqrt(c2))
        ref_w = bro.drho(loss, s / c2)
        assert np.all(np.abs(cost - ref_cost) <= 4e-16 * np.abs(ref_cost)), (loss, c2)
        assert np.all(np.abs(w - ref_w) <= 4e-16 * ref_w), (loss, c2)
        assert np.all(w > 0.0) and np.all(w <= 1.0)
    if loss == "huber":                                # the quadratic branch is exact, z = 1 included
        for c2 in (1.0, 9.0, 0.3):
            for s in (0.0, 1e-12 * c2, 0.5 * c2, c2):
                assert rhost.hc_ba_loss_cost(1, s, c2) == s and rhost.hc_ba_loss_weight(1, s, c2) == 1.0
            assert rhost.hc_ba_loss_weight(1, 1.01 * c2, c2) < 1.0


# ---- the weighted linearisation of the header -----------------------------------------------------------------------
@pytest.mark.parametrize("loss", bro.LOSSES)
@pytest.mark.parametrize("mu", [0.0, 1e-3, 10.0])
def test_weighted_reduced_system_equals_the_dense_schur_complement(rhost, loss, mu):
    """The sums of the weighed points == the Schur complement of J'WJ (W = the match weights, six rows each) of the
    oracle's dense Jacobian in the header's chart, and the back-substituted steps == the dense damped solve."""
    for b in (9, 44, 201):
        Cr, CalM, Rt2, Rt3, X = outlier_problem(b)
        n = Cr.shape[1]
        for c in (1.0, 3.0):
            Ks = [CalM[0:3], CalM[3:6], CalM[6:9]]
            u1 = np.zeros(3); u2 = np.zeros(3)
            rhost.hc_ba_basis(dp(cm(CalM)), dp(cm(Rt2)), dp(cm(Rt3)), dp(u1), dp(u2))
            ch = oba.Chart(Rt2[:, :3], Rt2[:, 3], Rt3[:, :3], Rt3[:, 3], X, U=np.column_stack([u1, u2]))
            J = ch.jacobian(Ks, np.zeros(11 + 3 * n), Cr).toarray()
            r = oba.residuals(Ks, Rt2[:, :3], Rt2[:, 3], Rt3[:, :3], Rt3[:, 3], X, Cr)
            s = np.sum(r.reshape(n, 6) ** 2, axis=1)
            wref = bro.drho(loss, s / c ** 2)
            Wr = np.repeat(wref, 6)
            H = J.T @ (Wr[:, None] * J); g = J.T @ (Wr * r)
            Hd = H + mu * np.diag(np.diag(H))
            Hcc, Hcp, Hpp = Hd[:11, :11], Hd[:11, 11:], Hd[11:, 11:]
            S = Hcc - Hcp @ np.linalg.solve(Hpp, Hcp.T)
            rhs = g[:11] - Hcp @ np.linalg.solve(Hpp, g[11:])
            w = np.zeros(n); sums = np.zeros(99); gp = np.zeros(3 * n); dc = np.zeros(11); dX = np.zeros(3 * n)
            ok = rhost.hc_ba_robust_system(dp(cm(CalM)), dp(cm(Rt2)), dp(cm(Rt3)), dp(cm(X)), dp(cm(Cr)), n, LOSS_ID[loss],
                                           C.c_double(c * c), C.c_double(mu), dp(w), dp(sums), dp(gp), dp(dc), dp(dX))
            assert ok == 1
            tag = (loss, b, c, mu)
            assert np.abs(w - wref).max() <= 1e-12, tag
            assert wref.min() < 0.1, tag                   # the outliers are down-weighted: W is not I
            iu = np.triu_indices(11)
            Su = (S - mu * np.diag(np.diag(H[:11, :11])))[iu]
            assert np.abs(sums[:66] - Su).max() <= 1e-11 * np.abs(S).max(), tag
            assert np.abs(sums[66:77] - rhs).max() <= 1e-11 * np.abs(rhs).max(), tag
            assert np.abs(sums[77:88] - np.diag(H)[:11]).max() <= 1e-12 * np.abs(np.diag(H)[:11]).max(), tag
            assert np.abs(sums[88:99] - g[:11]).max() <= 1e-12 * np.abs(g).max(), tag
            assert np.abs(gp - g[11:]).max() <= 1e-12 * np.abs(g).max(), tag
            step = np.linalg.solve(Hd, -g)
            assert np.abs(dc - step[:11]).max() <= 1e-9 * np.abs(step).max(), tag
            assert np.abs(dX - step[11:]).max() <= 1e-9 * np.abs(step).max(), tag


@pytest.mark.parametrize("loss", bro.LOSSES)
def test_weighted_gradient_equals_central_differences_of_half_the_cost(rhost, loss):
    """g of the weighed points (camera part: sums 88..98, point part: the eliminations' g_p) is the gradient of
    (1/2) sum c^2 rho(s_i / c^2) in the kernel's local chart (the camera update of the header, the points additively)."""
    for b in (5, 140):
        Cr, CalM, Rt2, Rt3, X = outlier_problem(b)
        n = Cr.shape[1]
        c2 = 4.0
        w = np.zeros(n); sums = np.zeros(99); gp = np.zeros(3 * n); dc = np.zeros(11); dX = np.zeros(3 * n)
        rhost.hc_ba_robust_system(dp(cm(CalM)), dp(cm(Rt2)), dp(cm(Rt3)), dp(cm(X)), dp(cm(Cr)), n, LOSS_ID[loss],
                                  C.c_double(c2), C.c_double(0.0), dp(w), dp(sums), dp(gp), dp(dc), dp(dX))

        def half_cost(dcam, dpts):
            a2, a3 = cm(Rt2), cm(Rt3)
            rhost.hc_ba_update(dp(cm(CalM)), dp(a2), dp(a3), dp(np.ascontiguousarray(dcam)))
            return 0.5 * rhost.hc_ba_robust_cost(dp(cm(CalM)), dp(a2), dp(a3), dp(cm(X) + dpts), dp(cm(Cr)), n,
                                                 LOSS_ID[loss], C.c_double(c2))
        h = 1e-6
        num_c = np.array([(half_cost(h * e, 0.0) - half_cost(-h * e, 0.0)) / (2 * h) for e in np.eye(11)])
        num_p = np.array([(half_cost(np.zeros(11), h * e) - half_cost(np.zeros(11), -h * e)) / (2 * h) for e in np.eye(3 * n)])
        scale = max(np.abs(sums[88:99]).max(), np.abs(gp).max())
        assert np.abs(num_c - sums[88:99]).max() <= 1e-6 * scale, (loss, b)
        assert np.abs(num_p - gp).max() <= 1e-6 * scale, (loss, b)


# ---- the oracle ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("loss", bro.LOSSES)
def test_oracle_jacobian_matches_central_differences(loss):
    rs = np.random.RandomState(0)
    for b in (3, 77):
        Cr, CalM, Rt2, Rt3, X = outlier_problem(b)
        pr = bro.Problem(Cr, CalM, Rt2, Rt3, X, loss, 2.0)
        p = rs.standard_normal(71) * 1e-3
        J = pr.scaled_jacobian(p)
        Jn = np.zeros_like(J)
        for k in range(71):
            e = np.zeros(71); e[k] = 1e-6
            Jn[:, k] = (pr.scaled(p + e) - pr.scaled(p - e)) / 2e-6
        assert np.abs(J - Jn).max() < 1e-7 * np.abs(J).max(), (loss, b)
        assert abs(np.sum(pr.scaled(p) ** 2) - pr.cost(p)) <= 1e-12 * pr.cost(p)     # |r~|^2 is the robust cost


def truth_start(Cr, CalM, R_t0, rs):
    """The true state of a sweep scene (|t2| = 1, points triangulated with the true cameras), perturbed as
    test_bundle_adjust_cpu.perturbed does (includes a factor 2 of scale)."""
    import oracle as o
    K = CalM[:3]
    Xh = o.triangulation3D([K @ np.eye(3, 4), K @ R_t0[0], K @ R_t0[1]], Cr)
    s = 1.0 / np.linalg.norm(R_t0[0][:, 3])
    Rt2 = np.column_stack([R_t0[0][:, :3], R_t0[0][:, 3] * s])
    Rt3 = np.column_stack([R_t0[1][:, :3], R_t0[1][:, 3] * s])
    return perturbed(Rt2, Rt3, Xh[:3] / Xh[3] * s, rs)


@pytest.mark.parametrize("loss", bro.LOSSES)
def test_oracle_result_is_stationary(loss):
    """At the oracle's result the central-difference gradient of (1/2) cost is <= 1e-8 of the start's (30 % outliers,
    n = 100, c = 3 px, from the perturbed truth)."""
    import ransac_oracle as ro
    Cr, CalM, R_t0, _ = ro.outlier_scenes(0.3, 2, 5)
    for b in range(2):
        s2, s3, sX = truth_start(Cr[b], CalM, R_t0, np.random.RandomState(b))
        pr = bro.Problem(Cr[b], CalM, s2, s3, sX, loss, 3.0)
        p = pr.solve()
        g0 = np.abs(pr.numeric_gradient(pr.p0)).max()
        g1 = np.abs(pr.numeric_gradient(p)).max()
        assert g1 <= 1e-8 * g0, (loss, b, g0, g1)
        assert np.abs(pr.gradient(p)).max() <= 1e-8 * g0, (loss, b)
        assert pr.cost(p) <= pr.cost(pr.p0)


def test_huber_with_c_above_every_residual_is_the_plain_oracle():
    """Huber with c^2 above every s_i at the plain minimiser: the quadratic branch throughout, so the plain problem."""
    rs = np.random.RandomState(7)
    for n, seed in ((7, 1), (20, 2), (60, 3)):
        CalM, Cr0, Rt2, Rt3, X = normalised_truth(n, seed)
        Cr = Cr0 + rs.standard_normal(Cr0.shape)                    # 1 px of noise
        s2, s3, sX = perturbed(Rt2, Rt3, X, rs)
        p2, p3, pX, prep = oba.bundle_adjust(Cr, CalM, s2, s3, sX)
        Ks = [CalM[0:3], CalM[3:6], CalM[6:9]]
        smax = np.max(np.sum(oba.residuals(Ks, p2[:, :3], p2[:, 3], p3[:, :3], p3[:, 3], pX, Cr).reshape(n, 6) ** 2, 1))
        c = np.sqrt(smax) * 1.5
        r2, r3, rX, cost, w, rep = bro.bundle_adjust_robust(Cr, CalM, s2, s3, sX, "huber", c)
        assert np.all(w == 1.0), n
        for a, b in ((p2, r2), (p3, r3)):
            assert rot_angle(a[:, :3], b[:, :3]) < 1e-9 and vec_angle(a[:, 3], b[:, 3]) < 1e-9, n
        assert np.abs(rX - pX).max() <= 1e-9 * np.abs(pX).max(), n
        assert abs(rep - prep) <= 1e-9 * prep and abs(cost - 3 * n * prep ** 2) <= 1e-9 * cost, n
