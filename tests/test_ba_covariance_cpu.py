"""Covariance of the bundle adjustment on the CPU: the oracle (tests/ba_covariance_oracle.py) against Monte Carlo, and the
covariance functions of csrc/tvf_ba.cuh compiled with g++ (the same source ba_covariance_kernel inlines) against the
oracle's dense inverse."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle as o
from oracle import bundle_adjust as oba
import ba_covariance_oracle as bco
from conftest import ROOT

dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
cm = lambda a: np.ascontiguousarray(np.asarray(a, dtype=np.float64).T).ravel()   # 2-D column-major

# Relative Frobenius distance between the empirical covariance of 2 000 adjusted noise draws and the prediction.  With
# the oracle at this draw count it measured 0.015-0.063 over six independent draw sets (seeds 0-5: 0.019, 0.052, 0.063,
# 0.049, 0.050, 0.015); the test uses seed 0 and allows about twice the largest.
MC_DRAWS = 2000
MC_TOL = 0.12


def _build(tmp_path_factory, src, name):
    inc = os.path.join(ROOT, "tft_vs_fund_b200", "csrc")
    so = str(tmp_path_factory.mktemp(name) / ("lib%s.so" % name))
    subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-ffp-contract=off", "-I", inc, "-x", "c++",
                           os.path.join(ROOT, "tests", "hostcheck", src), "-o", so])
    return C.CDLL(so)


@pytest.fixture(scope="module")
def covhost(tmp_path_factory):
    """csrc/tvf_ba.cuh's covariance functions built for the host (g++, no FMA contraction)."""
    return _build(tmp_path_factory, "ba_cov_hostcheck.cpp", "bacovhost")


@pytest.fixture(scope="module")
def bahost(tmp_path_factory):
    return _build(tmp_path_factory, "ba_hostcheck.cpp", "bahost_cov")


def truth_scene(n, seed):
    """A noise-free sweep scene with its ground truth in camera 1's frame, |t2| = 1."""
    CalM, R_t0, Cr, _ = o.experiments_subsample(n, 0.0, seed)
    K = CalM[:3]
    Xh = o.triangulation3D([K @ np.eye(3, 4), K @ R_t0[0], K @ R_t0[1]], Cr)
    s = 1.0 / np.linalg.norm(R_t0[0][:, 3])
    Rt2 = np.column_stack([R_t0[0][:, :3], R_t0[0][:, 3] * s])
    Rt3 = np.column_stack([R_t0[1][:, :3], R_t0[1][:, 3] * s])
    return CalM, Cr, Rt2, Rt3, Xh[:3] / Xh[3] * s


def host_cov(covhost, Cr, CalM, Rt2, Rt3, X):
    """hc_ba_cov on a state (gauge-normalised here as the kernel does)."""
    R2, t2, R3, t3, Xn = oba.normalise_gauge(Rt2[:, :3], Rt2[:, 3], Rt3[:, :3], Rt3[:, 3], np.asarray(X, float))
    n = Cr.shape[1]
    cc = np.zeros(144); cp = np.zeros(9 * n); s2 = np.zeros(1); c11 = np.zeros(121); u1 = np.zeros(3); u2 = np.zeros(3)
    st = covhost.hc_ba_cov(dp(cm(CalM)), dp(cm(np.column_stack([R2, t2]))), dp(cm(np.column_stack([R3, t3]))), dp(cm(Xn)),
                           dp(cm(Cr)), n, dp(cc), dp(cp), dp(s2), dp(c11), dp(u1), dp(u2))
    return st, cc.reshape(12, 12).T, cp.reshape(n, 3, 3).transpose(0, 2, 1), s2[0], c11.reshape(11, 11).T, np.column_stack([u1, u2])


def rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


# ---- oracle -------------------------------------------------------------------------------------------------------
def test_oracle_covariance_matches_monte_carlo():
    """2 000 noise draws (sigma = 1 px) of one n = 20 scene, each adjusted by the oracle from the truth: the empirical
    covariance of [w2, dt2, w3, dt3] about the truth matches covariance() at the truth."""
    CalM, Cr, Rt2, Rt3, X = truth_scene(20, 1)
    cc, _, _ = bco.covariance(Cr, CalM, Rt2, Rt3, X)
    rs = np.random.RandomState(0)
    Z = np.empty((MC_DRAWS, 12))
    for d in range(MC_DRAWS):
        g2, g3, _, _ = oba.bundle_adjust(Cr + rs.standard_normal(Cr.shape), CalM, Rt2, Rt3, X)
        Z[d] = bco.chart_coordinates(g2, g3, Rt2, Rt3)
    E = Z.T @ Z / MC_DRAWS
    err = rel(E, cc)
    ratio = np.sqrt(np.diag(E) / np.diag(cc))
    print("Monte Carlo, %d draws: relative Frobenius %.4f; std ratios %s" % (MC_DRAWS, err, np.round(ratio, 3)))
    assert err < MC_TOL
    assert np.all(np.abs(ratio - 1.0) < 0.1)


def test_oracle_covariance_is_basis_free_and_has_the_gauge_null_direction():
    CalM, Cr, Rt2, Rt3, X = truth_scene(20, 2)
    Cr = Cr + np.random.RandomState(1).standard_normal(Cr.shape)
    r2, r3, rX, _ = oba.bundle_adjust(Cr, CalM, Rt2, Rt3, X)
    cc, cp, s2 = bco.covariance(Cr, CalM, r2, r3, rX)
    Hi, _, _, U = bco.dense_inverse(Cr, CalM, r2, r3, rX)
    V = U @ np.array([[np.cos(0.7), -np.sin(0.7)], [np.sin(0.7), np.cos(0.7)]])       # another tangent basis
    Hv, _, _, _ = bco.dense_inverse(Cr, CalM, r2, r3, rX, U=V)
    G = bco.expansion(V)
    assert rel(G @ Hv[:11, :11] @ G.T, cc) < 1e-9
    v = np.zeros(12); v[3:6] = r2[:, 3]
    assert np.linalg.norm(cc @ v) <= 1e-12 * np.linalg.norm(cc)
    assert np.linalg.matrix_rank(cc, tol=1e-9 * np.linalg.norm(cc)) == 11
    assert 0.5 < s2 < 2.0                                                                   # sigma = 1 px


# ---- host build of tvf_ba.cuh -------------------------------------------------------------------------------------
def _golden_adjusted():
    """The sweep-golden problems adjusted by the oracle from the library-format starts of both methods (starts below
    10 px, the oracle's domain)."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "sweep_n20.npz"))
    for key in ("tft", "f"):
        for b in range(g["Corresp"].shape[0]):
            Cr, CalM = g["Corresp"][b], g["CalM"][b]
            R2, R3, X = g[key + "_Rt2"][b], g[key + "_Rt3"][b], g[key + "_Reconst"][b]
            Ks = [CalM[0:3], CalM[3:6], CalM[6:9]]
            if not oba.repr_error(Ks, R2[:, :3], R2[:, 3], R3[:, :3], R3[:, 3], X, Cr) < 10.0:
                continue
            r2, r3, rX, _ = oba.bundle_adjust(Cr, CalM, R2, R3, X)
            yield "%s %d" % (key, b), Cr, CalM, r2, r3, rX


def test_header_covariance_matches_the_dense_inverse(covhost):
    checked, worst = 0, 0.0
    for tag, Cr, CalM, r2, r3, rX in _golden_adjusted():
        cc, cp, s2 = bco.covariance(Cr, CalM, r2, r3, rX)
        st, hc, hp, hs2, _, _ = host_cov(covhost, Cr, CalM, r2, r3, rX)
        assert st == 0, tag
        e = max(rel(hc, cc), max(rel(hp[i], cp[i]) for i in range(Cr.shape[1])))
        worst = max(worst, e)
        assert e <= 1e-9, (tag, e)
        assert abs(hs2 - s2) <= 1e-12 * s2 + 1e-20, tag      # noise-free trials: sigma2 is rounding (~1e-25)
        assert np.array_equal(hc, hc.T) and all(np.array_equal(p, p.T) for p in hp), tag
        v = np.zeros(12); v[3:6] = r2[:, 3]
        assert np.linalg.norm(hc @ v) <= 1e-12 * np.linalg.norm(hc), tag
        checked += 1
    print("%d adjusted sweep problems: worst relative Frobenius %.2e" % (checked, worst))
    assert checked >= 150


def test_schur_identity(covhost, bahost):
    """The camera block of the dense inverse (in the header's tangent basis) == the inverse of the reduced matrix that
    the adjustment's own ba_point_accumulate sums at mu = 0, and == the header's chart covariance."""
    for tag, Cr, CalM, r2, r3, rX in list(_golden_adjusted())[::10]:
        st, _, _, _, C11, U = host_cov(covhost, Cr, CalM, r2, r3, rX)
        Hi, _, _, _ = bco.dense_inverse(Cr, CalM, r2, r3, rX, U=U)
        n = Cr.shape[1]
        sums = np.zeros(99); dc = np.zeros(11); dX = np.zeros(3 * n)
        X = rX / np.linalg.norm(r2[:, 3])
        bahost.hc_ba_system(dp(cm(CalM)), dp(cm(r2)), dp(cm(r3)), dp(cm(X)), dp(cm(Cr)), n, C.c_double(0.0), dp(sums),
                            dp(dc), dp(dX))
        S = np.zeros((11, 11)); S[np.triu_indices(11)] = sums[:66]
        S = S + np.triu(S, 1).T
        assert rel(np.linalg.inv(S), Hi[:11, :11]) <= 1e-9, tag
        assert rel(C11, Hi[:11, :11]) <= 1e-9, tag


def test_identical_points_are_singular(covhost):
    CalM, Cr, Rt2, Rt3, X = truth_scene(8, 1)
    Cr = np.repeat(Cr[:, :1], 8, axis=1); X = np.repeat(X[:, :1], 8, axis=1)
    st = host_cov(covhost, Cr, CalM, Rt2, Rt3, X)[0]
    assert st == 64
