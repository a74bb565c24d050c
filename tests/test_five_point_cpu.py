"""The calibrated five-point minimal pose on the CPU: csrc/tvf_fivept.cuh compiled with g++ (the same source
five_point_pose_kernel inlines) against the independent oracle in tests/five_point_oracle.py, on scenes whose three views
have different intrinsics (tests/distinct_k.py)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import distinct_k as dk
import five_point_oracle as fo
from conftest import ROOT, rot_angle, vec_angle

dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int))
ST_NO_POSE_2, ST_NO_POSE_3, ST_NONFINITE = 4, 8, 16


@pytest.fixture(scope="module")
def fhost(tmp_path_factory):
    inc = os.path.join(ROOT, "tft_vs_fund_b200", "csrc")
    so = str(tmp_path_factory.mktemp("fivepthost") / "libfivepthost.so")
    subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-ffp-contract=off", "-I", inc, "-x", "c++",
                           os.path.join(ROOT, "tests", "hostcheck", "five_point_hostcheck.cpp"), "-o", so])
    return C.CDLL(so)


def host_pose(fhost, Cr, CalM):
    """(Rt2, Rt3, E (10, 3, 3), n_E, status) of one sample"""
    p = np.ascontiguousarray(np.asarray(Cr, dtype=np.float64).T).ravel()
    cm = np.ascontiguousarray(np.asarray(CalM, dtype=np.float64).T).ravel()
    Rt2, Rt3, E = np.zeros(12), np.zeros(12), np.zeros(90)
    nE, st = np.zeros(1, np.int32), np.zeros(1, np.int32)
    fhost.hc_five_point_pose(dp(p), dp(cm), 1, dp(Rt2), dp(Rt3), dp(E), ip(nE), ip(st))
    return Rt2.reshape(4, 3).T, Rt3.reshape(4, 3).T, E.reshape(10, 3, 3).transpose(0, 2, 1), int(nE[0]), int(st[0])


def roots(fhost, p):
    p = np.ascontiguousarray(p, dtype=np.float64)
    r = np.zeros(10)
    k = fhost.hc_fp_real_roots(dp(p), len(p) - 1, dp(r))
    return r[:k]


def rays(Cr, CalM, v):
    return np.linalg.solve(CalM[3 * v:3 * v + 3], np.vstack([Cr[2 * v:2 * v + 2], np.ones(Cr.shape[1])]))


def true_E(Rt2):
    t = Rt2[:, 3]
    return fo.normalise_E(np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]]) @ Rt2[:, :3])


def constraints(E):
    return np.concatenate([[np.linalg.det(E)], (2 * E @ E.T @ E - np.trace(E @ E.T) * E).ravel()])


@pytest.mark.parametrize("seed", range(12))
def test_exact_scenes(fhost, seed):
    """The true E is among the roots (1e-9 relative, up to sign); every E satisfies the 5 epipolar equations (1e-10) and
    the ten constraints (1e-9: on seed 11 one ill-conditioned root of the degree-10 polynomial leaves 2.5e-10); n_E equals the oracle's real-root count where the roots are separated by > 1e-6; the
    selected pose is the truth (1e-8 rad)."""
    Cr, CalM, Rt0, _ = dk.scene(5, 0.0, seed)
    R2, R3, E, nE, st = host_pose(fhost, Cr, CalM)
    assert st == 0 and 1 <= nE <= 10
    assert np.all(np.isnan(E[nE:])) and np.all(np.isfinite(E[:nE]))
    Et = true_E(Rt0[0])
    assert min(min(np.abs(e - Et).max(), np.abs(e + Et).max()) for e in E[:nE]) < 1e-9
    q1, q2 = rays(Cr, CalM, 0), rays(Cr, CalM, 1)
    for e in E[:nE]:
        assert abs(np.linalg.norm(e) - 1) < 1e-12
        assert np.abs(constraints(e)).max() < 1e-9
        assert np.abs(np.einsum("ij,ik,kj->j", q2, e, q1)).max() < 1e-10 * np.linalg.norm(q1, axis=0).max() * np.linalg.norm(q2, axis=0).max()
    Eo, nEo = fo.essentials(q1, q2)
    zs = np.sort(np.array([e.ravel()[0] for e in Eo]))
    if nEo < 2 or np.min(np.diff(zs)) > 1e-6:
        assert nE == nEo
    s = 1.0 / np.linalg.norm(Rt0[0][:, 3])
    assert rot_angle(R2[:, :3], Rt0[0][:, :3]) < 1e-8 and vec_angle(R2[:, 3], Rt0[0][:, 3]) < 1e-8
    assert rot_angle(R3[:, :3], Rt0[1][:, :3]) < 1e-8 and vec_angle(R3[:, 3], Rt0[1][:, 3]) < 1e-8
    assert abs(np.linalg.norm(R2[:, 3]) - 1) < 1e-12
    assert np.abs(R3[:, 3] - Rt0[1][:, 3] * s).max() < 1e-8 * np.linalg.norm(R3[:, 3])


def test_sturm_root_finder(fhost):
    assert np.allclose(roots(fhost, np.polynomial.polynomial.polyfromroots([3, -2, 0.5, 7, -11])), [-11, -2, 0.5, 3, 7],
                       rtol=1e-13, atol=1e-13)
    clustered = [1.0, 1.0 + 1e-3, 1.0 + 2e-3, 2.0]
    r = roots(fhost, np.polynomial.polynomial.polyfromroots(clustered))
    assert len(r) == 4 and np.abs(r - clustered).max() < 1e-9
    r = roots(fhost, np.polynomial.polynomial.polyfromroots([1.5, 1.5, -4.0]))      # a double root counts once
    assert len(r) == 2 and abs(r[0] + 4) < 1e-12 and abs(r[1] - 1.5) < 1e-7
    p = np.append(np.polynomial.polynomial.polyfromroots([2.0, -3.0, 5.0]), [1e-17, 0.0])   # vanishing leading terms
    assert np.allclose(roots(fhost, p), [-3, 2, 5], rtol=1e-12)
    assert len(roots(fhost, [1.0, 0.0, 1.0])) == 0 and len(roots(fhost, [2.0, 0.0, 3.0, 0.0, 1.0])) == 0
    assert len(roots(fhost, [0.0, 0.0, 0.0])) == 0
    ten = np.linspace(-3.0, 4.0, 10)
    assert np.abs(roots(fhost, np.polynomial.polynomial.polyfromroots(ten)) - ten).max() < 1e-8


@pytest.mark.parametrize("seed", range(6))
def test_p3p(fhost, seed):
    """The true pose is among the roots; every root maps its 3 points onto their rays."""
    rs = np.random.RandomState(seed)
    X = rs.uniform(-2, 2, (3, 3)) + np.array([0, 0, 6.0])[:, None]
    ang = rs.uniform(-0.3, 0.3, 3)
    R = np.linalg.qr(np.eye(3) + np.array([[0, -ang[2], ang[1]], [ang[2], 0, -ang[0]], [-ang[1], ang[0], 0]]))[0]
    R = R * np.sign(np.diag(R))
    t = rs.uniform(-1, 1, 3)
    Y = R @ X + t[:, None]
    y = Y / np.linalg.norm(Y, axis=0)
    Rs, ts = np.zeros(36), np.zeros(12)
    k = fhost.hc_p3p(dp(np.ascontiguousarray(X.T)), dp(np.ascontiguousarray(y.T)), dp(Rs), dp(ts))
    assert 1 <= k <= 4
    Rs = Rs.reshape(4, 3, 3).transpose(0, 2, 1)[:k]; ts = ts.reshape(4, 3)[:k]
    assert min(np.abs(Rs[i] - R).max() + np.abs(ts[i] - t).max() for i in range(k)) < 1e-10
    for i in range(k):
        Yi = Rs[i] @ X + ts[i][:, None]
        assert np.abs(Yi / np.linalg.norm(Yi, axis=0) - y).max() < 1e-10
        assert np.abs(Rs[i] @ Rs[i].T - np.eye(3)).max() < 1e-10
    want = fo.p3p_grunert(X, y)
    assert len(want) == k


def test_refusals(fhost):
    Cr, CalM, _, _ = dk.scene(5, 0.0, 3)
    cases = {"identical": np.repeat(Cr[:, :1], 5, axis=1), "nan": Cr.copy(), "inf": Cr.copy(), "zero baseline": Cr.copy()}
    cases["nan"][3, 2] = np.nan
    cases["inf"][0, 4] = np.inf
    cases["zero baseline"][2:4] = cases["zero baseline"][0:2]       # views 1 and 2 the same image
    for name, c in cases.items():
        cal = CalM.copy()
        if name == "zero baseline":
            cal[3:6] = cal[0:3]
        R2, R3, E, nE, st = host_pose(fhost, c, cal)
        assert 0 <= nE <= 10 and np.all(np.isnan(E[nE:])), name
        if name == "zero baseline" and st == 0:
            # the other roots are genuine poses that explain the 5 matches; the zero-baseline solution itself has its
            # points at infinity and is dropped
            assert np.all(np.isfinite(R2)) and abs(np.linalg.norm(R2[:, 3]) - 1) < 1e-12
            continue
        assert st in (ST_NO_POSE_2, ST_NO_POSE_3, ST_NONFINITE), (name, st)
        assert np.all(np.isnan(R2)) and np.all(np.isnan(R3)), name


def test_noise_against_the_oracle(fhost):
    """At 1 px, the host build's pose equals the oracle's (1e-6 rad) wherever the oracle's selection is unambiguous (the
    two best view-3 errors differ by > 0.5 px)."""
    checked = 0
    for seed in range(40):
        Cr, CalM, _, _ = dk.scene(5, 1.0, seed)
        R2, R3, E, nE, st = host_pose(fhost, Cr, CalM)
        w2, w3, Ew, nEw, stw, gap = fo.five_point_pose(Cr, CalM)
        assert st == stw, seed
        if st or gap < 0.5:
            continue
        checked += 1
        for a, b in ((w2, R2), (w3, R3)):
            assert rot_angle(a[:, :3], b[:, :3]) < 1e-6 and vec_angle(a[:, 3], b[:, 3]) < 1e-6, seed
    assert checked >= 30
