"""Different intrinsics per view and per problem on the CPU (tests/distinct_k.py): the oracles recover the truth of such
scenes, a wrong K moves their answer far beyond the tolerances, and the host builds of the device code (csrc/tvf_pose.cuh,
tvf_ba.cuh, tvf_ransac.cuh compiled with g++, the same source the kernels inline) equal the oracles on them."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

import oracle as o
from oracle import bundle_adjust as oba
import ba_covariance_oracle as bco
import distinct_k as dk
import ransac_oracle as ro
from conftest import ROOT, assert_pose_close, rot_angle, vec_angle, votes8_equal
from make_golden_access import oracle_votes

dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int))
cm = lambda a: np.ascontiguousarray(np.asarray(a, dtype=np.float64).T).ravel()   # 2-D column-major

POSE_METHODS = {"tft": o.LinearTFTPoseEstimation, "f": o.LinearFPoseEstimation, "optf": o.OptimFPoseEstimation}
WRONG_K_MIN = 1e-3        # rad: the least a wrong K must move the oracle's rotations


def _build(tmp_path_factory, src):
    inc = os.path.join(ROOT, "tft_vs_fund_b200", "csrc")
    name = os.path.splitext(src)[0]
    so = str(tmp_path_factory.mktemp(name) / ("lib%s.so" % name))
    subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-ffp-contract=off", "-I", inc, "-x", "c++",
                           os.path.join(ROOT, "tests", "hostcheck", src), "-o", so])
    return C.CDLL(so)


@pytest.fixture(scope="module")
def bahost(tmp_path_factory):
    return _build(tmp_path_factory, "ba_hostcheck.cpp")


@pytest.fixture(scope="module")
def covhost(tmp_path_factory):
    return _build(tmp_path_factory, "ba_cov_hostcheck.cpp")


@pytest.fixture(scope="module")
def rhost(tmp_path_factory):
    return _build(tmp_path_factory, "ransac_hostcheck.cpp")


def vote_tie(votes8):
    """two candidates of a pair share the largest vote (or a vote is NaN)"""
    return any(np.isnan(v).any() or np.sum(v == np.max(v)) > 1 for v in (votes8[:4], votes8[4:]))


def pose_error(a, b):
    """largest rotation angle between two pose pairs (R_t_2, R_t_3), rad"""
    return max(rot_angle(a[0][:, :3], b[0][:, :3]), rot_angle(a[1][:, :3], b[1][:, :3]))


def assert_truth(R2, R3, R_t0, tol, tag):
    for got, true in ((R2, R_t0[0]), (R3, R_t0[1])):
        assert rot_angle(true[:, :3], got[:, :3]) < tol and vec_angle(true[:, 3], got[:, 3]) < tol, tag
    ratio = np.linalg.norm(R3[:, 3]) / np.linalg.norm(R2[:, 3])
    assert abs(ratio / (np.linalg.norm(R_t0[1][:, 3]) / np.linalg.norm(R_t0[0][:, 3])) - 1.0) < tol, tag


# ---- the fixture --------------------------------------------------------------------------------------------------
def test_fixture_draws_a_different_k_per_view_and_per_problem():
    Cr, CalM, R_t0, X = dk.batch(20, 0.0, [1, 2, 3])
    for b in range(3):
        Ks = [CalM[b][0:3], CalM[b][3:6], CalM[b][6:9]]
        for i in range(3):
            assert np.array_equal(Ks[i][2], [0.0, 0.0, 1.0]) and Ks[i][1, 0] == 0.0
            for j in range(i):
                assert abs(Ks[i][0, 0] - Ks[j][0, 0]) > 0.1 * Ks[0][0, 0], (b, i, j)
        # the points reproject onto the matches exactly with the true cameras
        Ps = [Ks[0] @ np.eye(3, 4), Ks[1] @ R_t0[b][0], Ks[2] @ R_t0[b][1]]
        assert np.abs(o.project3Dpoints(X[b], Ps) - Cr[b]).max() < 1e-9
    assert not np.array_equal(CalM[0], CalM[1]) and not np.array_equal(CalM[1], CalM[2])
    assert np.array_equal(dk.batch(20, 0.0, [2])[1][0], CalM[1])                  # seeded


# ---- oracles under different intrinsics -----------------------------------------------------------------------------
@pytest.mark.parametrize("method", ["tft", "f", "optf"])
@pytest.mark.parametrize("n", [8, 20, 100])
def test_oracle_pose_methods_return_the_truth(method, n):
    for seed in (1, 2):
        Cr, CalM, R_t0, _ = dk.scene(n, 0.0, seed)
        R2, R3 = POSE_METHODS[method](Cr, CalM)[:2]
        assert_truth(R2, R3, R_t0, 1e-9, (method, n, seed))


@pytest.mark.parametrize("n", [8, 30])
def test_oracle_votes_have_the_noise_free_pattern(n):
    """One candidate sees every point in front of both cameras (2n), its mirror every point behind both (-2n), the two
    twisted ones every point in front of exactly one (0)."""
    for seed in (1, 2):
        Cr, CalM, _, _ = dk.scene(n, 0.0, seed)
        for votes in oracle_votes(Cr, CalM):
            for p in range(2):
                assert np.array_equal(np.sort(votes[4 * p:4 * p + 4]), [-2 * n, 0, 0, 2 * n]), (n, seed, votes)


@pytest.mark.parametrize("n", [4, 20, 100])
def test_oracle_bundle_adjustment_returns_the_truth(n):
    rs = np.random.RandomState(n)
    for seed in (1, 2):
        Cr, CalM, R_t0, X = dk.scene(n, 0.0, seed)
        Rt2, Rt3, Xs = dk.gauge_truth(CalM, R_t0, X)
        dR = lambda: Rotation.from_rotvec(rs.standard_normal(3) * 1e-3 / np.sqrt(3)).as_matrix()
        s2 = np.column_stack([dR() @ Rt2[:, :3], Rt2[:, 3] + 1e-3 * rs.standard_normal(3)])
        s3 = np.column_stack([dR() @ Rt3[:, :3], Rt3[:, 3] * (1 + 1e-3 * rs.standard_normal(3))])
        g2, g3, gX, rep = oba.bundle_adjust(Cr, CalM, s2, s3, Xs * (1 + 1e-3 * rs.standard_normal(Xs.shape)))
        assert rep < 1e-9, (n, seed, rep)
        assert_truth(g2, g3, [Rt2, Rt3], 1e-9, (n, seed))
        assert np.abs(gX - Xs).max() < 1e-9 * np.abs(Xs).max()


def test_oracle_covariance_is_symmetric_psd_with_the_gauge_null_vector():
    for seed in (1, 2, 3):
        Cr, CalM, R_t0, X = dk.scene(20, 1.0, seed)
        r2, r3, rX, _ = oba.bundle_adjust(Cr, CalM, *dk.gauge_truth(CalM, R_t0, X))
        cc, cp, s2 = bco.covariance(Cr, CalM, r2, r3, rX)
        assert np.abs(cc - cc.T).max() <= 1e-12 * np.abs(cc).max()
        assert np.linalg.eigvalsh(cc).min() >= -1e-12 * np.linalg.norm(cc)
        v = np.zeros(12); v[3:6] = r2[:, 3]
        assert np.linalg.norm(cc @ v) <= 1e-12 * np.linalg.norm(cc)
        assert np.linalg.matrix_rank(cc, tol=1e-9 * np.linalg.norm(cc)) == 11
        assert all(np.linalg.eigvalsh(0.5 * (p + p.T)).min() > 0 for p in cp)
        assert 0.3 < s2 < 3.0, s2                                                       # sigma = 1 px


def test_oracle_inlier_test_at_the_truth_keeps_every_match():
    for seed in (1, 2):
        Cr, CalM, R_t0, _ = dk.scene(60, 0.0, seed)
        mask, mx = ro.inliers(Cr, CalM, R_t0[0], R_t0[1], 1e-6)
        assert mask.all() and mx.max() < 1e-8, (seed, mx.max())


# ---- the fixture discriminates -------------------------------------------------------------------------------------
def test_a_wrong_k_moves_the_oracles_far_beyond_the_tolerances():
    """Each wrong-K variant (K2 and K3 swapped, K1 for every view, another problem's K) moves the rotations of the pose
    methods and of the adjustment by more than 1e-3 rad, and the inlier test at the truth drops matches."""
    Cr, CalM, R_t0, X = dk.batch(30, 0.0, [1, 2, 3])
    worst = {}
    for b in range(3):
        variants = {k: (v[b] if v.ndim == 3 else v) for k, v in dk.wrong_k(CalM).items()}
        if b == 0:
            variants.pop("problem 0 for every problem")
        right = {m: POSE_METHODS[m](Cr[b], CalM[b])[:2] for m in ("tft", "f")}
        ba_right = oba.bundle_adjust(Cr[b], CalM[b], *dk.gauge_truth(CalM[b], R_t0[b], X[b]))
        for name, bad in variants.items():
            for m in ("tft", "f"):
                e = pose_error(right[m], POSE_METHODS[m](Cr[b], bad)[:2])
                worst[(name, m)] = min(worst.get((name, m), np.inf), e)
            e = pose_error(ba_right, oba.bundle_adjust(Cr[b], bad, *dk.gauge_truth(CalM[b], R_t0[b], X[b])))
            worst[(name, "ba")] = min(worst.get((name, "ba"), np.inf), e)
            assert not ro.inliers(Cr[b], bad, R_t0[b][0], R_t0[b][1], 1.0)[0].all(), (b, name)
    print("smallest rotation change under a wrong K (rad): %s" % {k: "%.2e" % v for k, v in worst.items()})
    assert min(worst.values()) > WRONG_K_MIN, worst


# ---- host builds of the device code against the oracles ------------------------------------------------------------
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("n", [8, 20, 60, 200])
def test_host_pose_tail_matches_the_oracle(hostcheck, mode, n):
    """hc_pose_tail (candidates, votes, selection, t3 scale, final DLT) against the oracle's pose, votes against the
    oracle's votes, and the certified vote-sign shortcuts (routes 1 and 2) against the accurate route."""
    for noise in (0.0, 1.0, 3.0):
        for seed in (1, 2, 3):
            Cr, CalM, R_t0, _ = dk.scene(n, noise, seed)
            Ks = [CalM[0:3], CalM[3:6], CalM[6:9]]
            tag = "mode %d n=%d noise=%g seed=%d" % (mode, n, noise, seed)
            if mode == 0:
                R2, R3, Rec, T, _ = o.LinearTFTPoseEstimation(Cr, CalM)
                model = T.ravel(order="F").copy()
            else:
                R2, R3, Rec, T, _, F21, F31 = o.LinearFPoseEstimation(Cr, CalM, return_F=True)
                model = np.concatenate([cm(F21), cm(F31)])
            rep = o.ReprError([Ks[0] @ np.eye(3, 4), Ks[1] @ R2, Ks[2] @ R3], Cr, Rec)
            Rt2 = np.zeros(12); Rt3 = np.zeros(12); rec = np.zeros(3 * n); rp = np.zeros(1); v = np.zeros(8, dtype=np.int32)
            st = hostcheck.hc_pose_tail(mode, dp(model), dp(cm(CalM)), dp(cm(Cr)), n, dp(Rt2), dp(Rt3), dp(rec), dp(rp), ip(v))
            assert st == 0, tag
            votes = oracle_votes(Cr, CalM)[mode]
            assert votes8_equal(v.astype(np.float64), votes), tag
            got = (Rt2.reshape(3, 4, order="F"), Rt3.reshape(3, 4, order="F"), rec.reshape(n, 3).T, T, rp[0])
            if not vote_tie(votes):               # a tie: either pose is the reference's, by LAPACK's signs
                assert_pose_close((R2, R3, Rec, T, rep), got, tag)
            if noise == 0.0:
                assert_truth(got[0], got[1], R_t0, 1e-9, tag)
            for route in (1, 2):
                c = np.zeros(3, dtype=np.int64)
                hostcheck.hc_vote_signs_check(route, mode, dp(model), dp(cm(CalM)), dp(cm(Cr)), n,
                                              c.ctypes.data_as(C.POINTER(C.c_longlong)))
                assert c[0] == 4 * n and c[2] == 0, (tag, route, c)


def test_host_pose_tail_fails_under_a_wrong_k(hostcheck):
    """The same comparison has power: the host tail run with a wrong K misses the oracle's pose by more than 1e-3 rad."""
    n = 30
    for seed in (1, 2):
        Cr, CalM, _, _ = dk.scene(n, 1.0, seed)
        R2, R3, _, T, _ = o.LinearTFTPoseEstimation(Cr, CalM)
        for name, bad in dk.wrong_k(CalM).items():
            Rt2 = np.zeros(12); Rt3 = np.zeros(12); rec = np.zeros(3 * n); rp = np.zeros(1); v = np.zeros(8, dtype=np.int32)
            hostcheck.hc_pose_tail(0, dp(T.ravel(order="F").copy()), dp(cm(bad)), dp(cm(Cr)), n, dp(Rt2), dp(Rt3), dp(rec),
                                   dp(rp), ip(v))
            e = pose_error((R2, R3), (Rt2.reshape(3, 4, order="F"), Rt3.reshape(3, 4, order="F")))
            assert not e < WRONG_K_MIN, (seed, name, e)


def ba_state(n, seed, noise=1.0):
    """A scene with its true state (|t2| = 1) slightly perturbed: a state where the residuals are not small."""
    Cr, CalM, R_t0, X = dk.scene(n, noise, seed)
    Rt2, Rt3, Xs = dk.gauge_truth(CalM, R_t0, X)
    rs = np.random.RandomState(seed)
    dR = lambda: Rotation.from_rotvec(rs.standard_normal(3) * 1e-3).as_matrix()
    return Cr, CalM, np.column_stack([dR() @ Rt2[:, :3], Rt2[:, 3]]), np.column_stack([dR() @ Rt3[:, :3], Rt3[:, 3]]), Xs


def test_host_bundle_adjust_jacobian_and_system_match_the_oracle(bahost):
    """hc_ba_jac point by point == the oracle's analytic Jacobian (same chart, the header's tangent basis of t2), and
    hc_ba_system's reduced camera system == the Schur complement of the oracle's dense normal equations."""
    for n, seed in ((4, 1), (20, 2), (60, 3)):
        Cr, CalM, Rt2, Rt3, X = ba_state(n, seed)
        Ks = [CalM[0:3], CalM[3:6], CalM[6:9]]
        u1 = np.zeros(3); u2 = np.zeros(3)
        bahost.hc_ba_basis(dp(cm(CalM)), dp(cm(Rt2)), dp(cm(Rt3)), dp(u1), dp(u2))
        ch = oba.Chart(Rt2[:, :3], Rt2[:, 3], Rt3[:, :3], Rt3[:, 3], X, U=np.column_stack([u1, u2]))
        J = ch.jacobian(Ks, np.zeros(11 + 3 * n), Cr).toarray()
        r = oba.residuals(Ks, Rt2[:, :3], Rt2[:, 3], Rt3[:, :3], Rt3[:, 3], X, Cr)
        scale = np.abs(J).max()
        for i in range(n):
            rr = np.zeros(6); Jp = np.zeros(18); Jc = np.zeros(66)
            bahost.hc_ba_jac(dp(cm(CalM)), dp(cm(Rt2)), dp(cm(Rt3)), dp(np.ascontiguousarray(X[:, i])),
                             dp(np.ascontiguousarray(Cr[:, i])), dp(rr), dp(Jp), dp(Jc))
            assert np.abs(rr - r[6 * i:6 * i + 6]).max() <= 1e-10 * max(1.0, np.abs(r).max()), (n, i)
            assert np.abs(Jp.reshape(6, 3) - J[6 * i:6 * i + 6, 11 + 3 * i:14 + 3 * i]).max() <= 1e-10 * scale, (n, i)
            assert np.abs(Jc.reshape(6, 11) - J[6 * i:6 * i + 6, :11]).max() <= 1e-10 * scale, (n, i)
        H = J.T @ J; g = J.T @ r
        S = H[:11, :11] - H[:11, 11:] @ np.linalg.solve(H[11:, 11:], H[:11, 11:].T)
        sums = np.zeros(99); dc = np.zeros(11); dX = np.zeros(3 * n)
        assert bahost.hc_ba_system(dp(cm(CalM)), dp(cm(Rt2)), dp(cm(Rt3)), dp(cm(X)), dp(cm(Cr)), n, C.c_double(0.0),
                                   dp(sums), dp(dc), dp(dX)) == 1
        assert np.abs(sums[:66] - S[np.triu_indices(11)]).max() <= 1e-10 * np.abs(S).max(), n
        assert np.abs(sums[88:99] - g[:11]).max() <= 1e-10 * np.abs(g).max(), n
        step = np.linalg.solve(H, -g)
        assert np.abs(dc - step[:11]).max() <= 1e-8 * np.abs(step).max(), n


def host_cov(covhost, Cr, CalM, Rt2, Rt3, X):
    R2, t2, R3, t3, Xn = oba.normalise_gauge(Rt2[:, :3], Rt2[:, 3], Rt3[:, :3], Rt3[:, 3], np.asarray(X, float))
    n = Cr.shape[1]
    cc = np.zeros(144); cp = np.zeros(9 * n); s2 = np.zeros(1); c11 = np.zeros(121); u1 = np.zeros(3); u2 = np.zeros(3)
    st = covhost.hc_ba_cov(dp(cm(CalM)), dp(cm(np.column_stack([R2, t2]))), dp(cm(np.column_stack([R3, t3]))), dp(cm(Xn)),
                           dp(cm(Cr)), n, dp(cc), dp(cp), dp(s2), dp(c11), dp(u1), dp(u2))
    return st, cc.reshape(12, 12).T, cp.reshape(n, 3, 3).transpose(0, 2, 1), s2[0]


def test_host_covariance_matches_the_oracle(covhost):
    rel = lambda a, b: np.linalg.norm(a - b) / np.linalg.norm(b)
    for n, seed in ((4, 1), (5, 2), (20, 3), (33, 4)):
        Cr, CalM, R_t0, X = dk.scene(n, 1.0, seed)
        r2, r3, rX, _ = oba.bundle_adjust(Cr, CalM, *dk.gauge_truth(CalM, R_t0, X))
        cc, cp, s2 = bco.covariance(Cr, CalM, r2, r3, rX)
        st, hc, hp, hs2 = host_cov(covhost, Cr, CalM, r2, r3, rX)
        assert st == 0, n
        assert rel(hc, cc) <= 1e-9 and max(rel(hp[i], cp[i]) for i in range(n)) <= 1e-9, n
        assert abs(hs2 - s2) <= 1e-12 * s2, n
        # power: the covariance under a wrong K is another matrix
        for name, bad in dk.wrong_k(CalM).items():
            assert rel(host_cov(covhost, Cr, bad, r2, r3, rX)[1], cc) > 1e-3, (n, name)


def host_inliers(rhost, CalM, R2, R3, Cr, th):
    n = Cr.shape[1]
    flags = np.zeros(n, dtype=np.int32); mx = np.zeros(n)
    rhost.hc_ransac_inliers(dp(cm(CalM)), dp(cm(R2)), dp(cm(R3)), dp(cm(Cr)), n, C.c_double(th), ip(flags), dp(mx))
    return flags.astype(bool), mx


def test_host_inlier_test_matches_the_oracle(rhost):
    Cr, CalM, R_t0, out = dk.outlier_scenes(0.3, 6, 5)
    rs = np.random.RandomState(6)
    checked = 0
    for b in range(Cr.shape[0]):
        R2, R3 = R_t0[b][0].copy(), R_t0[b][1].copy()
        if b % 2:                           # a perturbed pose, so that many residuals are near the threshold
            R2[:, 3] += rs.normal(0, 0.01, 3); R3[:, 3] += rs.normal(0, 0.01, 3)
        for th in (0.5, 1.0, 3.0):
            got, mx = host_inliers(rhost, CalM[b], R2, R3, Cr[b], th)
            want, wmx = ro.inliers(Cr[b], CalM[b], R2, R3, th)
            assert np.allclose(mx, wmx, rtol=1e-9, atol=1e-9), (b, th)
            far = np.abs(wmx - th) > 1e-9
            assert np.array_equal(got[far], want[far]), (b, th)
            checked += int(far.sum())
        if b % 2 == 0:                      # at the truth every true inlier is kept at 3 px (1 px noise)
            assert host_inliers(rhost, CalM[b], R2, R3, Cr[b], 5.0)[0][~out[b]].all(), b
    assert checked > 1500


# ---- the real-data driver ------------------------------------------------------------------------------------------
def test_relative_poses_stacks_the_cameras_k_in_triplet_order():
    """epfl.relative_poses (experiments_real.m:89-91) on three cameras with different K: CalM = [K_i; K_j; K_k] in the
    order the triplet names the images, and R_t0 relative to the first."""
    from tft_vs_fund_b200 import epfl
    rs = np.random.RandomState(2)
    K0 = np.array([[2760.0, 0.0, 1520.0], [0.0, 2760.0, 1006.0], [0.0, 0.0, 1.0]])
    cams = []
    for _ in range(4):
        K = dk.draw_ks(rs, K0)[0]
        R = Rotation.from_rotvec(rs.standard_normal(3) * 0.3).as_matrix()
        cams.append((K, R, rs.standard_normal(3)))
    for trip in ((0, 1, 2), (2, 0, 3), (3, 2, 1)):
        CalM, R_t0 = epfl.relative_poses([cams[i] for i in trip])
        assert np.array_equal(CalM, np.vstack([cams[i][0] for i in trip])), trip
        (K1, R1, t1), (K2, R2, t2), (K3, R3, t3) = [cams[i] for i in trip]
        X = rs.standard_normal((3, 5)) + [[0.0], [0.0], [8.0]]                      # world points
        for (Kv, Rv, tv), Rt in (((K2, R2, t2), R_t0[0]), ((K3, R3, t3), R_t0[1])):
            Xc1 = R1 @ X + t1[:, None]                                              # in camera 1's frame
            assert np.allclose(Rt[:, :3] @ Xc1 + Rt[:, 3:], Rv @ X + tv[:, None], atol=1e-12), trip
