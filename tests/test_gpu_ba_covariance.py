"""tvf_ba_covariance on the GPU against the CPU oracle (tests/ba_covariance_oracle.py), against Monte Carlo of the
library's own adjustment, its invariances and its edge cases."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle as o
from oracle import bundle_adjust as oba
import ba_covariance_oracle as bco
from conftest import ROOT
from test_ba_covariance_cpu import MC_TOL, truth_scene

pytestmark = pytest.mark.gpu

TOL_COV = 1e-6        # relative Frobenius, per problem
TOL_SIGMA2 = 1e-10    # relative (plus 1e-20 absolute for the noise-free trials, whose sigma2 is rounding)


def golden(name):
    return np.load(os.path.join(ROOT, "tests", "golden", name))


def rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def adjusted(tvf, Cr, CalM, method):
    fn = tvf.LinearTFTPoseEstimation if method == 1 else tvf.LinearFPoseEstimation
    r = fn(Cr, CalM)
    return r, tvf.bundle_adjust(Cr, CalM, r[0], r[1], r[2])


def check_against_oracle(tvf, Cr, CalM, ba, keep, label):
    cov = tvf.ba_covariance(Cr, CalM, ba[0], ba[1], ba[2], points=True)
    worst = 0.0
    for b in np.flatnonzero(keep):
        cb = CalM if CalM.ndim == 2 else CalM[b]
        tag = "%s problem %d" % (label, b)
        cc, cp, s2 = bco.covariance(Cr[b], cb, ba[0][b], ba[1][b], ba[2][b])
        g = cov[0][b]
        assert cov.status[b] == 0, tag
        e = max(rel(g, cc), max(rel(cov.cov_pts[b][:, :, i], cp[i]) for i in range(Cr.shape[2])))
        worst = max(worst, e)
        assert e <= TOL_COV, (tag, e)
        assert abs(cov[1][b] - s2) <= TOL_SIGMA2 * s2 + 1e-20, (tag, cov[1][b], s2)
        # symmetric bit for bit, positive semidefinite, null direction (0, t2, 0, 0)
        assert np.array_equal(g, g.T), tag
        assert np.linalg.eigvalsh(g).min() >= -1e-12 * np.linalg.norm(g), tag
        v = np.zeros(12); v[3:6] = ba[0][b][:, 3]
        assert np.linalg.norm(g @ v) <= 1e-12 * np.linalg.norm(g), tag
        assert all(np.array_equal(cov.cov_pts[b][:, :, i], cov.cov_pts[b][:, :, i].T) for i in range(Cr.shape[2])), tag
    return int(np.sum(keep)), worst


@pytest.mark.parametrize("method", [1, 7])
def test_matches_oracle_on_the_sweep_trials(tvf, method):
    g = golden("sweep_n20.npz")
    Cr, CalM = g["Corresp"], g["CalM"]
    start, ba = adjusted(tvf, Cr, CalM, method)
    keep = np.array([oba.repr_error([CalM[b][0:3], CalM[b][3:6], CalM[b][6:9]], start[0][b][:, :3], start[0][b][:, 3],
                                    start[1][b][:, :3], start[1][b][:, 3], start[2][b], Cr[b]) < 10.0
                     for b in range(Cr.shape[0])]) & (ba.status == 0)
    checked, worst = check_against_oracle(tvf, Cr, CalM, ba, keep, "sweep method %d" % method)
    print("method %d: %d sweep problems, worst relative Frobenius %.2e" % (method, checked, worst))
    assert checked >= 80


@pytest.mark.parametrize("name", ["example_n100.npz", "epfl_triplets.npz"])
def test_matches_oracle_on_example_and_epfl(tvf, name):
    g = golden(name)
    Cr, CalM = g["Corresp"], g["CalM"]
    for method in (1, 7):
        _, ba = adjusted(tvf, Cr, CalM, method)
        checked, worst = check_against_oracle(tvf, Cr, CalM, ba, ba.status == 0, "%s method %d" % (name, method))
        print("%s method %d: %d problems, worst relative Frobenius %.2e" % (name, method, checked, worst))
        assert checked >= 1


def test_monte_carlo_of_the_library_adjustment(tvf):
    """20 000 noise draws (sigma = 1 px) of one n = 20 scene, adjusted from the truth in one tvf_bundle_adjust batch:
    their empirical covariance about the truth matches the library's covariance at the truth."""
    D = 20000
    CalM, Cr, Rt2, Rt3, X = truth_scene(20, 1)
    cov = tvf.ba_covariance(Cr, CalM, Rt2, Rt3, X)
    rs = np.random.RandomState(7)
    Cn = Cr[None] + rs.standard_normal((D,) + Cr.shape)
    res = tvf.bundle_adjust(Cn, CalM, np.broadcast_to(Rt2, (D, 3, 4)), np.broadcast_to(Rt3, (D, 3, 4)),
                            np.broadcast_to(X, (D, 3, 20)))
    assert np.all(res.status == 0)
    Z = np.stack([bco.chart_coordinates(res[0][d], res[1][d], Rt2, Rt3) for d in range(D)])
    E = Z.T @ Z / D
    err = rel(E, cov[0])
    ratio = np.sqrt(np.diag(E) / np.diag(cov[0]))
    print("device Monte Carlo, %d draws: relative Frobenius %.4f; std ratios %s" % (D, err, np.round(ratio, 3)))
    assert err < MC_TOL
    assert np.all(np.abs(ratio - 1.0) < 0.05)
    # the a-posteriori noise estimate is unbiased: its mean over the draws is sigma^2 = 1
    s2 = tvf.ba_covariance(Cn[:2000], CalM, res[0][:2000], res[1][:2000], res[2][:2000])[1]
    assert abs(np.mean(s2) - 1.0) < 0.03, np.mean(s2)


def _bits_equal(a, b):
    return all(np.array_equal(np.asarray(x), np.asarray(y), equal_nan=True) for x, y in zip(a, b))


def test_bit_identity_across_batch_chunk_group_and_device_pointers(tvf):
    import torch
    from tft_vs_fund_b200 import _lib
    g = golden("sweep_n20.npz")
    Cr, CalM = g["Corresp"][:60], g["CalM"][:60]
    ba = tvf.bundle_adjust(Cr, CalM, g["f_Rt2"][:60], g["f_Rt3"][:60], g["f_Reconst"][:60])
    Rt2, Rt3, X = ba[0], ba[1], ba[2]
    full = tvf.ba_covariance(Cr, CalM, Rt2, Rt3, X, points=True)
    outs = lambda r: (r[0], r[1], r.cov_pts, r.status)
    for b in (0, 17, 59):
        one = tvf.ba_covariance(Cr[b:b + 1], CalM[b:b + 1], Rt2[b:b + 1], Rt3[b:b + 1], X[b:b + 1], points=True)
        assert _bits_equal([x[b:b + 1] for x in outs(full)], outs(one)), b
    h = _lib.handle()
    try:
        h.call("tvf_set_chunk", 7)
        chunked = tvf.ba_covariance(Cr, CalM, Rt2, Rt3, X, points=True)
    finally:
        h.call("tvf_set_chunk", 0)
    assert _bits_equal(outs(full), outs(chunked))
    grouped = tvf.api.ba_covariance(Cr, CalM, Rt2, Rt3, X, points=True, device=(0, 0))
    assert _bits_equal(outs(full), outs(grouped))
    # _dev == host
    dev = torch.device("cuda", 0)
    cm = lambda a, nd: torch.from_numpy(tvf.api._cm(a, nd)[0]).to(dev)
    B, n = Cr.shape[0], Cr.shape[2]
    d_c, d_m, d_r2, d_r3, d_x = cm(Cr, 2), cm(CalM, 2), cm(Rt2, 2), cm(Rt3, 2), cm(X, 2)
    o_cc = torch.empty((B, 144), dtype=torch.float64, device=dev)
    o_cp = torch.empty((B, 9 * n), dtype=torch.float64, device=dev)
    o_s2 = torch.empty(B, dtype=torch.float64, device=dev); o_st = torch.zeros(B, dtype=torch.int32, device=dev)
    p = lambda t: C.c_void_p(t.data_ptr())
    torch.cuda.synchronize()
    h.call("tvf_ba_covariance_dev", p(d_c), p(d_m), 1, n, B, p(d_r2), p(d_r3), p(d_x), p(o_cc), p(o_cp), p(o_s2), p(o_st))
    h.call("tvf_synchronize")
    back = lambda t, dims: tvf.api._from_cm(t.cpu().numpy().ravel(), B, dims, True)
    assert np.array_equal(back(o_cc, (12, 12)), full[0]) and np.array_equal(back(o_cp, (3, 3, n)), full.cov_pts)
    assert np.array_equal(o_s2.cpu().numpy(), full[1]) and np.array_equal(o_st.cpu().numpy(), full.status)
    # NULL optional outputs: the others are unchanged
    o_s2b = torch.empty(B, dtype=torch.float64, device=dev)
    h.call("tvf_ba_covariance_dev", p(d_c), p(d_m), 1, n, B, p(d_r2), p(d_r3), p(d_x), None, None, p(o_s2b), None)
    h.call("tvf_synchronize")
    assert np.array_equal(o_s2b.cpu().numpy(), full[1])
    dp = lambda a: a.ctypes.data_as(_lib.c_double_p)
    c, _, _ = tvf.api._cm(Cr, 2); mm, _, _ = tvf.api._cm(CalM, 2)
    r2, _, _ = tvf.api._cm(Rt2, 2); r3, _, _ = tvf.api._cm(Rt3, 2); xx, _, _ = tvf.api._cm(X, 2)
    cc = np.empty((B, 144))
    rc = h.lib.tvf_ba_covariance(h._h, dp(c), dp(mm), 1, n, B, dp(r2), dp(r3), dp(xx), dp(cc), None, None, None)
    assert rc == 0 and np.array_equal(tvf.api._from_cm(cc.ravel(), B, (12, 12), True), full[0])


def test_status_cases(tvf):
    from tft_vs_fund_b200 import _lib
    g = golden("sweep_n20.npz")
    Cr, CalM = g["Corresp"][:6].copy(), g["CalM"][:6]
    ba = tvf.bundle_adjust(Cr, CalM, g["tft_Rt2"][:6], g["tft_Rt3"][:6], g["tft_Reconst"][:6])
    Rt2, Rt3, X = ba[0].copy(), ba[1].copy(), ba[2].copy()
    clean = tvf.ba_covariance(Cr, CalM, Rt2, Rt3, X, points=True)
    assert np.all(clean.status == 0)
    Cr[2, 3, 5] = np.nan                       # NaN input
    Rt2[4, :, 3] = 0.0                         # |t2| = 0
    X[1, :, :] = X[1, :, :1]                   # all points of problem 1 identical ...
    Cr[1] = Cr[1][:, :1]                       # ... and so are their images
    dirty = tvf.ba_covariance(Cr, CalM, Rt2, Rt3, X, points=True)
    assert dirty.status[2] == _lib.ST_NONFINITE and dirty.status[4] == _lib.ST_NONFINITE
    assert dirty.status[1] == _lib.ST_COV_SINGULAR
    for b in (1, 2, 4):
        assert np.all(np.isnan(dirty[0][b])) and np.isnan(dirty[1][b]) and np.all(np.isnan(dirty.cov_pts[b])), b
    keep = [0, 3, 5]
    assert _bits_equal([x[keep] for x in (clean[0], clean[1], clean.cov_pts, clean.status)],
                       [x[keep] for x in (dirty[0], dirty[1], dirty.cov_pts, dirty.status)])
    h = _lib.handle()
    n, B = 3, 1
    c = np.zeros(6 * n); m = np.tile(np.eye(3), (3, 1)).T.copy(); r = np.zeros(12); x = np.zeros(3 * n)
    dp = lambda a: a.ctypes.data_as(_lib.c_double_p)
    rc = h.lib.tvf_ba_covariance(h._h, dp(c), dp(m), 0, n, B, dp(r), dp(r), dp(x), None, None, None, None)
    assert rc == _lib.TVF_ERR_ARG
    rc = h.lib.tvf_ba_covariance(h._h, dp(np.zeros(24)), dp(m), 0, 4, B, dp(r), dp(r), None, None, None, None, None)
    assert rc == _lib.TVF_ERR_ARG            # reconst is required


def test_api_single_problem_and_pose_rms_errors(tvf):
    g = golden("sweep_n20.npz")
    Cr, CalM = g["Corresp"][:5], g["CalM"][0]
    ba = tvf.bundle_adjust(Cr, CalM, g["tft_Rt2"][:5], g["tft_Rt3"][:5], g["tft_Reconst"][:5])
    batch = tvf.ba_covariance(Cr, CalM, ba[0], ba[1], ba[2], points=True)
    assert batch[0].shape == (5, 12, 12) and batch[1].shape == (5,) and batch.cov_pts.shape == (5, 3, 3, 20)
    one = tvf.ba_covariance(Cr[3], CalM, ba[0][3], ba[1][3], ba[2][3])
    assert one[0].shape == (12, 12) and isinstance(one[1], float) and isinstance(one.status, int) and one.cov_pts is None
    assert np.array_equal(one[0], batch[0][3]) and one[1] == batch[1][3]
    rot, tdir = tvf.pose_rms_errors(batch[0], ba[0], ba[1], sigma2=batch[1])
    assert rot.shape == (5, 2) and tdir.shape == (5, 2)
    r1, t1 = tvf.pose_rms_errors(one[0], ba[0][3], ba[1][3], sigma2=one[1])
    assert np.allclose(r1, rot[3], rtol=1e-14) and np.allclose(t1, tdir[3], rtol=1e-14)
    c = batch[0][3] * batch[1][3]
    t3 = ba[1][3][:, 3] / np.linalg.norm(ba[0][3][:, 3])
    P = np.eye(3) - np.outer(t3, t3) / (t3 @ t3)
    deg = 180 / np.pi
    assert np.isclose(r1[0], np.sqrt(np.trace(c[0:3, 0:3])) * deg) and np.isclose(r1[1], np.sqrt(np.trace(c[6:9, 6:9])) * deg)
    assert np.isclose(t1[0], np.sqrt(np.trace(c[3:6, 3:6])) * deg)
    assert np.isclose(t1[1], np.sqrt(np.trace(P @ c[9:12, 9:12] @ P) / (t3 @ t3)) * deg)


def test_predicted_errors_match_the_monte_carlo_angles(tvf):
    """pose_rms_errors at the truth == the RMS of AngError over 20 000 adjusted noise draws, within sampling error."""
    D = 20000
    CalM, Cr, Rt2, Rt3, X = truth_scene(20, 3)
    cov = tvf.ba_covariance(Cr, CalM, Rt2, Rt3, X)
    rot, tdir = tvf.pose_rms_errors(cov[0], Rt2, Rt3)
    rs = np.random.RandomState(5)
    res = tvf.bundle_adjust(Cr[None] + rs.standard_normal((D,) + Cr.shape), CalM, np.broadcast_to(Rt2, (D, 3, 4)),
                            np.broadcast_to(Rt3, (D, 3, 4)), np.broadcast_to(X, (D, 3, 20)))
    r2, t2 = tvf.AngError(Rt2, res[0]); r3, t3 = tvf.AngError(Rt3, res[1])
    emp_rot = np.sqrt([np.mean(r2 ** 2), np.mean(r3 ** 2)]); emp_t = np.sqrt([np.mean(t2 ** 2), np.mean(t3 ** 2)])
    print("predicted rot %s t %s; Monte Carlo rot %s t %s (degrees)" % (rot, tdir, emp_rot, emp_t))
    assert np.all(np.abs(emp_rot / rot - 1) < 0.03) and np.all(np.abs(emp_t / tdir - 1) < 0.03)


def test_run_real_with_covariance(tvf):
    from tft_vs_fund_b200 import epfl
    inp = np.load(os.path.join(ROOT, "tests", "golden", "epfl_inputs.npz"))
    for key in ("fountain_P11", "Herz_Jesu_P8"):
        data = epfl.dataset_from_arrays(inp[key + "_indexes_sorted"], inp[key + "_matches"], inp[key + "_offsets"],
                                        inp[key + "_K"], inp[key + "_R"], inp[key + "_t"])
        trips = range(1, 6)
        plain = epfl.run_real(data, trips, bundle_adjust=True)
        details = []
        cov = epfl.run_real(data, trips, details=details, bundle_adjust=True, covariance=True)
        for m in (1, 7):
            assert np.array_equal(cov[m], plain[m]), (key, m)
        for k in range(len(trips)):
            for m in (1, 7):
                ba = details[k]["ba"][m]
                assert np.isfinite(ba.sigma2) and ba.sigma2 > 0, (key, k, m)
                assert np.isfinite(ba.pred_rot_err) and ba.pred_rot_err > 0, (key, k, m)
                assert np.isfinite(ba.pred_t_err) and ba.pred_t_err > 0, (key, k, m)
        print("%s: sigma2 %s; predicted rot %s deg" % (key, [round(float(d["ba"][1].sigma2), 3) for d in details],
                                                       [round(d["ba"][1].pred_rot_err, 4) for d in details]))
