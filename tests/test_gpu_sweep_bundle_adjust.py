"""Bundle adjustment inside the device-resident sweeps (tvf_sweep_run_levels_ba) and the real-data driver: the method's
columns unchanged, the adjusted columns equal to the host twins and to the oracle's adjustment (oracle/bundle_adjust.py)."""
import os

import numpy as np
import pytest

import oracle as o
from oracle import bundle_adjust as oba
from conftest import ROOT

pytestmark = pytest.mark.gpu

TOL_PX = 1e-7        # mean ReprError, device against host twin and oracle
TOL_DEG = 1e-5       # mean AngError, device against host twin


def _levels(option):
    from tft_vs_fund_b200 import experiments
    _, params = experiments.experiment_levels(option)
    return experiments._sweep_levels(params), len(params)


def _table(h, name, method, first, count, levels, L):
    from tft_vs_fund_b200 import _lib
    t = np.zeros((L, 11 if name.endswith("_ba") else 5))
    h.call(name, method, first, count, levels, L, 1800.0, 1200.0, t.ctypes.data_as(_lib.c_double_p))
    return t


def test_method_columns_equal_tvf_sweep_run_levels_bit_for_bit(tvf):
    """With the same chunk size, columns 0-4 are exactly tvf_sweep_run_levels's table ('points': n varies per level,
    and methods 7 and 8 skip N = 7)."""
    from tft_vs_fund_b200 import _lib
    levels, L = _levels("points")
    h = _lib.handle(0)
    B = L * 40 + 3
    try:
        for chunk in (16, 1000):
            h.call("tvf_set_chunk", chunk)
            for m in (1, 7, 8):
                plain = _table(h, "tvf_sweep_run_levels", m, 0, B, levels, L)
                ba = _table(h, "tvf_sweep_run_levels_ba", m, 0, B, levels, L)
                assert np.array_equal(ba[:, :5], plain, equal_nan=True), (chunk, m)
                fin = np.isfinite(plain[:, 0])
                assert np.array_equal(np.isfinite(ba[:, 5]), fin) and np.all(ba[~fin, 8:] == 0.0), (chunk, m)
                assert np.array_equal(ba[fin, 8] + ba[fin, 9], ba[fin, 3] + ba[fin, 4]), (chunk, m)
    finally:
        h.call("tvf_set_chunk", 0)


@pytest.mark.parametrize("option", ["noise", "focal", "points", "angle"])
def test_device_equals_host_twin(tvf, option):
    """run_experiment(bundle_adjust=True) == run_experiment_host(bundle_adjust=True): skipped counts and mean iterations
    exact (a trial's pose and adjustment do not depend on its batch), means to rounding."""
    from tft_vs_fund_b200 import experiments
    n_sim = 6
    interval, dev = experiments.run_experiment(option, n_sim=n_sim, methods=(1, 7, 8), bundle_adjust=True)
    interval_h, host = experiments.run_experiment_host(option, n_sim=n_sim, methods=(1, 7, 8), bundle_adjust=True)
    assert list(interval) == list(interval_h)
    D, H = experiments.run_experiment, experiments.run_experiment_host
    for m in (1, 7, 8):
        assert dev[m].shape == host[m].shape == (len(interval), 6)
        assert np.array_equal(np.isfinite(dev[m]), np.isfinite(host[m])), m
        fin = np.isfinite(host[m][:, 0])
        assert np.array_equal(D.last_skipped[m], H.last_skipped[m]), m
        assert np.array_equal(D.last_skipped_ba[m], H.last_skipped_ba[m]), m
        assert np.array_equal(D.last_ba_iter[m], H.last_ba_iter[m], equal_nan=True), (m, D.last_ba_iter[m], H.last_ba_iter[m])
        for c0 in (0, 3):
            assert np.max(np.abs(dev[m][fin, c0] - host[m][fin, c0])) < TOL_PX, (m, c0)
            assert np.max(np.abs(dev[m][fin, c0 + 1:c0 + 3] - host[m][fin, c0 + 1:c0 + 3])) < TOL_DEG, (m, c0)
        assert np.all(np.isfinite(D.last_ba_iter[m][fin])) and np.all(D.last_ba_iter[m][fin] >= 1.0), m
    print("%s: mean BA iterations per level (method 1) %s; skipped after BA %s"
          % (option, np.round(D.last_ba_iter[1], 2), {m: int(v.sum()) for m, v in D.last_skipped_ba.items()}))


def test_run_sweep_device_equals_run_sweep(tvf):
    from tft_vs_fund_b200 import experiments
    total = 13 * 8
    dev = experiments.run_sweep_device(total, n=20, methods=(1, 7, 8), bundle_adjust=True)
    host = experiments.run_sweep(total, n=20, methods=(1, 7, 8), bundle_adjust=True)
    for m in (1, 7, 8):
        assert dev[m].shape == host[m].shape == (13, 6)
        assert np.array_equal(experiments.run_sweep_device.last_skipped[m], experiments.run_sweep.last_skipped[m])
        for c0 in (0, 3):
            assert np.max(np.abs(dev[m][:, c0] - host[m][:, c0])) < TOL_PX, (m, c0)
            assert np.max(np.abs(dev[m][:, c0 + 1:c0 + 3] - host[m][:, c0 + 1:c0 + 3])) < TOL_DEG, (m, c0)
    # the plain device sweep is untouched by the flag
    plain = experiments.run_sweep_device(total, n=20, methods=(1,))
    assert np.allclose(dev[1][:, :3], plain[1], rtol=1e-12, atol=0.0)


def test_sharded_ranges(tvf):
    """[0, B) == the sum of two ranges that cut through a seed's levels: counts and iteration sums exact."""
    from tft_vs_fund_b200 import _lib
    h = _lib.handle(0)
    for option in ("focal", "points"):
        levels, L = _levels(option)
        B = L * 40 + 7
        cut = L * 17 + 4
        whole = _table(h, "tvf_sweep_run_levels_ba", 1, 0, B, levels, L)
        parts = _table(h, "tvf_sweep_run_levels_ba", 1, 0, cut, levels, L) + \
            _table(h, "tvf_sweep_run_levels_ba", 1, cut, B - cut, levels, L)
        cnt = [3, 4, 8, 9, 10]
        assert np.array_equal(whole[:, cnt], parts[:, cnt]) and int(whole[:, 3].sum() + whole[:, 4].sum()) == B, option
        for c in (0, 1, 2, 5, 6, 7):
            assert np.max(np.abs(whole[:, c] - parts[:, c]) / np.abs(whole[:, c])) < 1e-12, (option, c)


@pytest.mark.parametrize("option", ["noise", "angle"])
def test_adjusted_means_match_the_oracle(tvf, option):
    """First and last level: every trial adjusted by oracle/bundle_adjust.py and evaluated with the oracle's AngError;
    averaged, it equals the device's after-adjustment means.  The oracle is trusted from starts below 10 px.  Where the
    oracle's own method-1 pose is such a start it adjusts that pose.  At N = 12 most linear-TFT starts of the 3 px and
    166 degree levels are 15-110 px off; there it starts from the library's adjusted pose (api.bundle_adjust, which the
    host-twin test ties to the device trial by trial) and must stay at that minimum."""
    from tft_vs_fund_b200 import experiments
    n_sim = 6
    _, dev = experiments.run_experiment(option, n_sim=n_sim, methods=(1,), bundle_adjust=True)
    _, params = experiments.experiment_levels(option)
    for lv in (0, len(params) - 1):
        p = params[lv]
        assert experiments.run_experiment.last_skipped_ba[1][lv] == 0, (option, lv)
        acc = np.zeros(3)
        from_oracle_pose = 0
        for it in range(1, n_sim + 1):
            CalM, R_t0, C, _ = o.experiments_subsample(p["N"], p["noise"], it, p["f"], p["angle"])
            Ks = [CalM[0:3], CalM[3:6], CalM[6:9]]
            start_err = lambda R2, R3, X: oba.repr_error(Ks, R2[:, :3], R2[:, 3], R3[:, :3], R3[:, 3], X, C)
            R2, R3, Rec, _, _ = o.LinearTFTPoseEstimation(C, CalM)
            if start_err(R2, R3, Rec) < 10.0:
                from_oracle_pose += 1
            else:
                r = tvf.LinearTFTPoseEstimation(C, CalM)
                R2, R3, Rec = tvf.bundle_adjust(C, CalM, r[0], r[1], r[2])[:3]
                assert start_err(R2, R3, Rec) < 10.0, (option, lv, it)           # the oracle's stated domain
            a2, a3, _, rep = oba.bundle_adjust(C, CalM, R2, R3, Rec)
            r2, t2 = o.AngError(R_t0[0], a2); r3, t3 = o.AngError(R_t0[1], a3)
            acc += np.array([rep, (r2 + r3) / 2, (t2 + t3) / 2]) / n_sim
        print("%s level %d: %d of %d trials adjusted from the oracle's own pose" % (option, lv, from_oracle_pose, n_sim))
        assert abs(dev[1][lv, 3] - acc[0]) < TOL_PX, (option, lv, dev[1][lv, 3], acc[0])
        assert np.max(np.abs(dev[1][lv, 4:] - acc[1:])) < 1e-4, (option, lv, dev[1][lv, 4:], acc[1:])


def test_run_real_with_bundle_adjust(tvf):
    """epfl.run_real(bundle_adjust=True) on the first 5 triplets of each dataset: the method columns are those of the
    plain call, bit for bit; the adjusted columns equal the oracle's adjustment of the same start, evaluated with the
    oracle's ReprError over all inliers and AngError."""
    from tft_vs_fund_b200 import epfl
    inp = np.load(os.path.join(ROOT, "tests", "golden", "epfl_inputs.npz"))
    for key in ("fountain_P11", "Herz_Jesu_P8"):
        data = epfl.dataset_from_arrays(inp[key + "_indexes_sorted"], inp[key + "_matches"], inp[key + "_offsets"],
                                        inp[key + "_K"], inp[key + "_R"], inp[key + "_t"])
        trips = range(1, 6)
        plain = epfl.run_real(data, trips)
        details = []
        ba = epfl.run_real(data, trips, details=details, bundle_adjust=True)
        for m in (1, 7):
            assert ba[m].shape == (5, 6)
            assert np.array_equal(ba[m][:, :3], plain[m]), (key, m)
        for k, trip in enumerate(trips):
            d = epfl.prepare_triplet(data, trip)
            inl, CalM, R_t0 = d["Corresp_inliers"], d["CalM"], d["R_t0"]
            C0 = inl[:, details[k]["sample"]]
            Ks = [CalM[0:3], CalM[3:6], CalM[6:9]]
            for m in (1, 7):
                res = details[k]["res"][m]
                start = oba.repr_error(Ks, res[0][:, :3], res[0][:, 3], res[1][:, :3], res[1][:, 3], res[2], C0)
                assert start < 10.0, (key, trip, m, start)
                a2, a3, _, _ = oba.bundle_adjust(C0, CalM, res[0], res[1], res[2])
                rep = o.ReprError([Ks[0] @ np.eye(3, 4), Ks[1] @ a2, Ks[2] @ a3], inl)
                r2, t2 = o.AngError(R_t0[0], a2); r3, t3 = o.AngError(R_t0[1], a3)
                got = ba[m][k, 3:]
                assert abs(got[0] - rep) < 1e-6, (key, trip, m, got[0], rep)
                assert np.max(np.abs(got[1:] - [(r2 + r3) / 2, (t2 + t3) / 2])) < 1e-4, (key, trip, m)
                assert not details[k]["ba"][m].status & tvf._lib.ST_NONFINITE, (key, trip, m)


def test_argument_errors_before_device_work(tvf):
    from tft_vs_fund_b200 import _lib
    h = _lib.handle(0)
    levels, L = _levels("noise")
    t = np.zeros((L, 11))
    tp = t.ctypes.data_as(_lib.c_double_p)
    fn = lambda *a: h.lib.tvf_sweep_run_levels_ba(h._h, *a)
    before = h.lib.tvf_launch_count(h._h)
    assert fn(2, 0, 26, levels, L, 1800.0, 1200.0, tp) == _lib.TVF_ERR_ARG
    assert fn(1, 0, 26, levels, L, 1800.0, 1200.0, None) == _lib.TVF_ERR_ARG
    levels[3].n = 61
    assert fn(1, 0, 26, levels, L, 1800.0, 1200.0, tp) == _lib.TVF_ERR_ARG
    assert h.lib.tvf_launch_count(h._h) == before
    assert np.all(t == 0.0)
