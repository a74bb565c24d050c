"""The refined RANSAC rule (tvf_ransac_pose_refined, include/tvf.h) on its CPU oracle, tests/ransac_refined_oracle.py:
the rule's invariants on small problems with noise-free inliers."""
import numpy as np
import pytest

import ransac_oracle as ro
import ransac_refined_oracle as rr


def problems():
    """Two 30-match problems at 1 px with 20 % outliers; on the second, method 1's LO rounds raise the count 16 -> 21 -> 23."""
    Cr, CalM, _, out = ro.outlier_scenes(0.2, 3, 61, noise=1.0)
    return [(Cr[b][:, :30], CalM, out[b][:30]) for b in (0, 1)]


@pytest.mark.parametrize("method", [1, 7])
def test_rule_invariants(method):
    H, th, s = 10, 1.5, ro.SAMPLE_SIZE[method]
    for k, (Cr, CalM, _) in enumerate(problems()):
        res = rr.ransac_refined(Cr, CalM, method, H, th, 7 + k)
        assert res["status"] == 0
        if method == 1 and k == 1:
            assert res["lo_done"] == 2
        # the sampler is tvf_ransac_pose's, and the sample is the winner's
        assert np.array_equal(res["sample"], ro.sample(7 + k, np.arange(H), Cr.shape[1], s)[res["best"]])
        # the winner has the largest score, the first of equal scores
        assert res["best"] == int(np.argmax(res["counts"]))
        # LO counts grow strictly, one accepted round per step, and the result is the last of them
        lc = res["lo_counts"]
        assert lc[0] == res["counts"][res["best"]] and np.all(np.diff(lc) > 0)
        assert res["lo_done"] == len(lc) - 1 and res["n_inliers"] == lc[-1] == int(res["inliers"].sum())
        mask, _ = ro.inliers(Cr, CalM, res["Rt2"], res["Rt3"], th)
        assert np.array_equal(mask, res["inliers"])
        # lo_rounds = 0: the adjusted winner itself
        zero = rr.ransac_refined(Cr, CalM, method, H, th, 7 + k, lo_rounds=0)
        assert zero["lo_done"] == 0 and zero["best"] == res["best"]
        idx = zero["sample"]
        want = rr.adjust(Cr[:, idx], CalM, *ro.solve(method, Cr[:, idx], CalM))
        assert np.array_equal(zero["Rt2"], want[0]) and np.array_equal(zero["Rt3"], want[1])
        assert zero["n_inliers"] == res["counts"][res["best"]]


def test_failed_problem():
    Cr, CalM, _ = problems()[0]
    res = rr.ransac_refined(np.full_like(Cr, np.nan), CalM, 1, 4, 2.0, 3)
    assert res["status"] == 128 and res["lo_done"] == 0 and res["n_inliers"] == 0
    assert np.all(res["sample"] == -1) and np.all(np.isnan(res["Rt2"])) and not res["inliers"].any()
