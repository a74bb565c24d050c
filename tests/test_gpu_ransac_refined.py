"""tvf_ransac_pose_refined on the GPU: the result rebuilt from public calls bit for bit (which also shows that the packed
small-n adjustment equals bundle_adjust_kernel), invariances, the CPU oracle (tests/ransac_refined_oracle.py),
robustness on synthetic scenes with 30 % and 50 % outliers, the raw-match mode of epfl.run_real, and edge cases."""
import ctypes as C

import numpy as np
import pytest

import oracle as o
import ransac_oracle as ro
import ransac_refined_oracle as rr
from conftest import assert_pose_close
from test_gpu_ransac import composition_cases, epfl_dataset, pose_batch, same

pytestmark = pytest.mark.gpu

ST_NONFINITE = 16


def rebuild(tvf, method, Cr, CalM, H, th, seed, lo_rounds):
    """The refined result of one problem from public calls: every hypothesis by tvf_pose, adjusted on its sample by
    tvf_bundle_adjust (reconst0 NULL) and scored by tvf_consensus; the best (ties to the smallest h); LO rounds of
    tvf_bundle_adjust + tvf_consensus on the current consensus; the rule of include/tvf.h."""
    s = ro.SAMPLE_SIZE[method]
    idx = ro.sample(seed, np.arange(H), Cr.shape[1], s)
    S = np.stack([Cr[:, i] for i in idx])
    R2, R3, st = pose_batch(tvf, method, S, CalM)
    ba = tvf.bundle_adjust(S, CalM, R2, R3)
    _, cnt = tvf.consensus(np.broadcast_to(Cr, (H,) + Cr.shape), CalM, ba[0], ba[1], threshold=th)
    cnt = np.where((st != 0) | (ba.status & ST_NONFINITE != 0), -1, cnt)
    h = int(np.argmax(cnt))
    if cnt[h] < 0:
        return np.full((3, 4), np.nan), np.full((3, 4), np.nan), np.zeros(Cr.shape[1], bool), 0, np.full(s, -1), 0, 128
    P2, P3 = ba[0][h], ba[1][h]
    mask, c = tvf.consensus(Cr, CalM, P2, P3, threshold=th)
    done = 0
    for _ in range(lo_rounds):
        if c < 4:
            break
        r = tvf.bundle_adjust(Cr[:, mask], CalM, P2, P3)
        if r.status & ST_NONFINITE:
            break
        m2, c2 = tvf.consensus(Cr, CalM, r[0], r[1], threshold=th)
        if not c2 > c:
            break
        P2, P3, mask, c, done = r[0], r[1], m2, c2, done + 1
    return P2, P3, mask, c, idx[h], done, 0


def refined(tvf, Cr, CalM, **kw):
    res = tvf.ransac_pose(Cr, CalM, refine=True, **kw)
    return list(res) + [res.lo_done, res.status]


@pytest.mark.parametrize("method", [1, 7])
def test_result_is_composed_of_public_calls(tvf, method):
    H = 24
    for label, Cr, CalM in composition_cases():
        n = Cr.shape[2]
        if n < ro.SAMPLE_SIZE[method]:
            continue
        if method == 1 and n == 8:                 # n = s for the TFT method
            Cr = Cr[:, :, :7]
        got = refined(tvf, Cr, CalM, method=method, hypotheses=H, threshold=2.0, seed=11, lo_rounds=4)
        for b in range(Cr.shape[0]):
            want = rebuild(tvf, method, Cr[b], CalM, H, 2.0, 11 + b, 4)
            assert same([x[b] for x in got], want), (label, b)


def test_invariances(tvf):
    import torch
    from tft_vs_fund_b200 import _lib
    Cr, CalM, _, _ = ro.outlier_scenes(0.3, 30, 41)
    CalMb = np.broadcast_to(CalM, (30, 9, 3)).copy()
    kw = dict(method=1, hypotheses=40, threshold=3.0, lo_rounds=8)
    full = refined(tvf, Cr, CalMb, seed=5, **kw)
    assert np.any(full[5] > 0)
    for b in (0, 13, 29):
        one = refined(tvf, Cr[b:b + 1], CalMb[b:b + 1], seed=5 + b, **kw)
        assert same([x[b:b + 1] for x in full], one), b
    h = _lib.handle()
    try:
        h.call("tvf_set_chunk", 7)
        chunked = refined(tvf, Cr, CalMb, seed=5, **kw)
    finally:
        h.call("tvf_set_chunk", 0)
    assert same(full, chunked)
    assert same(full, refined(tvf.api, Cr, CalMb, seed=5, device=(0, 0), **kw))
    # _dev == host
    dev = torch.device("cuda", 0)
    B, n = Cr.shape[0], Cr.shape[2]
    d_c = torch.from_numpy(tvf.api._cm(Cr, 2)[0]).to(dev)
    d_m = torch.from_numpy(tvf.api._cm(CalMb, 2)[0]).to(dev)
    d_s = torch.from_numpy((np.uint64(5) + np.arange(B, dtype=np.uint64)).view(np.int64)).to(dev)
    o2 = torch.empty((B, 12), dtype=torch.float64, device=dev); o3 = torch.empty_like(o2)
    om = torch.zeros((B, n), dtype=torch.uint8, device=dev); oc = torch.zeros(B, dtype=torch.int32, device=dev)
    osm = torch.zeros((B, 7), dtype=torch.int32, device=dev); ost = torch.zeros(B, dtype=torch.int32, device=dev)
    olo = torch.zeros(B, dtype=torch.int32, device=dev)
    p = lambda t: C.c_void_p(t.data_ptr())
    torch.cuda.synchronize()
    h.call("tvf_ransac_pose_refined_dev", 1, p(d_c), p(d_m), 1, n, B, 40, 3.0, p(d_s), 8, p(o2), p(o3), p(om), p(oc),
           p(osm), p(olo), p(ost))
    h.call("tvf_synchronize")
    back = lambda t: tvf.api._from_cm(t.cpu().numpy().ravel(), B, (3, 4), True)
    dev_res = [back(o2), back(o3), om.cpu().numpy().astype(bool), oc.cpu().numpy(), osm.cpu().numpy(),
               olo.cpu().numpy(), ost.cpu().numpy()]
    assert same(full, dev_res)


@pytest.mark.parametrize("method", [1, 7])
def test_against_the_oracle(tvf, method):
    """Noise-free inliers: sample, n_inliers, inliers and lo_done equal the oracle's wherever no match of a competitive
    hypothesis or of an LO round lies within 1e-6 px of the threshold; where the winning sample is free of outliers the
    adjusted pose is the true one in both, and the poses agree to the parity tolerances.  (A sample with an outlier
    adjusts to a pose that depends on where each minimiser stops, so its pose is not compared.)"""
    H, th = 16, 2.0
    Cr, CalM, _, out = ro.outlier_scenes(0.2, 10, 31, noise=0.0)
    Cr, out = Cr[:, :, :32], out[:, :32]
    got = refined(tvf, Cr, CalM, method=method, hypotheses=H, threshold=th, seed=100, lo_rounds=8)
    clean = 0
    for b in range(Cr.shape[0]):
        want = rr.ransac_refined(Cr[b], CalM, method, H, th, 100 + b)
        if rr.near_threshold(want, 1e-6) or want["status"] != 0 or out[b][want["sample"]].any():
            continue
        clean += 1
        assert got[6][b] == 0
        assert np.array_equal(got[4][b], want["sample"]) and got[3][b] == want["n_inliers"], b
        assert np.array_equal(got[2][b], want["inliers"]) and got[5][b] == want["lo_done"], b
        fn = lambda R2, R3: (R2, R3, np.zeros((3, 1)), o.TFT_from_P(CalM[0:3] @ np.eye(3, 4), CalM[3:6] @ R2, CalM[6:9] @ R3), 0.0)
        assert_pose_close(fn(want["Rt2"], want["Rt3"]), fn(got[0][b], got[1][b]), "problem %d" % b)
    print("method %d: %d of %d problems compared" % (method, clean, Cr.shape[0]))
    assert clean >= 0.7 * Cr.shape[0]


# Bounds from the CPU oracle (tests/ransac_refined_oracle.py) on ro.outlier_scenes(f, count, 51) (n = 100, 1 px noise,
# H = ro.hypotheses_for(f, s), threshold 2 px, seed 1000 + b), the reference being the adjustment on the true inliers
# from the true pose.  30 % outliers, 3 scenes: recall 0.94-0.97 (mean 0.957) for methods 1 and 7, precision 1.0, median
# rotation error 1.96 x (method 1) and 1.58 x (method 7) the reference's.  50 % outliers, 2 scenes: recall 0.90 / 0.98
# (method 1) and 0.84 / 1.0 (method 7), precision 1.0, median ratio 1.02 and 1.92.  The bounds leave room for the 30
# scenes tested here.
ROBUST_BOUNDS = {0.3: dict(recall=0.85, precision=0.95, ratio=3.0), 0.5: dict(recall=0.80, precision=0.95, ratio=3.0)}


@pytest.mark.parametrize("f", [0.3, 0.5])
@pytest.mark.parametrize("method", [1, 7])
def test_robustness(tvf, method, f):
    count, th = 30, 2.0
    Cr, CalM, R_t0, out = ro.outlier_scenes(f, count, 51)
    H = ro.hypotheses_for(f, ro.SAMPLE_SIZE[method])
    got = refined(tvf, Cr, CalM, method=method, hypotheses=H, threshold=th, seed=1000, lo_rounds=8)
    assert np.all(got[6] == 0)
    truth = ~out
    rot, rref, rec, prec = [], [], [], []
    for b in range(count):
        rot.append((o.AngError(R_t0[0], got[0][b])[0] + o.AngError(R_t0[1], got[1][b])[0]) / 2)
        r = tvf.bundle_adjust(Cr[b][:, truth[b]], CalM, R_t0[0], R_t0[1])
        rref.append((o.AngError(R_t0[0], r[0])[0] + o.AngError(R_t0[1], r[1])[0]) / 2)
        tp = np.sum(got[2][b] & truth[b])
        rec.append(tp / truth[b].sum()); prec.append(tp / max(1, got[2][b].sum()))
    ratio = np.median(rot) / np.median(rref)
    print("method %d, %d %% outliers, H = %d: recall %.3f precision %.3f median rot err %.3f deg (%.2f x the adjustment on "
          "the true inliers), LO rounds %s" % (method, 100 * f, H, np.mean(rec), np.mean(prec), np.median(rot), ratio,
                                               np.bincount(got[5])))
    bnd = ROBUST_BOUNDS[f]
    assert np.mean(rec) >= bnd["recall"] and np.mean(prec) >= bnd["precision"] and ratio <= bnd["ratio"]


# run_real(raw_matches=True, ransac_refine=True) on the triplets of test_gpu_ransac.test_run_real_raw_matches (1024
# hypotheses, 1 px).  Measured on the GPU (NVIDIA B200): per-triplet recall 0.978-1.0 and precision 0.967-0.999 over both
# datasets and methods 1 / 7; the unrefined estimator's recall bound there is 0.002.  The SciPy oracle was not run on
# these triplets: 1024 adjusted hypotheses per triplet take it minutes each.
REFINED_RECALL_MIN = 0.9
REFINED_MEAN_RECALL_MIN = 0.95
REFINED_PRECISION_MIN = 0.9


def test_run_real_raw_matches_refined(tvf):
    from tft_vs_fund_b200 import epfl
    for key in ("fountain_P11", "Herz_Jesu_P8"):
        data = epfl_dataset(key)
        trips = range(1, 6)
        plain = epfl.run_real(data, trips, raw_matches=True)
        details = []
        raw = epfl.run_real(data, trips, details=details, raw_matches=True, ransac_refine=True)
        again = epfl.run_real(data, trips, raw_matches=True)
        assert all(np.array_equal(plain[m], again[m]) for m in (1, 7))            # the default path is unaffected
        rec = [details[k]["consensus"][m]["recall"] for k in range(len(trips)) for m in (1, 7)]
        prec = [details[k]["consensus"][m]["precision"] for k in range(len(trips)) for m in (1, 7)]
        print("%s refined raw matches: recall %s precision %s rot err %s" % (
            key, np.round(rec, 3), np.round(prec, 3), {m: np.round(raw[m][:, 1], 3) for m in (1, 7)}))
        assert min(rec) >= REFINED_RECALL_MIN and np.mean(rec) >= REFINED_MEAN_RECALL_MIN, rec
        assert min(prec) >= REFINED_PRECISION_MIN, prec
        for m in (1, 7):
            assert np.all(np.isfinite(raw[m][:, :3])), (key, m)
            assert all(details[k]["res"][m].lo_done >= 0 for k in range(len(trips)))


def test_edge_cases(tvf):
    from tft_vs_fund_b200 import _lib
    d = tvf.sweep_batch(6, 40, noise_levels=[1.0])
    Cr, CalM = d["Corresp"].copy(), d["CalM"]
    # n = s: every hypothesis is the whole set, adjusted
    for method, s in ((1, 7), (7, 8)):
        got = refined(tvf, Cr[:, :, :s], CalM, method=method, hypotheses=5, threshold=1.0, seed=3, lo_rounds=8)
        want = [rebuild(tvf, method, Cr[b][:, :s], CalM, 5, 1.0, 3 + b, 8) for b in range(6)]
        assert all(same([x[b] for x in got], want[b]) for b in range(6))
        assert np.all(np.sort(got[4], axis=1) == np.arange(s))
    # an all-NaN problem fails and leaves its neighbours as they are without it
    Cr[2] = np.nan
    kw = dict(method=1, hypotheses=30, threshold=3.0, lo_rounds=8)
    got = refined(tvf, Cr, CalM, seed=1, **kw)
    ref = refined(tvf, np.delete(Cr, 2, axis=0), CalM, seed=np.delete(np.arange(1, 7, dtype=np.uint64), 2), **kw)
    assert got[6][2] == _lib.ST_RANSAC_FAILED and got[5][2] == 0 and got[3][2] == 0
    assert np.all(np.isnan(got[0][2])) and np.all(np.isnan(got[1][2])) and not got[2][2].any() and np.all(got[4][2] == -1)
    keep = [0, 1, 3, 4, 5]
    assert same([x[keep] for x in got], ref)
    # lo_rounds outside 0 .. 32
    for lo in (-1, 33):
        with pytest.raises(_lib.TvfError, match="lo_rounds"):
            tvf.ransac_pose(Cr, CalM, method=1, hypotheses=4, refine=True, lo_rounds=lo)
    # lo_rounds = 0: the adjusted winner
    zero = refined(tvf, Cr[:1], CalM, method=1, hypotheses=30, threshold=3.0, seed=1, lo_rounds=0)
    assert same([x[0] for x in zero], rebuild(tvf, 1, Cr[0], CalM, 30, 3.0, 1, 0))
    # NULL outputs: every output may be NULL
    from tft_vs_fund_b200 import api
    h = _lib.handle()
    c, _, B = api._cm(Cr[3:5], 2)
    calm, cb = api._calm(CalM, B)
    seeds = np.arange(B, dtype=np.uint64)
    h.call("tvf_ransac_pose_refined", 1, api._p(c), api._p(calm), cb, c.shape[1], B, 8, 3.0, api._vp(seeds), 4,
           None, None, None, None, None, None, None)
