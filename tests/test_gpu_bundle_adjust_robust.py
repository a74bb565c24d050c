"""tvf_bundle_adjust_robust on the GPU against the CPU oracle (tests/ba_robust_oracle.py), its consistency with the
plain adjustment, its invariances, its robustness to outliers and its edge cases."""
import ctypes as C

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

import oracle as o
import ba_robust_oracle as bro
import distinct_k as dk
import ransac_oracle as ro
from conftest import rot_angle, vec_angle

pytestmark = pytest.mark.gpu

TOL_ANG = 1e-6       # rad, R and t directions
TOL_REL = 1e-7       # |t3| and Reconst, relative
TOL_COST = 1e-10     # cost, relative
# weights, absolute.  The IRLS model has no rho'' term, so near the minimum the kernel converges linearly (on Huber's
# linear branch the model doubles the curvature along each match's residual) and stops on the 1e-15 relative cost change
# of tvf_bundle_adjust's rule: a cost gap of ~1e-15 of the cost leaves residuals ~1e-7 px from the stationary point,
# weights ~1e-7 (measured on the B200: 2.3e-7 at f = 0, Huber, c = 1 px), while poses, points and cost agree well
# inside their tolerances
TOL_W = 1e-6


def perturbed_truth(CalM, R_t0, Cr, rs, rot=1e-3, rel=1e-3):
    """The true state (|t2| = 1, points triangulated with the true cameras) perturbed as
    test_bundle_adjust_cpu.perturbed does (a factor 2 of scale included)."""
    K1, K2, K3 = CalM[0:3], CalM[3:6], CalM[6:9]
    Xh = o.triangulation3D([K1 @ np.eye(3, 4), K2 @ R_t0[0], K3 @ R_t0[1]], Cr)
    s = 1.0 / np.linalg.norm(R_t0[0][:, 3])
    X = Xh[:3] / Xh[3] * s
    dR = lambda: Rotation.from_rotvec(rs.standard_normal(3) * rot / np.sqrt(3)).as_matrix()
    t2 = R_t0[0][:, 3] * s + rel * rs.standard_normal(3)
    return (np.column_stack([dR() @ R_t0[0][:, :3], t2 * 2.0]),
            np.column_stack([dR() @ R_t0[1][:, :3], (R_t0[1][:, 3] * s + rel * rs.standard_normal(3)) * 2.0]),
            (X + rel * rs.standard_normal(X.shape)) * 2.0)


def compare(res, b, ref, tag):
    r2, r3, rX, cost, w, _ = ref
    g2, g3, gX = res[0][b], res[1][b], res[2][b]
    assert res.status[b] == 0, tag
    for a, c in ((r2, g2), (r3, g3)):
        assert rot_angle(a[:, :3], c[:, :3]) < TOL_ANG, tag
        assert vec_angle(a[:, 3], c[:, 3]) < TOL_ANG, tag
    assert abs(np.linalg.norm(g3[:, 3]) - np.linalg.norm(r3[:, 3])) <= TOL_REL * np.linalg.norm(r3[:, 3]), tag
    assert np.abs(gX - rX).max() <= TOL_REL * np.abs(rX).max(), tag
    assert abs(res.cost[b] - cost) <= TOL_COST * cost, (tag, res.cost[b], cost)
    assert np.abs(res.weights[b] - w).max() <= TOL_W, tag


def run_parity(tvf, Cs, Ms, starts, losses, scales, label):
    Cr = np.stack(Cs); CalM = np.stack(Ms)
    S2 = np.stack([s[0] for s in starts]); S3 = np.stack([s[1] for s in starts]); SX = np.stack([s[2] for s in starts])
    for loss in losses:
        for c in scales:
            res = tvf.bundle_adjust(Cr, CalM, S2, S3, SX, loss=loss, scale=c)
            for b in range(Cr.shape[0]):
                ref = bro.bundle_adjust_robust(Cr[b], CalM[b], S2[b], S3[b], SX[b], loss, c)
                compare(res, b, ref, "%s %s c=%g problem %d" % (label, loss, c, b))


@pytest.mark.parametrize("f", [0.0, 0.1, 0.3])
def test_matches_oracle_on_outlier_scenes(tvf, f):
    Cr, CalM, R_t0, _ = ro.outlier_scenes(f, 2, 17)
    rs = np.random.RandomState(int(10 * f))
    starts = [perturbed_truth(CalM, R_t0, Cr[b], rs) for b in range(2)]
    run_parity(tvf, list(Cr), [CalM] * 2, starts, bro.LOSSES, (1.0, 3.0), "f=%g" % f)


@pytest.mark.parametrize("n", [4, 7, 20, 100, 500])
def test_matches_oracle_at_several_sizes(tvf, n):
    rs = np.random.RandomState(n)
    Cs, Ms, starts = [], [], []
    for seed in ((1, 2) if n <= 100 else (1,)):
        CalM, R_t0, Cr, _ = o.experiments_subsample(n, 1.0, seed)
        Cs.append(Cr); Ms.append(CalM); starts.append(perturbed_truth(CalM, R_t0, Cr, rs))
    run_parity(tvf, Cs, Ms, starts, bro.LOSSES, (1.0, 3.0) if n <= 100 else (3.0,), "n=%d" % n)


def test_distinct_intrinsics_per_view_and_problem(tvf):
    """K1, K2, K3 differ per view and per problem (tests/distinct_k.py, 20 % outliers): the oracle agrees, and the same
    call with K2 and K3 swapped does not."""
    Cr, CalM, R_t0, _ = dk.outlier_scenes(0.2, 3, 40, n=40)
    rs = np.random.RandomState(3)
    starts = [perturbed_truth(CalM[b], R_t0[b], Cr[b], rs) for b in range(3)]
    S2, S3, SX = (np.stack([s[k] for s in starts]) for k in range(3))
    res = tvf.bundle_adjust(Cr, CalM, S2, S3, SX, loss="cauchy", scale=2.0)
    swapped = tvf.bundle_adjust(Cr, dk.wrong_k(CalM)["K2 and K3 swapped"], S2, S3, SX, loss="cauchy", scale=2.0)
    for b in range(3):
        ref = bro.bundle_adjust_robust(Cr[b], CalM[b], S2[b], S3[b], SX[b], "cauchy", 2.0)
        compare(res, b, ref, "distinct K problem %d" % b)
        with pytest.raises(AssertionError):
            compare(swapped, b, ref, "swapped")


def test_huber_with_a_huge_scale_is_the_plain_adjustment(tvf):
    """Huber at c = 1e6 px: every match on the quadratic branch (weight exactly 1), so tvf_bundle_adjust's problem; a
    different kernel contracts differently, so equal to 1e-12, not bit for bit.  The cost never exceeds the start's."""
    g = np.load(__import__("os").path.join(__import__("conftest").ROOT, "tests", "golden", "sweep_n20.npz"))
    Cr, CalM = g["Corresp"][:60], g["CalM"][:60]
    Rt2, Rt3, X = g["tft_Rt2"][:60], g["tft_Rt3"][:60], g["tft_Reconst"][:60]
    plain = tvf.bundle_adjust(Cr, CalM, Rt2, Rt3, X)
    rob = tvf.bundle_adjust(Cr, CalM, Rt2, Rt3, X, loss="huber", scale=1e6)
    assert np.all(rob.weights == 1.0) and np.array_equal(rob.status, plain.status)
    ok = plain.status == 0
    for k in (0, 1, 2):
        d = np.abs(np.asarray(rob[k]) - np.asarray(plain[k]))[ok].reshape(int(ok.sum()), -1).max(1)
        m = np.abs(np.asarray(plain[k]))[ok].reshape(int(ok.sum()), -1).max(1)
        assert np.all(d <= 1e-12 * m), k
    assert np.all(np.abs(rob.repr_err - plain.repr_err)[ok] <= 1e-12 * plain.repr_err[ok])
    assert np.all(np.abs(rob.cost - 3 * 20 * rob.repr_err ** 2)[ok] <= 1e-12 * rob.cost[ok])
    for loss in bro.LOSSES:
        r = tvf.bundle_adjust(Cr, CalM, Rt2, Rt3, X, loss=loss, scale=1.0)
        for b in range(60):
            start = bro.Problem(Cr[b], CalM[b], Rt2[b], Rt3[b], X[b], loss, 1.0)
            if r.status[b] & tvf._lib.ST_NONFINITE:
                continue
            assert r.cost[b] <= start.cost(start.p0) * (1 + 1e-12), (loss, b)


# ---- bit-identity ---------------------------------------------------------------------------------------------------
def _outs(r):
    return (r[0], r[1], r[2], r[3], r.repr_err, r.status, r.cost, r.weights)


def _bits_equal(a, b):
    return all(np.array_equal(np.asarray(x), np.asarray(y), equal_nan=True) for x, y in zip(a, b))


def test_bit_identity_across_batch_chunk_group_and_device_pointers(tvf):
    import torch
    from tft_vs_fund_b200 import _lib
    Cr, CalM, R_t0, _ = ro.outlier_scenes(0.2, 24, 5)
    start = tvf.LinearTFTPoseEstimation(Cr, CalM)
    Rt2, Rt3, X = start[0], start[1], start[2]
    kw = dict(loss="cauchy", scale=2.0)
    full = tvf.bundle_adjust(Cr, CalM, Rt2, Rt3, X, **kw)
    for b in (0, 11, 23):
        one = tvf.bundle_adjust(Cr[b:b + 1], CalM, Rt2[b:b + 1], Rt3[b:b + 1], X[b:b + 1], **kw)
        assert _bits_equal([np.asarray(x)[b:b + 1] for x in _outs(full)], _outs(one)), b
    h = _lib.handle()
    try:
        h.call("tvf_set_chunk", 5)
        chunked = tvf.bundle_adjust(Cr, CalM, Rt2, Rt3, X, **kw)
    finally:
        h.call("tvf_set_chunk", 0)
    assert _bits_equal(_outs(full), _outs(chunked))
    assert _bits_equal(_outs(full), _outs(tvf.api.bundle_adjust(Cr, CalM, Rt2, Rt3, X, device=(0, 0), **kw)))
    # NULL outputs: the rest unchanged
    B, n = Cr.shape[0], Cr.shape[2]
    cm = lambda a: tvf.api._cm(a, 2)[0]
    c, r2, r3, x0 = cm(Cr), cm(Rt2), cm(Rt3), cm(X)
    calm = np.ascontiguousarray(CalM.T)
    o2 = np.empty((B, 12)); o3 = np.empty((B, 12))
    dp = lambda a: a.ctypes.data_as(_lib.c_double_p)
    h.call("tvf_bundle_adjust_robust", dp(c), dp(calm), 0, n, B, 3, C.c_double(2.0), dp(r2), dp(r3), dp(x0), dp(o2), dp(o3),
           None, None, None, None, None, None)
    assert np.array_equal(tvf.api._from_cm(o2, B, (3, 4), True), full[0])
    assert np.array_equal(tvf.api._from_cm(o3, B, (3, 4), True), full[1])
    # _dev == host
    dev = torch.device("cuda", 0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    d_c, d_m, d_r2, d_r3, d_x = t(c), t(calm), t(r2), t(r3), t(x0)
    e = lambda *s: torch.empty(s, dtype=torch.float64, device=dev)
    O2, O3, OX, OR, OC, OW = e(B, 12), e(B, 12), e(B, 3 * n), e(B), e(B), e(B, n)
    OI = torch.zeros(B, dtype=torch.int32, device=dev); OS = torch.zeros(B, dtype=torch.int32, device=dev)
    p = lambda x: C.c_void_p(x.data_ptr())
    torch.cuda.synchronize()
    h.call("tvf_bundle_adjust_robust_dev", p(d_c), p(d_m), 0, n, B, 3, C.c_double(2.0), p(d_r2), p(d_r3), p(d_x), p(O2),
           p(O3), p(OX), p(OR), p(OC), p(OW), p(OI), p(OS))
    h.call("tvf_synchronize")
    back = lambda x, dims: tvf.api._from_cm(x.cpu().numpy().ravel(), B, dims, True)
    got = (back(O2, (3, 4)), back(O3, (3, 4)), back(OX, (3, n)), OI.cpu().numpy(), OR.cpu().numpy(), OS.cpu().numpy(),
           OC.cpu().numpy(), OW.cpu().numpy())
    assert _bits_equal(_outs(full), got)


def test_ragged_equals_uniform_on_each_problem(tvf):
    """n_b in {0, 3, 4, 31, 32, 33, 100, 1400}, shuffled, through the host form (chunked and not) and the _dev form:
    every problem of n_b >= 4 equals the uniform call on it alone, bit for bit; n_b < 4 is TVF_ST_TOO_FEW_MATCHES with
    NaN cost and weights."""
    import torch
    from tft_vs_fund_b200 import _lib
    sizes = [0, 3, 4, 31, 32, 33, 100, 1400]
    order = np.random.RandomState(2).permutation(len(sizes))
    sizes = [sizes[k] for k in order]
    Cs, starts = [], []
    CalM = None
    for k, n in enumerate(sizes):
        CalM, R_t0, Cr, _ = o.experiments_subsample(max(n, 8), 1.0, 10 + k)    # one CalM for every seed of the sweep
        Cr = Cr[:, :n]
        starts.append(perturbed_truth(CalM, R_t0, Cr, np.random.RandomState(k)) if n > 0
                      else (R_t0[0], R_t0[1], np.zeros((3, 0))))
        Cr = Cr.copy()
        if n >= 8:                                     # a fifth of the matches replaced by uniform pixels
            rs = np.random.RandomState(k)
            cols = rs.choice(n, n // 5, replace=False)
            Cr[0::2, cols] = rs.uniform(0, 1800, (3, cols.size)); Cr[1::2, cols] = rs.uniform(0, 1200, (3, cols.size))
        Cs.append(Cr)
    S2 = np.stack([s[0] for s in starts]); S3 = np.stack([s[1] for s in starts])
    kw = dict(loss="soft_l1", scale=1.5)
    rag = tvf.bundle_adjust(Cs, CalM, S2, S3, [s[2] for s in starts], **kw)
    h = _lib.handle()
    try:
        h.call("tvf_set_chunk", 3)
        rag_c = tvf.bundle_adjust(Cs, CalM, S2, S3, [s[2] for s in starts], **kw)
    finally:
        h.call("tvf_set_chunk", 0)
    for b, n in enumerate(sizes):
        for r in (rag, rag_c):
            if n < 4:
                assert r.status[b] == tvf._lib.ST_TOO_FEW_MATCHES and np.isnan(r.cost[b]) and np.all(np.isnan(r.weights[b]))
                assert np.array_equal(r[0][b], S2[b]) and np.array_equal(r[1][b], S3[b])
                continue
            one = tvf.bundle_adjust(Cs[b], CalM, S2[b], S3[b], starts[b][2], **kw)
            assert np.array_equal(r[0][b], one[0]) and np.array_equal(r[1][b], one[1]), (b, n)
            assert np.array_equal(r[2][b], one[2]) and r[3][b] == one[3] and r.status[b] == one.status, (b, n)
            assert r.repr_err[b] == one.repr_err and r.cost[b] == one.cost and np.array_equal(r.weights[b], one.weights)
    # _dev form
    c, offs = tvf.api._pack(Cs, 6)
    x0, _ = tvf.api._pack([s[2] for s in starts], 3)
    r2, r3 = tvf.api._pose_pair(S2, S3, len(sizes), True)
    calm = np.ascontiguousarray(CalM.T)
    dev = torch.device("cuda", 0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    B, m = len(sizes), int(offs[-1])
    e = lambda *s: torch.empty(s, dtype=torch.float64, device=dev)
    O2, O3, OX, OR, OC, OW = e(B, 12), e(B, 12), e(3 * m), e(B), e(B), e(m)
    OI = torch.zeros(B, dtype=torch.int32, device=dev); OS = torch.zeros(B, dtype=torch.int32, device=dev)
    p = lambda x: C.c_void_p(x.data_ptr())
    d_c, d_m, d_r2, d_r3, d_x = t(c), t(calm), t(r2), t(r3), t(x0)
    torch.cuda.synchronize()
    h.call("tvf_bundle_adjust_robust_ragged_dev", p(d_c), p(d_m), 0, offs.ctypes.data_as(C.c_void_p), B, 2, C.c_double(1.5),
           p(d_r2), p(d_r3), p(d_x), p(O2), p(O3), p(OX), p(OR), p(OC), p(OW), p(OI), p(OS))
    h.call("tvf_synchronize")
    assert np.array_equal(tvf.api._from_cm(O2.cpu().numpy().ravel(), B, (3, 4), True), rag[0], equal_nan=True)
    assert np.array_equal(OC.cpu().numpy(), rag.cost, equal_nan=True)
    assert np.array_equal(OW.cpu().numpy(), np.concatenate(rag.weights), equal_nan=True)
    assert np.array_equal(OS.cpu().numpy(), rag.status)


def test_pageable_staged_path_equals_pinned_path(tvf):
    """> 4 MB of pageable buffers go through the pinned staging buffers; pinned buffers are used in place; the same bits
    either way, and through a group handle."""
    from tft_vs_fund_b200 import _lib
    B, n = 20_001, 20
    d = tvf.scene.sweep_batch_device(B, n, first_trial=5)
    start = tvf.LinearTFTPoseEstimation(d["Corresp"], d["CalM"])
    cm = lambda a: tvf.api._cm(a, 2)[0]
    inputs = [cm(d["Corresp"]), np.ascontiguousarray(np.broadcast_to(d["CalM"].T, (B, 3, 9))), cm(start[0]), cm(start[1]),
              cm(start[2])]
    shapes = [(B, 12), (B, 12), (B, 3 * n), (B,), (B,), (B, n), (B,), (B,)]
    dtypes = [np.float64] * 6 + [np.int32] * 2

    def run(h, alloc):
        ins = [alloc(a.shape, a.dtype) for a in inputs]
        for a, b in zip(ins, inputs):
            a[...] = b
        out = [alloc(s, t) for s, t in zip(shapes, dtypes)]
        p = lambda a: a.ctypes.data_as(_lib.c_int32_p if a.dtype == np.int32 else _lib.c_double_p)
        h.call("tvf_bundle_adjust_robust", p(ins[0]), p(ins[1]), 1, n, B, 1, C.c_double(2.0), p(ins[2]), p(ins[3]), p(ins[4]),
               *[p(a) for a in out])
        return [a.copy() for a in out]

    pins = []

    def pinned(shape, dtype):
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        ptr = _lib.load().tvf_host_alloc(nbytes)
        assert ptr
        pins.append(ptr)
        return np.frombuffer((C.c_char * nbytes).from_address(ptr), dtype=dtype).reshape(shape)
    pageable = lambda shape, dtype: np.empty(shape, dtype)
    h, grp = _lib.handle(), _lib.handle((0, 0))
    try:
        for x in (h, grp):
            x.call("tvf_set_chunk", 3000)
        ref = run(h, pinned)
        runs = {"pageable": run(h, pageable), "group (0, 0)": run(grp, pageable)}
        h.call("tvf_set_host_register", 1)
        runs["registered"] = run(h, pageable)
    finally:
        for x in (h, grp):
            x.call("tvf_set_chunk", 0)
            x.call("tvf_set_host_register", 0)
        for ptr in pins:
            _lib.load().tvf_host_free(C.c_void_p(ptr))
    assert np.count_nonzero(ref[7] == 0) > B // 2
    for name, got in runs.items():
        for k, (a, b) in enumerate(zip(ref, got)):
            assert np.array_equal(a, b, equal_nan=True), (name, k)


# ---- robustness -----------------------------------------------------------------------------------------------------
# outlier_scenes(0.3, 30, 51), plain tvf_ransac_pose (method 1, H = hypotheses_for(0.3, 7), 1 px, seed 1000 + b), then
# from its pose (points triangulated) one adjustment over all 100 matches; the reference is the plain adjustment on the
# true inliers from the truth.  CPU oracle (tests/ba_robust_oracle.py, oracle/bundle_adjust.py, ransac_oracle.ransac),
# rotation error in degrees (mean of views 2 and 3):
#   scene  RANSAC  robust (Cauchy, c = 3 px)  plain over all matches  plain on the true inliers
#   0        5.00       0.199                      78.2                     0.183
#   1      110         112                        111                       0.070
#   2      157         158                        145                       0.128
# So the robust adjustment polishes a pose in the minimiser's basin to the accuracy of the adjustment on the true
# inliers (1.09x), where the plain one over all matches is dragged away (430x); it cannot rescue a wrong RANSAC pose,
# and at 1 px plain RANSAC returns one on most of these scenes (its consensus is partial).  The bounds are on the medians
# over the scenes whose RANSAC pose is within 10 degrees (2 of the 30 on the B200: 1.13x and 515x there): robust within
# 2x of the reference, plain at least 10x worse.
ROBUST_BOUNDS = dict(basin_deg=10.0, robust_ratio=2.0, plain_ratio=10.0)


def test_robustness_of_cauchy_over_all_raw_matches(tvf):
    count = 30
    Cr, CalM, R_t0, out = ro.outlier_scenes(0.3, count, 51)
    H = ro.hypotheses_for(0.3, 7)
    rp = tvf.ransac_pose(Cr, CalM, method=1, hypotheses=H, threshold=1.0, seed=1000)
    assert np.all(rp.status == 0)
    rob = tvf.bundle_adjust(Cr, CalM, rp[0], rp[1], loss="cauchy", scale=3.0)
    plain = tvf.bundle_adjust(Cr, CalM, rp[0], rp[1])
    err = lambda R2, R3: (o.AngError(R_t0[0], R2)[0] + o.AngError(R_t0[1], R3)[0]) / 2
    e_ran = np.array([err(rp[0][b], rp[1][b]) for b in range(count)])
    e_rob = np.array([err(rob[0][b], rob[1][b]) for b in range(count)])
    e_plain = np.array([err(plain[0][b], plain[1][b]) for b in range(count)])
    e_ref = []
    for b in range(count):
        r = tvf.bundle_adjust(Cr[b][:, ~out[b]], CalM, R_t0[0], R_t0[1])
        e_ref.append(err(r[0], r[1]))
    e_ref = np.array(e_ref)
    basin = e_ran < ROBUST_BOUNDS["basin_deg"]
    ratio_rob = np.median(e_rob[basin]) / np.median(e_ref[basin])
    ratio_plain = np.median(e_plain[basin]) / np.median(e_ref[basin])
    print("30 %% outliers, %d of %d RANSAC poses within %g deg; there median rot err: RANSAC %.3f, robust %.4f, plain over "
          "all %.3f, plain on the true inliers %.4f deg (ratios %.2f / %.1f); all scenes: robust %.3f, plain %.3f"
          % (basin.sum(), count, ROBUST_BOUNDS["basin_deg"], np.median(e_ran[basin]), np.median(e_rob[basin]),
             np.median(e_plain[basin]), np.median(e_ref[basin]), ratio_rob, ratio_plain, np.median(e_rob),
             np.median(e_plain)))
    assert basin.sum() >= 2
    assert ratio_rob <= ROBUST_BOUNDS["robust_ratio"]
    assert ratio_plain >= ROBUST_BOUNDS["plain_ratio"]


# ---- edge cases -----------------------------------------------------------------------------------------------------
def test_nonfinite_inputs_are_flagged_and_neighbours_unchanged(tvf):
    g = np.load(__import__("os").path.join(__import__("conftest").ROOT, "tests", "golden", "sweep_n20.npz"))
    Cr, CalM = g["Corresp"][:6].copy(), g["CalM"][:6]
    Rt2, Rt3, X = g["tft_Rt2"][:6], g["tft_Rt3"][:6], g["tft_Reconst"][:6]
    kw = dict(loss="huber", scale=1.0)
    clean = tvf.bundle_adjust(Cr, CalM, Rt2, Rt3, X, **kw)
    Cr[2, 3, 5] = np.nan
    dirty = tvf.bundle_adjust(Cr, CalM, Rt2, Rt3, X, **kw)
    assert dirty.status[2] == tvf._lib.ST_NONFINITE and dirty[3][2] == 0
    assert np.array_equal(dirty[0][2], Rt2[2]) and np.array_equal(dirty[1][2], Rt3[2]) and np.array_equal(dirty[2][2], X[2])
    assert np.isnan(dirty.cost[2]) and np.all(np.isnan(dirty.weights[2]))
    keep = [0, 1, 3, 4, 5]
    for a, b in zip(_outs(clean), _outs(dirty)):
        assert np.array_equal(np.asarray(a)[keep], np.asarray(b)[keep])
    z = Rt2.copy(); z[4, :, 3] = 0.0
    res = tvf.bundle_adjust(g["Corresp"][:6], CalM, z, Rt3, X, **kw)
    assert res.status[4] == tvf._lib.ST_NONFINITE and res[3][4] == 0 and np.isnan(res.cost[4])


def test_argument_errors_before_any_device_work(tvf):
    from tft_vs_fund_b200 import _lib
    h = _lib.handle()
    n, B = 20, 2
    dp = lambda a: a.ctypes.data_as(_lib.c_double_p)
    c = np.zeros(6 * n * B); m = np.tile(np.eye(3), (3, 1)).T.copy(); r = np.tile(np.eye(3, 4).T.ravel(), B)
    o2, o3 = np.zeros(12 * B), np.zeros(12 * B)
    launches = h.lib.tvf_launch_count(h._h)
    for loss, scale in ((0, 1.0), (4, 1.0), (-1, 1.0), (1, 0.0), (2, -1.0), (3, np.nan), (1, np.inf), (1, 1e200)):
        rc = h.lib.tvf_bundle_adjust_robust(h._h, dp(c), dp(m), 0, n, B, loss, scale, dp(r), dp(r), None, dp(o2), dp(o3),
                                            None, None, None, None, None, None)
        assert rc == _lib.TVF_ERR_ARG, (loss, scale)
    assert h.lib.tvf_launch_count(h._h) == launches
    rc = h.lib.tvf_bundle_adjust_robust(h._h, dp(c), dp(m), 0, 3, 1, 1, 1.0, dp(r), dp(r), None, dp(o2), dp(o3), None, None,
                                        None, None, None, None)
    assert rc == _lib.TVF_ERR_ARG
    # B = 0 runs and returns
    assert h.lib.tvf_bundle_adjust_robust(h._h, dp(c), dp(m), 0, n, 0, 1, 1.0, dp(r), dp(r), None, dp(o2), dp(o3), None, None,
                                          None, None, None, None) == 0
    offs = np.zeros(1, dtype=np.int64)
    assert h.lib.tvf_bundle_adjust_robust_ragged(h._h, dp(c), dp(m), 0, offs.ctypes.data_as(C.c_void_p), 0, 3, 2.0, dp(r),
                                                 dp(r), None, dp(o2), dp(o3), None, None, None, None, None, None) == 0
    with pytest.raises(ValueError):
        tvf.bundle_adjust(np.zeros((6, 20)), np.tile(np.eye(3), (3, 1)), np.eye(3, 4), np.eye(3, 4), loss="l2", scale=1.0)
    with pytest.raises(ValueError):
        tvf.bundle_adjust(np.zeros((6, 20)), np.tile(np.eye(3), (3, 1)), np.eye(3, 4), np.eye(3, 4), loss="cauchy")
    with pytest.raises(_lib.TvfError):
        tvf.bundle_adjust(np.zeros((6, 3)), np.tile(np.eye(3), (3, 1)), np.eye(3, 4), np.eye(3, 4), loss="huber", scale=1.0)


def test_api_single_problem_and_batch(tvf):
    Cr, CalM, R_t0, _ = ro.outlier_scenes(0.1, 4, 9)
    start = tvf.LinearTFTPoseEstimation(Cr, CalM)
    batch = tvf.bundle_adjust(Cr, CalM, start[0], start[1], start[2], loss="soft_l1", scale=1.0)
    assert batch.cost.shape == (4,) and batch.weights.shape == (4, 100)
    one = tvf.bundle_adjust(Cr[2], CalM, start[0][2], start[1][2], start[2][2], loss="soft_l1", scale=1.0)
    assert isinstance(one.cost, float) and one.weights.shape == (100,)
    assert one.cost == batch.cost[2] and np.array_equal(one.weights, batch.weights[2])
    assert np.array_equal(one[0], batch[0][2])
    plain = tvf.bundle_adjust(Cr, CalM, start[0], start[1], start[2])
    assert plain.cost is None and plain.weights is None
