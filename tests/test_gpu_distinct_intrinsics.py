"""Every calibrated entry point on the GPU with a different K per view and per problem (tests/distinct_k.py): the pose
methods, R_t_from_TFT, the bundle adjustment and its covariance against the live oracles at the kernel-selection
boundaries; every problem of a batch with its own K == the call on that problem alone with its K shared (9 x 3), for the
uniform and the ragged forms, under chunks, a group handle, the _dev forms and pageable buffers; plain and refined RANSAC
against their CPU oracles; a wrong K fails the comparisons; the MEX gateways with CalM 9 x 3 x B."""
import ctypes as C

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

import oracle as o
from oracle import bundle_adjust as oba
import distinct_k as dk
import parity_workers as pw
import ransac_oracle as ro
import ransac_refined_oracle as rr
from conftest import TOL_ANGLE, TOL_MODEL, assert_pose_close, library_votes_as_float, rel_frob_up_to_sign, rot_angle, \
    vec_angle, votes8_equal
from test_gpu_ba_covariance import check_against_oracle as covariance_against_oracle
from test_gpu_bundle_adjust import check_against_oracle as adjustment_against_oracle
from test_mex_gateways import _run as run_gateway, built  # noqa: F401  (built: the gateways' fixture)

pytestmark = pytest.mark.gpu

TOL_TRUTH = 1e-8          # rad: a noise-free problem's pose against the truth
WRONG_K_MIN = 1e-4        # rad: the least a wrong K must move the library's answer away from the oracle's


@pytest.fixture(scope="module")
def pool():
    with pw.pool() as p:
        yield p


def vote_tie(votes8):
    return any(np.isnan(v).any() or np.sum(v == np.max(v)) > 1 for v in (votes8[:4], votes8[4:]))


def assert_truth(R2, R3, R_t0, tag):
    for got, true in ((R2, R_t0[0]), (R3, R_t0[1])):
        assert rot_angle(true[:, :3], got[:, :3]) < TOL_TRUTH and vec_angle(true[:, 3], got[:, 3]) < TOL_TRUTH, tag
    ratio = np.linalg.norm(R3[:, 3]) / np.linalg.norm(R2[:, 3])
    assert abs(ratio * np.linalg.norm(R_t0[0][:, 3]) / np.linalg.norm(R_t0[1][:, 3]) - 1.0) < TOL_TRUTH, tag


def pose_error(a2, a3, b2, b3):
    return max(rot_angle(a2[:, :3], b2[:, :3]), rot_angle(a3[:, :3], b3[:, :3]))


def noisy_batch(n, levels=(0.0, 1.0, 3.0), count_per_level=2):
    """count_per_level problems at each noise level (px), every problem with its own three K"""
    noise = np.repeat(levels, count_per_level)
    return dk.batch(n, noise, range(1, noise.size + 1)) + (noise,)


# ---- pose methods against the oracle --------------------------------------------------------------------------------
# the kernel-selection boundaries of test_gpu_parity_r2.py and the large-n estimator
POSE_NS = [7, 8, 9, 12, 25, 32, 33, 64, 65, 128, 129, 256, 257, 300, 1024, 1027, 2500]


@pytest.mark.parametrize("n", POSE_NS)
def test_linear_pose_methods_and_r_t_from_tft_against_the_oracle(tvf, pool, n):
    from tft_vs_fund_b200 import _lib
    Cr, CalM, R_t0, _, noise = noisy_batch(n)
    B = Cr.shape[0]
    ref = pool.starmap(pw.solve_both, [(Cr[b], CalM[b]) for b in range(B)])
    methods = (("tft", tvf.LinearTFTPoseEstimation),) + ((("f", tvf.LinearFPoseEstimation),) if n >= 8 else ())
    for method, fn in methods:
        res = fn(Cr, CalM)
        for b in range(B):
            tag = "%s n=%d problem %d noise %g" % (method, n, b, noise[b])
            r = ref[b][method]
            if isinstance(r, str):              # the reference stops here (no candidate with a non-negative vote)
                assert res.status[b] & (_lib.ST_NO_POSE_2 | _lib.ST_NO_POSE_3), tag
                continue
            assert votes8_equal(library_votes_as_float(res.votes[b]), r[5]), (tag, res.votes[b], r[5])
            if noise[b] == 0.0:
                assert res.status[b] == 0, tag
                assert_truth(res[0][b], res[1][b], R_t0[b], tag)
            if vote_tie(r[5]):
                continue
            assert_pose_close(r[:5], (res[0][b], res[1][b], res[2][b], res[3][b], res.repr_err[b]), tag)
            if method == "f":
                assert rel_frob_up_to_sign(r[6], res.F21[b]) < TOL_MODEL and rel_frob_up_to_sign(r[7], res.F31[b]) < TOL_MODEL
    # R_t_from_TFT on the oracle's tensors, per-problem CalM
    ok = [b for b in range(B) if not isinstance(ref[b]["tft"], str)]
    T = np.stack([ref[b]["tft"][3] for b in ok])
    R2, R3, votes = tvf.R_t_from_TFT(T, CalM[ok], Cr[ok], return_votes=True)
    for k, b in enumerate(ok):
        o2, o3, v2, v3 = o.R_t_from_TFT(T[k], CalM[b], Cr[b], return_votes=True)
        want = np.array(list(v2) + list(v3), dtype=np.float64)
        assert votes8_equal(library_votes_as_float(votes[k]), want), (n, b)
        if vote_tie(want):
            continue
        for a, c in ((o2, R2[k]), (o3, R3[k])):
            assert rot_angle(a[:, :3], c[:, :3]) < TOL_ANGLE and vec_angle(a[:, 3], c[:, 3]) < TOL_ANGLE, (n, b)
        assert abs(np.linalg.norm(R3[k][:, 3]) / np.linalg.norm(o3[:, 3]) - 1.0) < 1e-9, (n, b)


@pytest.mark.parametrize("n", [8, 30, 100, 250])
def test_optimf_pose_against_the_oracle(tvf, n):
    Cr, CalM, R_t0, _, noise = noisy_batch(n)
    res = tvf.OptimFPoseEstimation(Cr, CalM)
    for b in range(Cr.shape[0]):
        tag = "optf n=%d problem %d noise %g" % (n, b, noise[b])
        Ks = [CalM[b][0:3], CalM[b][3:6], CalM[b][6:9]]
        R2, R3, Rec, T, it, F21, F31 = o.OptimFPoseEstimation(Cr[b], CalM[b], return_F=True)
        rep = o.ReprError([Ks[0] @ np.eye(3, 4), Ks[1] @ R2, Ks[2] @ R3], Cr[b], Rec)
        f2 = o.recover_R_t_F(Ks[0], Ks[1], F21, Cr[b][0:2], Cr[b][2:4], return_votes=True)[2]
        f3 = o.recover_R_t_F(Ks[0], Ks[2], F31, Cr[b][0:2], Cr[b][4:6], return_votes=True)[2]
        votes = np.array(list(f2) + list(f3), dtype=np.float64)
        assert votes8_equal(library_votes_as_float(res.votes[b]), votes), tag
        assert int(res[4][b]) == int(it), tag
        assert rel_frob_up_to_sign(F21, res.F21[b]) < TOL_MODEL and rel_frob_up_to_sign(F31, res.F31[b]) < TOL_MODEL, tag
        if noise[b] == 0.0:
            assert_truth(res[0][b], res[1][b], R_t0[b], tag)
        if not vote_tie(votes):
            assert_pose_close((R2, R3, Rec, T, rep), (res[0][b], res[1][b], res[2][b], res[3][b], res.repr_err[b]), tag)


# ---- bundle adjustment and covariance against the oracles -----------------------------------------------------------
def perturbed_truth(CalM, R_t0, X, rs, rot=5e-4, rel=5e-4):
    """the true states (|t2| = 1) of a batch, perturbed: (B,3,4), (B,3,4), (B,3,n)"""
    out = [], [], []
    for b in range(CalM.shape[0]):
        Rt2, Rt3, Xs = dk.gauge_truth(CalM[b], R_t0[b], X[b])
        dR = lambda: Rotation.from_rotvec(rs.standard_normal(3) * rot / np.sqrt(3)).as_matrix()
        out[0].append(np.column_stack([dR() @ Rt2[:, :3], Rt2[:, 3] + rel * rs.standard_normal(3)]))
        out[1].append(np.column_stack([dR() @ Rt3[:, :3], Rt3[:, 3] * (1 + rel * rs.standard_normal(3))]))
        out[2].append(Xs * (1 + rel * rs.standard_normal(Xs.shape)))
    return tuple(np.stack(a) for a in out)


@pytest.mark.parametrize("n", [4, 5, 8, 9, 20, 33, 100])
def test_bundle_adjust_against_the_oracle(tvf, n):
    # 1 px at most, as test_gpu_bundle_adjust.py: at n = 4 (one degree of freedom) and 3 px a problem can reach the
    # iteration cap (TVF_ST_BA_NOCONV) before the oracle's minimum
    Cr, CalM, R_t0, X, noise = noisy_batch(n, levels=(0.0, 0.5, 1.0))
    S2, S3, SX = perturbed_truth(CalM, R_t0, X, np.random.RandomState(n))
    res, checked = adjustment_against_oracle(tvf, Cr, CalM, S2, S3, SX, "n=%d" % n)
    assert checked == Cr.shape[0]
    for b in np.flatnonzero(noise == 0.0):
        assert res.repr_err[b] < 1e-9, (n, b)
        assert_truth(res[0][b], res[1][b], R_t0[b], (n, b))


@pytest.mark.parametrize("n", [4, 5, 8, 9, 20, 31, 32, 33, 64, 65, 100])
def test_covariance_against_the_oracle(tvf, n):
    Cr, CalM, R_t0, X = dk.batch(n, 1.0, range(1, 5))
    S = [np.stack(a) for a in zip(*[dk.gauge_truth(CalM[b], R_t0[b], X[b]) for b in range(4)])]
    ba = tvf.bundle_adjust(Cr, CalM, *S)
    assert np.all(ba.status == 0)
    checked, worst = covariance_against_oracle(tvf, Cr, CalM, ba, ba.status == 0, "n=%d" % n)
    print("n = %d: %d problems, worst relative Frobenius %.2e" % (n, checked, worst))
    assert checked == 4


# ---- every problem with its own K in one batch == that problem alone with its K shared ------------------------------
B_BITS = 21              # three chunks of 7


def same_bits(a, b):
    """two lists of outputs hold the same bits (a list inside: a ragged per-match output)"""
    bits = lambda x: (np.asarray(x).dtype.str, np.asarray(x).shape, np.ascontiguousarray(x).tobytes())
    return len(a) == len(b) and all(same_bits(x, y) if isinstance(x, list) else bits(x) == bits(y) for x, y in zip(a, b))


def differences(got, want):
    """{output index: problems whose bits differ} of two lists of batched outputs"""
    return {i: [b for b in range(B_BITS) if not same_bits([x[b]], [y[b]])] for i, (x, y) in enumerate(zip(got, want))
            if not same_bits([x], [y])}


@pytest.fixture(scope="module")
def bitdata(tvf):
    """Clean scenes (n = 40, 1 px) and scenes with outliers (n = 60, noise-free inliers, a share growing from 5 % to 30 %
    with the problem index, so that the consensus sizes fall with it and the refit's regrouping by consensus size
    reverses the order; with noisy inliers the minimal solves explain almost nothing and no refit would run),
    each with its own K; ragged forms of both (n_b from 4 to 60); starts and adjusted states."""
    Cr, CalM, R_t0, X = dk.batch(40, 1.0, range(1, B_BITS + 1))
    Co, CalMo, R_t0o, _ = dk.outlier_scenes(np.linspace(0.05, 0.3, B_BITS), B_BITS, 101, noise=0.0, n=60)
    S2, S3, SX = perturbed_truth(CalM, R_t0, X, np.random.RandomState(3))
    ba = tvf.bundle_adjust(Cr, CalM, S2, S3, SX)
    nb = [40, 9, 23, 4, 33, 17, 38, 12, 5, 31, 27, 40, 8, 19, 36, 6, 25, 14, 40, 11, 30]
    no = [60, 12, 45, 31, 8, 52, 7, 40, 19, 60, 26, 9, 55, 33, 14, 48, 21, 60, 10, 37, 28]
    d = dict(Cr=Cr, CalM=CalM, T=tvf.LinearTFTPoseEstimation(Cr, CalM)[3], S2=S2, S3=S3, SX=SX, B2=ba[0], B3=ba[1], BX=ba[2],
             Co=Co, CalMo=CalMo, R2t=R_t0o[:, 0], R3t=R_t0o[:, 1], seeds=np.arange(500, 500 + B_BITS, dtype=np.uint64),
             Cs=[Cr[b][:, :nb[b]] for b in range(B_BITS)], SXs=[SX[b][:, :nb[b]] for b in range(B_BITS)],
             Cso=[Co[b][:, :no[b]] for b in range(B_BITS)])
    bar = tvf.bundle_adjust(d["Cs"], CalM, S2, S3, d["SXs"])
    d.update(B2s=bar[0], B3s=bar[1], BXs=bar[2])
    return d


def entry_points(api, d):
    """name -> (f(sel, K, device) -> list of outputs, each indexable by problem; the name of the CalM it takes)"""
    L = lambda key, sel: [d[key][i] for i in sel]
    pose = lambda r: [r[0], r[1], r[2], r[3], r.repr_err, r.status, r.votes] + \
        ([r.F21, r.F31] if r.F21 is not None else []) + ([r[4]] if isinstance(r[4], np.ndarray) else [])
    ba = lambda r: [r[0], r[1], r[2], r[3], r.repr_err, r.status]
    cov = lambda r: [r[0], r[1], r.cov_pts, r.status]
    ran = lambda r, refine: list(r) + [r.status] + ([r.lo_done] if refine else [])
    E = {}
    for name, fn in (("tft", api.LinearTFTPoseEstimation), ("f", api.LinearFPoseEstimation), ("optf", api.OptimFPoseEstimation)):
        E[name] = (lambda s, K, dev, fn=fn: pose(fn(d["Cr"][s], K, device=dev)), "CalM")
    E["R_t_from_TFT"] = (lambda s, K, dev: list(api.R_t_from_TFT(d["T"][s], K, d["Cr"][s], device=dev, return_votes=True)),
                         "CalM")
    E["bundle_adjust"] = (lambda s, K, dev: ba(api.bundle_adjust(d["Cr"][s], K, d["S2"][s], d["S3"][s], d["SX"][s],
                                                                 device=dev)), "CalM")
    E["bundle_adjust, triangulated start"] = (lambda s, K, dev: ba(api.bundle_adjust(d["Cr"][s], K, d["S2"][s], d["S3"][s],
                                                                                     device=dev)), "CalM")
    E["ba_covariance"] = (lambda s, K, dev: cov(api.ba_covariance(d["Cr"][s], K, d["B2"][s], d["B3"][s], d["BX"][s],
                                                                  points=True, device=dev)), "CalM")
    E["consensus"] = (lambda s, K, dev: list(api.consensus(d["Co"][s], K, d["R2t"][s], d["R3t"][s], threshold=2.0,
                                                           device=dev)), "CalMo")
    E["bundle_adjust ragged"] = (lambda s, K, dev: ba(api.bundle_adjust(L("Cs", s), K, d["S2"][s], d["S3"][s], L("SXs", s),
                                                                        device=dev)), "CalM")
    E["ba_covariance ragged"] = (lambda s, K, dev: cov(api.ba_covariance(L("Cs", s), K, d["B2s"][s], d["B3s"][s],
                                                                         L("BXs", s), points=True, device=dev)), "CalM")
    E["consensus ragged"] = (lambda s, K, dev: list(api.consensus(L("Cso", s), K, d["R2t"][s], d["R3t"][s], threshold=2.0,
                                                                  device=dev)), "CalMo")
    for method in (1, 7):
        for refine in (False, True):
            for ragged in (False, True):
                key = "Cso" if ragged else "Co"
                E["ransac method %d%s%s" % (method, " refined" if refine else "", " ragged" if ragged else "")] = (
                    lambda s, K, dev, method=method, refine=refine, key=key: ran(api.ransac_pose(
                        L(key, s) if key == "Cso" else d[key][s], K, method=method, hypotheses=64, threshold=2.0,
                        seed=d["seeds"][s], device=dev, refine=refine, lo_rounds=4), refine), "CalMo")
    return E


@pytest.fixture(scope="module")
def full_batch(tvf, bitdata):
    """every entry point on the whole batch, each problem with its own K"""
    return {name: fn(np.arange(B_BITS), bitdata[k], None) for name, (fn, k) in entry_points(tvf.api, bitdata).items()}


def test_every_problem_equals_its_single_call_with_a_shared_k(tvf, bitdata, full_batch):
    for name, (fn, key) in entry_points(tvf.api, bitdata).items():
        full = full_batch[name]
        for b in range(B_BITS):
            one = fn(np.array([b]), bitdata[key][b], None)            # CalM 9 x 3: calm_batched = 0
            assert same_bits([x[b] for x in full], [x[0] for x in one]), (name, b)


def test_ransac_refit_regrouping_permutes_the_problems(tvf, bitdata, full_batch):
    """The refit and the LO rounds gather each problem's K by the problem's place in the order of consensus sizes: in this
    batch that order is not the problem order, so the gathers are exercised."""
    Co, K = bitdata["Co"], bitdata["CalMo"]
    for method in (1, 7):
        s = ro.SAMPLE_SIZE[method]
        fn = tvf.LinearTFTPoseEstimation if method == 1 else tvf.LinearFPoseEstimation
        for refine in (False, True):
            smp = full_batch["ransac method %d%s" % (method, " refined" if refine else "")][4]
            S = np.stack([Co[b][:, smp[b]] for b in range(B_BITS)])
            P = fn(S, K)
            R2, R3 = (P[0], P[1]) if not refine else tvf.bundle_adjust(S, K, P[0], P[1])[:2]
            cnt = tvf.consensus(Co, K, R2, R3, threshold=2.0)[1]          # the winning hypothesis' count, before the refit
            order = [b for b in np.argsort(cnt, kind="stable") if cnt[b] >= s]
            assert len(order) >= B_BITS - 2 and order != sorted(order), (method, refine, cnt)


def test_invariance_under_chunks_group_handle_and_device_pointers(tvf, bitdata, full_batch):
    import torch
    from tft_vs_fund_b200 import _lib, api
    E = entry_points(api, bitdata)
    h = _lib.handle()
    try:
        h.call("tvf_set_chunk", 7)
        for name, (fn, key) in E.items():
            got = fn(np.arange(B_BITS), bitdata[key], None)
            assert same_bits(got, full_batch[name]), ("chunk 7", name, differences(got, full_batch[name]))
    finally:
        h.call("tvf_set_chunk", 0)
    for name, (fn, key) in E.items():
        got = fn(np.arange(B_BITS), bitdata[key], (0, 0))
        assert same_bits(got, full_batch[name]), ("group (0, 0)", name, differences(got, full_batch[name]))

    # the _dev forms, calm_batched = 1, == the host forms
    d = bitdata
    B = B_BITS
    dev = torch.device("cuda", 0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    p = lambda x: C.c_void_p(x.data_ptr()) if x is not None else None
    f64 = lambda *shape: torch.empty(shape, dtype=torch.float64, device=dev)
    i32 = lambda *shape: torch.zeros(shape, dtype=torch.int32, device=dev)
    back = lambda x, dims: api._from_cm(x.cpu().numpy().ravel(), B, dims, True)
    n = d["Cr"].shape[2]
    d_c, d_k = t(api._cm(d["Cr"], 2)[0]), t(api._calm(d["CalM"], B)[0])
    # tvf_pose_dev, method 1
    o2, o3, oX, oT, orep, ov, ost = f64(B, 12), f64(B, 12), f64(B, 3 * n), f64(B, 27), f64(B), i32(B, 10), i32(B)
    out = _lib.PoseOut(p(o2), p(o3), p(oX), p(oT), p(orep), None, None, None, p(ov), p(ost))
    torch.cuda.synchronize()
    h.call("tvf_pose_dev", _lib.METHOD_IDS["tft"], p(d_c), p(d_k), 1, n, B, C.byref(out))
    h.call("tvf_synchronize")
    want = full_batch["tft"]
    assert same_bits([back(o2, (3, 4)), back(o3, (3, 4)), back(oX, (3, n)), back(oT, (3, 3, 3)), orep.cpu().numpy(),
                      ost.cpu().numpy(), ov.cpu().numpy()], want[:7])
    # tvf_bundle_adjust_dev and tvf_ba_covariance_dev
    b2, b3, bX, brep, bit, bst = f64(B, 12), f64(B, 12), f64(B, 3 * n), f64(B), i32(B), i32(B)
    cc, cp, cs2, cst = f64(B, 144), f64(B, 9 * n), f64(B), i32(B)
    s2, s3 = api._pose_pair(d["S2"], d["S3"], B, True)
    d_s2, d_s3, d_sx = t(s2), t(s3), t(api._cm(d["SX"], 2)[0])
    torch.cuda.synchronize()
    h.call("tvf_bundle_adjust_dev", p(d_c), p(d_k), 1, n, B, p(d_s2), p(d_s3), p(d_sx), p(b2), p(b3), p(bX), p(brep), p(bit),
           p(bst))
    h.call("tvf_ba_covariance_dev", p(d_c), p(d_k), 1, n, B, p(b2), p(b3), p(bX), p(cc), p(cp), p(cs2), p(cst))
    h.call("tvf_synchronize")
    assert same_bits([back(b2, (3, 4)), back(b3, (3, 4)), back(bX, (3, n)), bit.cpu().numpy(), brep.cpu().numpy(),
                      bst.cpu().numpy()], full_batch["bundle_adjust"])
    assert same_bits([back(cc, (12, 12)), cs2.cpu().numpy(), back(cp, (3, 3, n)), cst.cpu().numpy()],
                     full_batch["ba_covariance"])
    # tvf_ransac_pose_dev (uniform) and tvf_ransac_pose_refined_ragged_dev
    no = d["Co"].shape[2]
    d_o, d_ko, d_seed = t(api._cm(d["Co"], 2)[0]), t(api._calm(d["CalMo"], B)[0]), t(d["seeds"].view(np.int64))
    r2, r3, rm, rc, rs_, rst = f64(B, 12), f64(B, 12), torch.zeros(B * no, dtype=torch.uint8, device=dev), i32(B), i32(B, 7), i32(B)
    torch.cuda.synchronize()
    h.call("tvf_ransac_pose_dev", 1, p(d_o), p(d_ko), 1, no, B, 64, 2.0, p(d_seed), p(r2), p(r3), p(rm), p(rc), p(rs_), p(rst))
    h.call("tvf_synchronize")
    assert same_bits([back(r2, (3, 4)), back(r3, (3, 4)), rm.cpu().numpy().reshape(B, no).astype(bool), rc.cpu().numpy(),
                      rs_.cpu().numpy(), rst.cpu().numpy()], full_batch["ransac method 1"])
    c, offs = api._pack(d["Cso"], 6)
    d_cr = t(c)
    g2, g3, gm, gc, gs, glo, gst = f64(B, 12), f64(B, 12), torch.zeros(int(offs[-1]), dtype=torch.uint8, device=dev), i32(B), \
        i32(B, 7), i32(B), i32(B)
    torch.cuda.synchronize()
    h.call("tvf_ransac_pose_refined_ragged_dev", 1, p(d_cr), p(d_ko), 1, offs.ctypes.data_as(C.c_void_p), B, 64, 2.0,
           p(d_seed), 4, p(g2), p(g3), p(gm), p(gc), p(gs), p(glo), p(gst))
    h.call("tvf_synchronize")
    want = full_batch["ransac method 1 refined ragged"]
    got = [back(g2, (3, 4)), back(g3, (3, 4)), [m.astype(bool) for m in api._unpack(gm.cpu().numpy(), offs, ())],
           gc.cpu().numpy(), gs.cpu().numpy(), gst.cpu().numpy(), glo.cpu().numpy()]
    assert same_bits(got[:2] + got[3:], want[:2] + want[3:])
    assert all(np.array_equal(a, b) for a, b in zip(got[2], want[2]))


def test_pageable_staged_path_with_a_k_per_problem(tvf, bitdata, full_batch):
    """A batch large enough for the pinned staging buffers (> 4 MB per call, ten chunks), each problem with its own K
    (the 21 problems above, repeated): pageable buffers with 1 and 3 host threads == pinned buffers used in place, and
    every problem == its single call."""
    from tft_vs_fund_b200 import _lib, api
    d = bitdata
    B = 30_001
    idx = np.arange(B) % B_BITS
    n = d["Cr"].shape[2]
    cm = lambda a: api._cm(a, 2)[0]
    inputs = [cm(d["Cr"])[idx], api._calm(d["CalM"], B_BITS)[0][idx], cm(d["S2"])[idx], cm(d["S3"])[idx], cm(d["SX"])[idx]]
    shapes = [(B, 12), (B, 12), (B, 3 * n), (B,), (B,), (B,), (B, 144), (B, 9 * n), (B,), (B,),
              (B, 12), (B, 12), (B, 3 * n), (B, 27), (B,), (B,)]
    dtypes = [np.float64] * 4 + [np.int32] * 2 + [np.float64] * 3 + [np.int32] + [np.float64] * 5 + [np.int32]

    def run(h, alloc):
        """bundle_adjust from the starts, the covariance at its result, and the TFT pose, every array from `alloc`"""
        ins = [alloc(a.shape, a.dtype) for a in inputs]
        for a, b in zip(ins, inputs):
            a[...] = b
        o = [alloc(s, t) for s, t in zip(shapes, dtypes)]
        p = lambda a: a.ctypes.data_as(_lib.c_int32_p if a.dtype == np.int32 else _lib.c_double_p)
        h.call("tvf_bundle_adjust", p(ins[0]), p(ins[1]), 1, n, B, p(ins[2]), p(ins[3]), p(ins[4]), *[p(a) for a in o[:6]])
        h.call("tvf_ba_covariance", p(ins[0]), p(ins[1]), 1, n, B, p(o[0]), p(o[1]), p(o[2]), *[p(a) for a in o[6:10]])
        h.call("tvf_linear_tft_pose", p(ins[0]), p(ins[1]), 1, n, B, *[p(a) for a in o[10:]])
        return [a.copy() for a in o]

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
        runs = {}
        for threads in (1, 3):
            h.call("tvf_set_host_threads", threads)
            runs["threads %d" % threads] = run(h, pageable)
        h.call("tvf_set_host_threads", 0)
        runs["group (0, 0)"] = run(grp, pageable)
    finally:
        for x in (h, grp):
            x.call("tvf_set_chunk", 0)
            x.call("tvf_set_host_threads", 0)
        for ptr in pins:
            _lib.load().tvf_host_free(C.c_void_p(ptr))
    for name, got in runs.items():
        for k, (a, b) in enumerate(zip(ref, got)):
            assert np.array_equal(a, b, equal_nan=True), (name, k)
    # every problem of the large batch is the single call of its scene
    ba, cov, tft = full_batch["bundle_adjust"], full_batch["ba_covariance"], full_batch["tft"]
    pose = lambda x: api._from_cm(x.ravel(), B, (3, 4), True)
    assert np.array_equal(pose(ref[0]), ba[0][idx]) and np.array_equal(pose(ref[1]), ba[1][idx])
    assert np.array_equal(api._from_cm(ref[2].ravel(), B, (3, n), True), ba[2][idx])
    assert np.array_equal(ref[3], ba[4][idx]) and np.array_equal(ref[4], ba[3][idx]) and np.array_equal(ref[5], ba[5][idx])
    assert np.array_equal(api._from_cm(ref[6].ravel(), B, (12, 12), True), cov[0][idx]) and np.array_equal(ref[8], cov[1][idx])
    assert np.array_equal(pose(ref[10]), tft[0][idx]) and np.array_equal(api._from_cm(ref[13].ravel(), B, (3, 3, 3), True),
                                                                        tft[3][idx])


# ---- RANSAC against the oracles --------------------------------------------------------------------------------------
@pytest.mark.parametrize("method", [1, 7])
def test_ransac_against_the_oracle(tvf, method):
    """Noise-free inliers, 20 % outliers, a K per view and per problem: sample, n_inliers and inliers equal the oracle's
    wherever no match of a competitive hypothesis lies within 1e-6 px of the threshold (>= 90 % of the problems), and
    the poses agree to the parity tolerances."""
    H, th = 64, 2.0
    Cr, CalM, _, _ = dk.outlier_scenes(0.2, 12, 31, noise=0.0, n=40)
    got = tvf.ransac_pose(Cr, CalM, method=method, hypotheses=H, threshold=th, seed=100)
    clean = 0
    for b in range(Cr.shape[0]):
        want = ro.ransac(Cr[b], CalM[b], method, H, th, 100 + b)
        if ro.near_threshold(want, 1e-6):
            continue
        clean += 1
        assert got.status[b] == want["status"], b
        assert np.array_equal(got[4][b], want["sample"]) and got[3][b] == want["n_inliers"], b
        assert np.array_equal(got[2][b], want["inliers"]), b
        if want["status"] == 0:
            Kb = CalM[b]
            fn = lambda R2, R3: (R2, R3, np.zeros((3, 1)), o.TFT_from_P(Kb[0:3] @ np.eye(3, 4), Kb[3:6] @ R2, Kb[6:9] @ R3), 0.0)
            assert_pose_close(fn(want["Rt2"], want["Rt3"]), fn(got[0][b], got[1][b]), "problem %d" % b)
    print("method %d: %d of %d problems away from the threshold" % (method, clean, Cr.shape[0]))
    assert clean >= 0.9 * Cr.shape[0]


@pytest.mark.parametrize("method", [1, 7])
def test_refined_ransac_against_the_oracle(tvf, method):
    """As test_gpu_ransac_refined.test_against_the_oracle, with a K per view and per problem."""
    H, th = 16, 2.0
    Cr, CalM, _, out = dk.outlier_scenes(0.2, 10, 41, noise=0.0, n=32)
    got = tvf.ransac_pose(Cr, CalM, method=method, hypotheses=H, threshold=th, seed=100, refine=True, lo_rounds=8)
    clean = 0
    for b in range(Cr.shape[0]):
        want = rr.ransac_refined(Cr[b], CalM[b], method, H, th, 100 + b)
        if rr.near_threshold(want, 1e-6) or want["status"] != 0 or out[b][want["sample"]].any():
            continue
        clean += 1
        assert got.status[b] == 0, b
        assert np.array_equal(got[4][b], want["sample"]) and got[3][b] == want["n_inliers"], b
        assert np.array_equal(got[2][b], want["inliers"]) and got.lo_done[b] == want["lo_done"], b
        Kb = CalM[b]
        fn = lambda R2, R3: (R2, R3, np.zeros((3, 1)), o.TFT_from_P(Kb[0:3] @ np.eye(3, 4), Kb[3:6] @ R2, Kb[6:9] @ R3), 0.0)
        assert_pose_close(fn(want["Rt2"], want["Rt3"]), fn(got[0][b], got[1][b]), "problem %d" % b)
    print("method %d: %d of %d problems compared" % (method, clean, Cr.shape[0]))
    assert clean >= 0.7 * Cr.shape[0]


# ---- the comparisons have power ------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [20, 300])
def test_a_wrong_k_fails_the_oracle_comparisons(tvf, n):
    """The library called with each wrong-K variant (K2 and K3 swapped, K1 for every view, problem 0's K for every
    problem) misses the oracle's answer for the right K by more than 1e-4 rad: poses of both linear methods and of the
    adjustment, and the covariance by more than 1e-3 relative."""
    Cr, CalM, R_t0, X = dk.batch(n, 1.0, range(1, 5))
    S = [np.stack(a) for a in zip(*[dk.gauge_truth(CalM[b], R_t0[b], X[b]) for b in range(4)])]
    ref = {m: [fn(Cr[b], CalM[b])[:2] for b in range(4)] for m, fn in (("tft", o.LinearTFTPoseEstimation),
                                                                      ("f", o.LinearFPoseEstimation))}
    ref_ba = [oba.bundle_adjust(Cr[b], CalM[b], S[0][b], S[1][b], S[2][b]) for b in range(4)]
    right_ba = tvf.bundle_adjust(Cr, CalM, *S)
    right_cov = tvf.ba_covariance(Cr, CalM, right_ba[0], right_ba[1], right_ba[2])[0]
    for name, bad in dk.wrong_k(CalM).items():
        probs = range(1, 4) if name.startswith("problem 0") else range(4)
        for m, fn in (("tft", tvf.LinearTFTPoseEstimation), ("f", tvf.LinearFPoseEstimation)):
            res = fn(Cr, bad)
            for b in probs:
                e = pose_error(ref[m][b][0], ref[m][b][1], res[0][b], res[1][b])
                assert not e < WRONG_K_MIN, (name, m, b, e)
        res = tvf.bundle_adjust(Cr, bad, *S)
        cov = tvf.ba_covariance(Cr, bad, right_ba[0], right_ba[1], right_ba[2])[0]
        for b in probs:
            e = pose_error(ref_ba[b][0], ref_ba[b][1], res[0][b], res[1][b])
            assert not e < WRONG_K_MIN, (name, "ba", b, e)
            assert np.linalg.norm(cov[b] - right_cov[b]) > 1e-3 * np.linalg.norm(right_cov[b]), (name, "cov", b)


# ---- MEX ------------------------------------------------------------------------------------------------------------
def test_mex_gateways_with_a_calm_per_problem(tvf, built, tmp_path):  # noqa: F811
    """[R_t_2,R_t_3,Reconst,T,iter] = gateway(Corresp 6xNxB, CalM 9x3xB), each problem with its own K, == the Python API
    bit for bit."""
    Cr, CalM, _, _ = dk.batch(25, 1.0, range(1, 6))
    B, n = Cr.shape[0], Cr.shape[2]
    for gw, fn in (("LinearTFTPoseEstimation", tvf.LinearTFTPoseEstimation), ("LinearFPoseEstimation", tvf.LinearFPoseEstimation),
                   ("OptimFPoseEstimation", tvf.OptimFPoseEstimation)):
        outs = run_gateway(built, gw, 5, [(Cr.transpose(0, 2, 1), (6, n, B)), (CalM.transpose(0, 2, 1), (9, 3, B))],
                           str(tmp_path))
        assert [x.shape for x in outs[:4]] == [(3, 4, B), (3, 4, B), (3, n, B), (3, 3, 3, B)], gw
        res = fn(Cr, CalM)
        for k in range(4):
            assert np.array_equal(np.moveaxis(outs[k], -1, 0), res[k]), (gw, k)
