"""Ragged batches on the GPU (include/tvf.h: problems with different match counts in one call): every problem of
tvf_ransac_pose[_refined]_ragged, tvf_bundle_adjust_ragged, tvf_ba_covariance_ragged and tvf_consensus_ragged is bit for
bit the uniform call on that problem alone, on the 120 EPFL triplets and on synthetic batches of edge sizes; invariance
under chunk, group handle and form; problems below the minimum; argument errors; the batched real-data driver."""
import ctypes as C
import os

import numpy as np
import pytest

import ransac_oracle as ro
from conftest import ROOT

pytestmark = pytest.mark.gpu

ST_TOO_FEW = 256


def bits(x):
    a = np.ascontiguousarray(x)
    return a.dtype.str, a.shape, a.tobytes()


def same_bits(a, b):
    return all(bits(x) == bits(y) for x, y in zip(a, b))


def epfl_problems():
    """(list of Corresp 6 x N_b, CalM (120, 9, 3)) of the 120 EPFL triplets, all raw matches."""
    from tft_vs_fund_b200 import epfl
    inp = np.load(os.path.join(ROOT, "tests", "golden", "epfl_inputs.npz"))
    Cs, Ks = [], []
    for key in ("fountain_P11", "Herz_Jesu_P8"):
        data = epfl.dataset_from_arrays(inp[key + "_indexes_sorted"], inp[key + "_matches"], inp[key + "_offsets"],
                                        inp[key + "_K"], inp[key + "_R"], inp[key + "_t"])
        for it in range(1, data.indexes_sorted.shape[0] + 1):
            im = [int(v) for v in data.indexes_sorted[it - 1, 0:3]]
            Cs.append(data.corresp(*im).T.copy())
            Ks.append(epfl.relative_poses([data.camera(i) for i in im])[0])
    return Cs, np.stack(Ks)


@pytest.fixture(scope="module")
def epfl_all():
    return epfl_problems()


def edge_batch(s, seed=3):
    """n_b in {0, 3, s-1, s, s+1, 31, 32, 33, 100, 1400} in shuffled order: synthetic scenes with 30 % outliers (the first
    n_b columns) and the committed 1400-match EPFL triplet; per-problem CalM."""
    Cr, CalM, _, _ = ro.outlier_scenes(0.3, 9, 51)
    g = np.load(os.path.join(ROOT, "tests", "golden", "epfl_full_triplet.npz"))
    sizes = [0, 3, s - 1, s, s + 1, 31, 32, 33, 100]
    Cs = [Cr[k][:, :n].copy() for k, n in enumerate(sizes)] + [g["Corresp"].copy()]
    Ks = [CalM] * len(sizes) + [g["CalM"]]
    order = np.random.RandomState(seed).permutation(len(Cs))
    return [Cs[i] for i in order], np.stack([Ks[i] for i in order])


def ransac_fields(res, refine):
    return list(res) + [res.status] + ([res.lo_done] if refine else [])


def check_ransac_per_problem(tvf, Cs, Ks, method, refine, H, seeds):
    s = ro.SAMPLE_SIZE[method]
    kw = dict(method=method, hypotheses=H, threshold=1.0, refine=refine)
    rag = tvf.ransac_pose(Cs, Ks, seed=seeds, **kw)
    for b, Cb in enumerate(Cs):
        got = [rag[0][b], rag[1][b], rag[2][b], rag[3][b], rag[4][b], rag.status[b]] + ([rag.lo_done[b]] if refine else [])
        if Cb.shape[1] < s:
            assert rag.status[b] == ST_TOO_FEW, b
            assert np.all(np.isnan(rag[0][b])) and np.all(np.isnan(rag[1][b])), b
            assert rag[2][b].shape == (Cb.shape[1],) and not rag[2][b].any() and rag[3][b] == 0, b
            assert np.all(rag[4][b] == -1) and (not refine or rag.lo_done[b] == 0), b
            continue
        one = tvf.ransac_pose(Cb[None], Ks[b:b + 1], seed=seeds[b:b + 1], **kw)
        want = [x[0] for x in ransac_fields(one, refine)]
        assert same_bits([np.asarray(x) for x in got], [np.asarray(x).astype(np.asarray(y).dtype) for x, y in zip(want, got)]), b
    return rag


@pytest.mark.parametrize("refine", [False, True])
@pytest.mark.parametrize("method", [1, 7])
def test_ransac_equals_uniform_calls_on_epfl(tvf, epfl_all, method, refine):
    Cs, Ks = epfl_all
    assert len(Cs) == 120
    check_ransac_per_problem(tvf, Cs, Ks, method, refine, 256, np.arange(1, 121, dtype=np.uint64))


@pytest.mark.parametrize("refine", [False, True])
@pytest.mark.parametrize("method", [1, 7])
def test_ransac_equals_uniform_calls_on_edge_sizes(tvf, method, refine):
    Cs, Ks = edge_batch(ro.SAMPLE_SIZE[method])
    check_ransac_per_problem(tvf, Cs, Ks, method, refine, 64, np.arange(40, 40 + len(Cs), dtype=np.uint64))


def adjusted_sets(tvf, Cs, Ks):
    """consensus columns and poses of a plain RANSAC over (Cs, Ks), with the too-few sizes 0 and 3 appended"""
    res = tvf.ransac_pose(Cs, Ks, method=1, hypotheses=128, threshold=1.0, seed=7)
    keep = [b for b in range(len(Cs)) if res.status[b] == 0]
    Cm = [Cs[b][:, res[2][b]] for b in keep] + [Cs[keep[0]][:, :0], Cs[keep[0]][:, :3]]
    K = np.concatenate([Ks[keep], Ks[keep[:2]]])
    R2 = np.concatenate([res[0][keep], res[0][keep[:2]]])
    R3 = np.concatenate([res[1][keep], res[1][keep[:2]]])
    return Cm, K, R2, R3


@pytest.mark.parametrize("which", ["epfl", "edge"])
def test_bundle_adjust_and_covariance_equal_uniform_calls(tvf, epfl_all, which):
    Cs, Ks = epfl_all if which == "epfl" else edge_batch(7)
    Cm, K, R2, R3 = adjusted_sets(tvf, Cs, Ks)
    ba = tvf.bundle_adjust(Cm, K, R2, R3)
    cov = tvf.ba_covariance(Cm, K, ba[0], ba[1], ba[2], points=True)
    ba0 = tvf.bundle_adjust(Cm, K, R2, R3, [np.nan_to_num(X) for X in ba[2]])     # the reconst0 path
    for b, Cb in enumerate(Cm):
        n = Cb.shape[1]
        if n < 4:
            assert ba.status[b] == ST_TOO_FEW and ba[3][b] == 0 and np.isnan(ba.repr_err[b]), b
            assert same_bits([ba[0][b], ba[1][b]], [R2[b], R3[b]]) and ba[2][b].shape == (3, n) and np.all(np.isnan(ba[2][b]))
            assert cov.status[b] == ST_TOO_FEW and np.all(np.isnan(cov[0][b])) and np.isnan(cov[1][b]), b
            assert cov.cov_pts[b].shape == (3, 3, n) and np.all(np.isnan(cov.cov_pts[b])), b
            continue
        one = tvf.bundle_adjust(Cb[None], K[b:b + 1], R2[b:b + 1], R3[b:b + 1])
        assert same_bits([ba[0][b], ba[1][b], ba[2][b], ba[3][b], ba.repr_err[b], ba.status[b]],
                         [one[0][0], one[1][0], one[2][0], one[3][0], one.repr_err[0], one.status[0]]), b
        X0 = np.nan_to_num(ba[2][b])[None]
        one0 = tvf.bundle_adjust(Cb[None], K[b:b + 1], R2[b:b + 1], R3[b:b + 1], X0)
        assert same_bits([ba0[0][b], ba0[2][b], ba0.status[b]], [one0[0][0], one0[2][0], one0.status[0]]), b
        c1 = tvf.ba_covariance(Cb[None], K[b:b + 1], ba[0][b:b + 1], ba[1][b:b + 1], ba[2][b][None], points=True)
        assert same_bits([cov[0][b], cov[1][b], cov.cov_pts[b], cov.status[b]],
                         [c1[0][0], c1[1][0], c1.cov_pts[0], c1.status[0]]), b


def test_consensus_equals_uniform_calls(tvf, epfl_all):
    Cs, Ks = epfl_all
    Cs = Cs[:40] + [Cs[0][:, :0]]
    Ks = np.concatenate([Ks[:40], Ks[:1]])
    R = np.stack([np.eye(3, 4)] * len(Cs))
    R[:, 0, 3] = 1.0
    R3 = R.copy(); R3[:, 1, 3] = 0.5
    mask, cnt = tvf.consensus(Cs, Ks, R, R3, threshold=5.0)
    assert cnt[-1] == 0 and mask[-1].shape == (0,)
    for b, Cb in enumerate(Cs[:-1]):
        m1, c1 = tvf.consensus(Cb[None], Ks[b:b + 1], R[b:b + 1], R3[b:b + 1], threshold=5.0)
        assert np.array_equal(mask[b], m1[0]) and cnt[b] == c1[0], b


def test_invariances(tvf, epfl_all):
    """chunks that cut the batch between and around large problems, a group handle, _dev == host, and a ragged call on
    equal n == the uniform batched call"""
    import torch
    from tft_vs_fund_b200 import _lib, api
    Cs, Ks = edge_batch(7)
    seeds = np.arange(9, 9 + len(Cs), dtype=np.uint64)
    kw = dict(method=1, hypotheses=48, threshold=1.0, seed=seeds, refine=True, lo_rounds=4)
    full = ransac_fields(tvf.ransac_pose(Cs, Ks, **kw), True)
    full = [np.concatenate(full[2])] + full[:2] + full[3:]
    h = _lib.handle()
    for chunk in (1, 3, 7):
        try:
            h.call("tvf_set_chunk", chunk)
            got = ransac_fields(tvf.ransac_pose(Cs, Ks, **kw), True)
        finally:
            h.call("tvf_set_chunk", 0)
        assert same_bits([np.concatenate(got[2])] + got[:2] + got[3:], full), chunk
    got = ransac_fields(api.ransac_pose(Cs, Ks, device=(0, 0), **kw), True)
    assert same_bits([np.concatenate(got[2])] + got[:2] + got[3:], full)

    # _dev == host for RANSAC, the adjustment and the covariance
    dev = torch.device("cuda", 0)
    c, offs = api._pack(Cs, 6)
    B, M = len(Cs), int(offs[-1])
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    op = offs.ctypes.data_as(C.c_void_p)
    d_c, d_k, d_s = d(c), d(api._calm(Ks, B)[0]), d(seeds.view(np.int64))
    o2 = torch.empty((B, 12), dtype=torch.float64, device=dev); o3 = torch.empty_like(o2)
    om = torch.zeros(M, dtype=torch.uint8, device=dev); oc = torch.zeros(B, dtype=torch.int32, device=dev)
    osm = torch.zeros((B, 7), dtype=torch.int32, device=dev); ost = torch.zeros(B, dtype=torch.int32, device=dev)
    olo = torch.zeros(B, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    h.call("tvf_ransac_pose_refined_ragged_dev", 1, p(d_c), p(d_k), 1, op, B, 48, 1.0, p(d_s), 4, p(o2), p(o3), p(om), p(oc),
           p(osm), p(olo), p(ost))
    h.call("tvf_synchronize")
    back = lambda t: api._from_cm(t.cpu().numpy().ravel(), B, (3, 4), True)
    assert same_bits([om.cpu().numpy().astype(bool), back(o2), back(o3), oc.cpu().numpy(), osm.cpu().numpy(),
                      ost.cpu().numpy(), olo.cpu().numpy()], full)

    Cm, K, R2, R3 = adjusted_sets(tvf, *edge_batch(7))
    ba = tvf.bundle_adjust(Cm, K, R2, R3)
    cov = tvf.ba_covariance(Cm, K, ba[0], ba[1], ba[2], points=True)
    c, offs = api._pack(Cm, 6)
    B, M = len(Cm), int(offs[-1])
    op = offs.ctypes.data_as(C.c_void_p)
    d_c, d_k = d(c), d(api._calm(K, B)[0])
    d_r2, d_r3 = d(api._pose_pair(R2, R3, B, True)[0]), d(api._pose_pair(R2, R3, B, True)[1])
    b2 = torch.empty((B, 12), dtype=torch.float64, device=dev); b3 = torch.empty_like(b2)
    bX = torch.empty(3 * M, dtype=torch.float64, device=dev); brep = torch.empty(B, dtype=torch.float64, device=dev)
    bit = torch.zeros(B, dtype=torch.int32, device=dev); bst = torch.zeros(B, dtype=torch.int32, device=dev)
    cc = torch.empty((B, 144), dtype=torch.float64, device=dev); cp = torch.empty(9 * M, dtype=torch.float64, device=dev)
    cs2 = torch.empty(B, dtype=torch.float64, device=dev); cst = torch.zeros(B, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    h.call("tvf_bundle_adjust_ragged_dev", p(d_c), p(d_k), 1, op, B, p(d_r2), p(d_r3), None, p(b2), p(b3), p(bX), p(brep),
           p(bit), p(bst))
    h.call("tvf_ba_covariance_ragged_dev", p(d_c), p(d_k), 1, op, B, p(b2), p(b3), p(bX), p(cc), p(cp), p(cs2), p(cst))
    h.call("tvf_synchronize")
    assert same_bits([back(b2), back(b3), np.concatenate([X.T.ravel() for X in ba[2]]), brep.cpu().numpy(),
                      bit.cpu().numpy(), bst.cpu().numpy()],
                     [ba[0], ba[1], bX.cpu().numpy(), ba.repr_err, ba[3], ba.status])
    assert same_bits([api._from_cm(cc.cpu().numpy().ravel(), B, (12, 12), True), cs2.cpu().numpy(), cst.cpu().numpy()],
                     [cov[0], cov[1], cov.status])
    assert same_bits(api._unpack(cp.cpu().numpy(), offs, (3, 3)), cov.cov_pts)

    # ragged on equal n == the uniform batched call
    Cr, CalM, _, _ = ro.outlier_scenes(0.3, 12, 61)
    for refine in (False, True):
        u = ransac_fields(tvf.ransac_pose(Cr, CalM, method=7, hypotheses=32, threshold=2.0, seed=5, refine=refine), refine)
        r = ransac_fields(tvf.ransac_pose(list(Cr), CalM, method=7, hypotheses=32, threshold=2.0, seed=5, refine=refine), refine)
        assert same_bits([np.stack(r[2])] + r[:2] + r[3:], [u[2]] + u[:2] + u[3:]), refine


def test_nan_problem_and_empty_batch(tvf):
    from tft_vs_fund_b200 import _lib
    Cs, Ks = edge_batch(7)
    big = max(range(len(Cs)), key=lambda b: Cs[b].shape[1] if Cs[b].shape[1] <= 100 else -1)
    Cn = [C.copy() for C in Cs]
    Cn[big][:] = np.nan
    seeds = np.arange(len(Cs), dtype=np.uint64)
    res = tvf.ransac_pose(Cn, Ks, method=1, hypotheses=30, threshold=1.0, seed=seeds)
    one = tvf.ransac_pose(Cn[big][None], Ks[big:big + 1], method=1, hypotheses=30, threshold=1.0, seed=seeds[big:big + 1])
    assert res.status[big] == one.status[0] == _lib.ST_RANSAC_FAILED
    ref = tvf.ransac_pose(Cs, Ks, method=1, hypotheses=30, threshold=1.0, seed=seeds)
    for b in range(len(Cs)):
        if b != big:
            assert same_bits([res[0][b], res[2][b], res[3][b], res.status[b]], [ref[0][b], ref[2][b], ref[3][b], ref.status[b]])
    # B = 0: offsets [0], NULL outputs
    h = _lib.handle()
    z = np.zeros(1, dtype=np.int64)
    zp, buf = z.ctypes.data_as(C.c_void_p), np.zeros(6)
    K = np.zeros(27)
    dp = lambda a: a.ctypes.data_as(_lib.c_double_p)
    assert h.call("tvf_ransac_pose_ragged", 1, dp(buf), dp(K), 0, zp, 0, 16, 1.0, zp, None, None, None, None, None, None) == 0
    assert h.call("tvf_bundle_adjust_ragged", dp(buf), dp(K), 0, zp, 0, dp(buf), dp(buf), None, dp(buf), dp(buf), None, None,
                  None, None) == 0
    assert h.call("tvf_ba_covariance_ragged", dp(buf), dp(K), 0, zp, 0, dp(buf), dp(buf), dp(buf), None, None, None, None) == 0
    assert h.call("tvf_consensus_ragged", dp(buf), dp(K), 0, zp, 0, dp(buf), dp(buf), 1.0, None, None) == 0
    assert tvf.ransac_pose([], np.eye(3).repeat(3, 0), method=1)[3].shape == (0,)


def test_bad_offsets(tvf):
    from tft_vs_fund_b200 import _lib
    h = _lib.handle()
    buf, K = np.zeros(6 * 20), np.zeros(27)
    dp = lambda a: a.ctypes.data_as(_lib.c_double_p)
    out = np.zeros(24)
    for offs in ([1, 10, 20], [0, 12, 10], [0, 20, 20 - (1 << 40)]):
        o = np.array(offs, dtype=np.int64)
        op = o.ctypes.data_as(C.c_void_p)
        for name, args in (("tvf_ransac_pose_ragged", (1, dp(buf), dp(K), 0, op, 2, 16, 1.0, op) + (None,) * 6),
                           ("tvf_bundle_adjust_ragged", (dp(buf), dp(K), 0, op, 2, dp(out), dp(out), None, dp(out), dp(out),
                                                         None, None, None, None)),
                           ("tvf_ba_covariance_ragged", (dp(buf), dp(K), 0, op, 2, dp(out), dp(out), dp(buf), None, None,
                                                         None, None)),
                           ("tvf_consensus_ragged", (dp(buf), dp(K), 0, op, 2, dp(out), dp(out), 1.0, None, None))):
            assert getattr(h.lib, name)(h._h, *args) == _lib.TVF_ERR_ARG, (name, offs)
        assert getattr(h.lib, "tvf_bundle_adjust_ragged")(h._h, dp(buf), dp(K), 0, None, 2, dp(out), dp(out), None, dp(out),
                                                          dp(out), None, None, None, None) == _lib.TVF_ERR_ARG


@pytest.mark.parametrize("refine", [False, True])
def test_run_real_batched_equals_the_loop(tvf, refine):
    from test_gpu_ransac import epfl_dataset
    from tft_vs_fund_b200 import epfl
    for key in ("fountain_P11", "Herz_Jesu_P8"):
        data = epfl_dataset(key)
        for extra in (dict(), dict(bundle_adjust=True, covariance=True)):
            kw = dict(raw_matches=True, ransac_refine=refine, **extra)
            d1, d2 = [], []
            loop = epfl.run_real(data, range(1, 6), details=d1, **kw)
            batch = epfl.run_real(data, range(1, 6), details=d2, batched=True, **kw)
            assert all(np.array_equal(loop[m], batch[m]) for m in (1, 7)), (key, extra)
            for r1, r2 in zip(d1, d2):
                assert r1.keys() == r2.keys()
                for m in (1, 7):
                    assert same_bits(list(r1["res"][m]), list(r2["res"][m]))
                    assert (r1["res"][m].status, r1["res"][m].lo_done) == (r2["res"][m].status, r2["res"][m].lo_done)
                    c1, c2 = r1["consensus"][m], r2["consensus"][m]
                    assert np.array_equal(c1["mask"], c2["mask"]) and (c1["size"], c1["precision"], c1["recall"]) == \
                        (c2["size"], c2["precision"], c2["recall"])
                    if "ba" in r1 and m in r1["ba"]:
                        b1, b2 = r1["ba"][m], r2["ba"][m]
                        assert same_bits(list(b1), list(b2)) and (b1.repr_err, b1.status) == (b2.repr_err, b2.status)
                        assert same_bits([b1.sigma2, b1.pred_rot_err, b1.pred_t_err], [b2.sigma2, b2.pred_rot_err, b2.pred_t_err])
