"""The RANSAC estimator's per-thread pieces on the CPU: csrc/tvf_ransac.cuh compiled with g++ (the same source the
kernels inline) against the NumPy twin in tests/ransac_oracle.py -- the sampler integer for integer, and the inlier
test against the oracle's triangulation."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle as o
import ransac_oracle as ro
from conftest import ROOT

cm = lambda a: np.ascontiguousarray(np.asarray(a, dtype=np.float64).T).ravel()   # 2-D column-major
dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int))


@pytest.fixture(scope="module")
def rhost(tmp_path_factory):
    inc = os.path.join(ROOT, "tft_vs_fund_b200", "csrc")
    so = str(tmp_path_factory.mktemp("ransachost") / "libransachost.so")
    subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-ffp-contract=off", "-I", inc, "-x", "c++",
                           os.path.join(ROOT, "tests", "hostcheck", "ransac_hostcheck.cpp"), "-o", so])
    lib = C.CDLL(so)
    lib.hc_ransac_mix64.restype = C.c_uint64
    lib.hc_ransac_mix64.argtypes = [C.c_uint64]
    return lib


def host_samples(rhost, seeds, hs, ns, ss):
    seeds = np.ascontiguousarray(seeds, dtype=np.uint64); hs = np.ascontiguousarray(hs, dtype=np.uint32)
    ns = np.ascontiguousarray(ns, dtype=np.int32); ss = np.ascontiguousarray(ss, dtype=np.int32)
    out = np.full((seeds.size, 8), -7, dtype=np.int32)
    rhost.hc_ransac_samples(seeds.ctypes.data_as(C.c_void_p), hs.ctypes.data_as(C.c_void_p), ip(ns), ip(ss),
                            int(seeds.size), ip(out))
    return out


def test_mix64_is_splitmix64(rhost):
    # splitmix64 seeded with 0 yields 0xE220A8397B1DCDAF first: its output function of 0 + golden gamma
    assert rhost.hc_ransac_mix64(0) == 0xE220A8397B1DCDAF == int(ro.mix64(np.uint64(0)))
    for z in (1, 12345, 2 ** 63, 2 ** 64 - 1):
        assert rhost.hc_ransac_mix64(z) == int(ro.mix64(np.uint64(z)))


def test_sampler_equals_the_numpy_twin(rhost):
    """10^5 (seed, h, j, n, s) draws: the header's indices equal the twin's integer for integer."""
    rs = np.random.RandomState(3)
    count = 100000 // 7
    seeds = rs.randint(0, 2 ** 63, size=count, dtype=np.int64).astype(np.uint64) * np.uint64(2) + rs.randint(0, 2, count).astype(np.uint64)
    hs = rs.randint(0, 1 << 24, size=count).astype(np.uint32)
    ss = rs.choice([7, 8], size=count)
    ns = ss + rs.choice([0, 1, 2, 5, 30, 1393, 10 ** 6], size=count)
    got = host_samples(rhost, seeds, hs, ns, ss)
    draws = 0
    for s in (7, 8):
        for n in np.unique(ns[ss == s]):
            sel = np.flatnonzero((ss == s) & (ns == n))
            for k in sel:
                want = ro.sample(seeds[k], [hs[k]], int(n), s)[0]
                assert np.array_equal(got[k, :s], want), (seeds[k], hs[k], n, s)
                draws += s
    assert draws >= 100000 - 7 * 8


def test_samples_distinct_and_in_range(rhost):
    rs = np.random.RandomState(4)
    for s in (7, 8):
        for n in (s, s + 1, s + 3, 40, 1400):
            count = 2000
            seeds = rs.randint(0, 2 ** 62, size=count, dtype=np.int64).astype(np.uint64)
            got = host_samples(rhost, seeds, np.arange(count), np.full(count, n), np.full(count, s))[:, :s]
            assert np.all((got >= 0) & (got < n)), (n, s)
            assert all(len(set(r)) == s for r in got), (n, s)
            if n == s:
                assert np.all(np.sort(got, axis=1) == np.arange(s))


def random_problem(rs, n):
    """Random cameras (rotations, translations, calibrations) and matches near and far from consistent."""
    CalM, R_t0, Cr, _ = o.experiments_subsample(n, 1.0, int(rs.randint(1, 1000)))
    Cr = Cr.copy()
    bad = rs.rand(n) < 0.3
    Cr[:, bad] += rs.uniform(-8.0, 8.0, size=(6, int(bad.sum())))
    return CalM, R_t0, Cr


def host_inliers(rhost, CalM, R2, R3, Cr, th):
    n = Cr.shape[1]
    flags = np.zeros(n, dtype=np.int32); mx = np.zeros(n)
    rhost.hc_ransac_inliers(dp(cm(CalM)), dp(cm(R2)), dp(cm(R3)), dp(cm(Cr)), n, C.c_double(th), ip(flags), dp(mx))
    return flags.astype(bool), mx


def test_inlier_test_equals_the_oracle(rhost):
    rs = np.random.RandomState(5)
    checked = 0
    for trial in range(12):
        CalM, R_t0, Cr = random_problem(rs, 60)
        R2 = R_t0[0].copy(); R3 = R_t0[1].copy()
        if trial % 2:                       # a perturbed pose, so that many residuals are near the threshold
            R2[:, 3] += rs.normal(0, 0.01, 3); R3[:, 3] += rs.normal(0, 0.01, 3)
        for th in (0.5, 1.0, 3.0):
            got, mx = host_inliers(rhost, CalM, R2, R3, Cr, th)
            want, wmx = ro.inliers(Cr, CalM, R2, R3, th)
            assert np.allclose(mx, wmx, rtol=1e-9, atol=1e-9)
            far = np.abs(wmx - th) > 1e-9
            assert np.array_equal(got[far], want[far]), (trial, th)
            checked += int(far.sum())
    assert checked > 1500


def test_inlier_test_nan_and_inf(rhost):
    rs = np.random.RandomState(6)
    CalM, R_t0, Cr = random_problem(rs, 10)
    Cr[3, 2] = np.nan
    Cr[0, 5] = np.inf
    Cr[5, 7] = -np.inf
    got, mx = host_inliers(rhost, CalM, R_t0[0], R_t0[1], Cr, 1e6)
    want, wmx = ro.inliers(Cr, CalM, R_t0[0], R_t0[1], 1e6)
    assert not got[2] and not got[5] and not got[7]
    assert not np.isfinite(mx[[2, 5, 7]]).any()
    assert np.array_equal(got, want) and np.array_equal(np.isfinite(mx), np.isfinite(wmx))
    # a pose that is not finite: every match is an outlier
    got, mx = host_inliers(rhost, CalM, np.full((3, 4), np.nan), R_t0[1], Cr, 1e6)
    assert not got.any() and not np.isfinite(mx).any()
