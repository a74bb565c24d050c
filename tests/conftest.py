import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def libtvf_path():
    """libtvf.so, (re)built with nvcc when sources are newer (cross-compiles without a GPU)."""
    from tft_vs_fund_b200 import build
    return build.build()


@pytest.fixture(scope="session")
def hostcheck():
    """TEST-ONLY host build of the csrc headers (thread-level device math compiled with g++)."""
    src = os.path.join(ROOT, "tests", "hostcheck", "hostcheck.cpp")
    out_dir = os.path.join(ROOT, "tests", "hostcheck", "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libhostcheck.so")
    inc = os.path.join(ROOT, "tft_vs_fund_b200", "csrc")
    deps = [src] + [os.path.join(inc, f) for f in ("tvf_math.cuh", "tvf_pose.cuh", "tvf_scene.cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-ffp-contract=off", "-I", inc,
                               "-x", "c++", src, "-o", so])
    return ctypes.CDLL(so)


@pytest.fixture(scope="session")
def tvf(libtvf_path):
    """The product package with a live handle (GPU tests only)."""
    import tft_vs_fund_b200 as pkg
    pkg.handle()          # raises loudly when there is no CUDA device / library
    return pkg


@pytest.fixture(scope="session")
def epfl_data(tmp_path_factory):
    """Directory with fountain-P11/ and Herz-Jesu-P8/ laid out as the reference's Data/ folders (Corresp_triplets.mat
    and one .camera file per image), written from tests/golden/epfl_inputs.npz: indexes_sorted and the match lists of
    the tested triplets, and the calibration and orientation of every image.  Image names and sizes are not stored
    there, so the images are named 0000, 0001, ... and given the EPFL size 3072 x 2048."""
    import scipy.io as sio
    inp = np.load(os.path.join(ROOT, "tests", "golden", "epfl_inputs.npz"))
    root = tmp_path_factory.mktemp("epfl_data")
    for ds in ("fountain-P11", "Herz-Jesu-P8"):
        key = ds.replace("-", "_")
        K, R, t = inp[key + "_K"], inp[key + "_R"], inp[key + "_t"]
        idx, offs, matches = inp[key + "_indexes_sorted"], inp[key + "_offsets"], inp[key + "_matches"]
        names = ["%04d" % i for i in range(len(K))]
        path = root / ds
        path.mkdir()
        for name, Ki, Ri, ti in zip(names, K, R, t):
            # readCalibrationOrientation_EPFL.m:8-20: K, a skipped line, R' row by row, camera centre C (t = -R*C), size.
            # The stored R are orthonormal only to the digits of the data files, so C solves R*C = -t (not C = -R'*t).
            rows = list(Ki) + [np.zeros(3)] + list(Ri.T) + [np.linalg.solve(Ri, -ti), [3072.0, 2048.0]]
            (path / (name + ".camera")).write_text("".join(" ".join(repr(float(v)) for v in r) + "\n" for r in rows))
        cells = np.empty((len(K),) * 3, dtype=object)
        for ijk in np.ndindex(cells.shape):
            cells[ijk] = np.zeros((0, 6))
        for r, (i, j, k, _) in enumerate(idx):
            cells[i - 1, j - 1, k - 1] = matches[offs[r]:offs[r + 1]]
        sio.savemat(str(path / "Corresp_triplets.mat"), {"indexes_sorted": idx.astype(np.float64), "Corresp": cells,
                                                         "im_names": np.array(names, dtype=object).reshape(1, -1)})
    return str(root)


# ---- comparison helpers shared by the tests --------------------------------------------------
def rel_frob_up_to_sign(a, b):
    a = np.asarray(a, dtype=np.float64).ravel(); b = np.asarray(b, dtype=np.float64).ravel()
    a = a / np.linalg.norm(a); b = b / np.linalg.norm(b)
    return min(np.linalg.norm(a - b), np.linalg.norm(a + b))


def rot_angle(Ra, Rb):
    """angle of Ra'*Rb in radians, accurate near 0 (acos loses half the digits there)."""
    D = Ra.T @ Rb
    s = 0.5 * np.sqrt((D[2, 1] - D[1, 2]) ** 2 + (D[0, 2] - D[2, 0]) ** 2 + (D[1, 0] - D[0, 1]) ** 2)
    c = 0.5 * (np.trace(D) - 1.0)
    return float(np.arctan2(s, c))


def vec_angle(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float(np.arctan2(np.linalg.norm(np.cross(a, b)), np.dot(a, b)))


# tolerances of BASELINE.json's north_star
TOL_MODEL = 1e-9      # T and F: relative Frobenius, up to sign and scale
TOL_ANGLE = 1e-6      # R / t angular difference, rad
TOL_REPR = 1e-8       # reprojection error, px


def assert_pose_close(ref, got, n_label=""):
    """ref/got: (R_t_2, R_t_3, Reconst, T, repr_err)."""
    R2, R3, Rec, T, rep = ref
    g2, g3, gRec, gT, grep = got
    assert rel_frob_up_to_sign(T, gT) < TOL_MODEL, n_label
    for a, b in ((R2, g2), (R3, g3)):
        assert rot_angle(a[:, :3], b[:, :3]) < TOL_ANGLE, n_label
        assert vec_angle(a[:, 3], b[:, 3]) < TOL_ANGLE, n_label
    assert abs(np.linalg.norm(R3[:, 3]) - np.linalg.norm(g3[:, 3])) <= 1e-9 * np.linalg.norm(R3[:, 3]), n_label
    assert abs(np.linalg.norm(g2[:, 3]) - 1.0) < 1e-12, n_label
    assert np.max(np.abs(Rec - gRec)) <= 1e-8 * max(1.0, np.max(np.abs(Rec))), n_label
    # 1e-8 px; the relative term only matters for failed (hundreds-of-px) solutions whose own
    # sensitivity to a 1-ulp input change already exceeds 1e-8 px (DESIGN.md, "tolerances")
    assert abs(rep - grep) <= TOL_REPR + 1e-10 * abs(rep), n_label


# ---- cheirality votes ---------------------------------------------------------------------------
# The four candidates of recover_R_t are (R,t),(R,-t),(Rp,-t),(Rp,t) with R = U*W*V', Rp = U*W'*V', t = U(:,3)
# (R_t_from_TFT.m:84-97).  svd(E) is defined only up to the signs of its singular-vector pairs (and E has two nearly
# equal singular values); that freedom maps t -> -t and/or swaps R with Rp, i.e. it RELABELS the candidates by one of
# these four permutations (ours[k] = theirs[p[k]]).  The set of (candidate, vote) pairs is invariant; the labels are
# not even stable between two runs of the same LAPACK (thread count changes the last bits of T and with them the
# labels -- observed while generating the goldens), let alone between NumPy and MATLAB.
VOTE_RELABELINGS = ([0, 1, 2, 3], [1, 0, 3, 2], [3, 2, 1, 0], [2, 3, 0, 1])


def votes8_equal(a8, b8):
    """Two 4 + 4 vote vectors (floats, NaN = MATLAB's NaN sum) agree pair by pair under an admissible relabeling."""
    a8 = np.asarray(a8, dtype=np.float64); b8 = np.asarray(b8, dtype=np.float64)
    return all(any(np.array_equal(a8[4 * p:4 * p + 4], b8[4 * p:4 * p + 4][perm], equal_nan=True)
                   for perm in VOTE_RELABELINGS) for p in range(2))


def library_votes_as_float(v10):
    """10 int32 of the library (4 + 4 votes, one NaN bit mask per pair) -> 8 floats with NaN where the mask says so."""
    v10 = np.asarray(v10)
    out = v10[:8].astype(np.float64)
    for p in range(2):
        for k in range(4):
            if (int(v10[8 + p]) >> k) & 1:
                out[4 * p + k] = np.nan
    return out
