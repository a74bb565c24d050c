"""Known-answer tests that pin the oracle (SURVEY.md section 4): the reference ships no
golden vectors, so these come from closed forms and ground truth the reference itself provides."""
import os

import numpy as np
import pytest

import oracle as o
from conftest import rel_frob_up_to_sign, rot_angle, vec_angle


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("n", [12, 20, 100])
def test_noise_free_tft_equals_closed_form(seed, n):
    CalM, R_t0, C, _ = o.experiments_subsample(n, 0.0, seed)
    K = CalM[:3]
    R2, R3, Rec, T, it = o.LinearTFTPoseEstimation(C, CalM)
    Tgt = o.TFT_from_P(K @ np.eye(3, 4), K @ R_t0[0], K @ R_t0[1])       # TFT_from_P.m:25-33
    assert rel_frob_up_to_sign(T, Tgt) < 1e-12
    assert it == 0
    assert rot_angle(R_t0[0][:, :3], R2[:, :3]) < 1e-9 and rot_angle(R_t0[1][:, :3], R3[:, :3]) < 1e-9
    assert vec_angle(R_t0[0][:, 3], R2[:, 3]) < 1e-9 and vec_angle(R_t0[1][:, 3], R3[:, 3]) < 1e-9
    assert abs(np.linalg.norm(R2[:, 3]) - 1) < 1e-13
    gt_ratio = np.linalg.norm(R_t0[1][:, 3]) / np.linalg.norm(R_t0[0][:, 3])
    assert abs(np.linalg.norm(R3[:, 3]) - gt_ratio) < 1e-9
    assert o.ReprError([K @ np.eye(3, 4), K @ R2, K @ R3], C, Rec) < 1e-9


@pytest.mark.parametrize("seed", [1, 5])
def test_noise_free_f_method(seed):
    CalM, R_t0, C, _ = o.experiments_subsample(20, 0.0, seed)
    K = CalM[:3]
    R2, R3, Rec, T, it = o.LinearFPoseEstimation(C, CalM)
    assert rot_angle(R_t0[0][:, :3], R2[:, :3]) < 1e-9 and rot_angle(R_t0[1][:, :3], R3[:, :3]) < 1e-9
    Tgt = o.TFT_from_P(K @ np.eye(3, 4), K @ R_t0[0], K @ R_t0[1])
    assert rel_frob_up_to_sign(T, Tgt) < 1e-9
    assert o.ReprError([K @ np.eye(3, 4), K @ R2, K @ R3], C, Rec) < 1e-9


def test_design_matrix_structure():
    """12 non-zeros per row (linearTFT.m:50-61); rank(E)=15 with singular values sqrt2 x3, 1 x12, 0 x3."""
    from oracle.reference_port import _tft_design_matrix
    rs = np.random.RandomState(0)
    p = [rs.standard_normal((2, 9)) for _ in range(3)]
    A = _tft_design_matrix(*p)
    assert np.all((A != 0).sum(axis=1) == 12)
    e31 = rs.standard_normal(3); e31 /= np.linalg.norm(e31)
    e21 = rs.standard_normal(3); e21 /= np.linalg.norm(e21)
    E = np.hstack([np.kron(np.eye(3), np.kron(e31.reshape(3, 1), np.eye(3))), -np.kron(np.eye(9), e21.reshape(3, 1))])
    s = np.linalg.svd(E, compute_uv=False)
    assert o.matlab_rank(E) == 15
    assert np.allclose(s[:3], np.sqrt(2)) and np.allclose(s[3:15], 1.0) and np.all(s[15:] < 1e-12)


def test_linearF_guard_and_rank():
    rs = np.random.RandomState(1)
    with pytest.raises(o.LinearFError, match="At least 8 correspondences"):
        o.linearF(rs.standard_normal((2, 7)), rs.standard_normal((2, 7)))
    with pytest.raises(o.LinearFError):
        o.linearF(rs.standard_normal((2, 9)), rs.standard_normal((2, 8)))
    CalM, _, C, _ = o.experiments_subsample(20, 1.0, 3)
    F = o.linearF(C[0:2], C[2:4])
    assert abs(np.linalg.det(F / np.linalg.norm(F))) < 1e-15
    # homogeneous input is divided through (linearF.m:39-42)
    w = rs.uniform(0.5, 2.0, 20)
    Fh = o.linearF(np.vstack([C[0:2] * w, w]), np.vstack([C[2:4], np.ones(20)]))
    assert rel_frob_up_to_sign(F, Fh) < 1e-9


def test_angerror_degrees_and_complex_acos():
    R_t = np.column_stack([np.eye(3), [1.0, 0, 0]])
    c, s = np.cos(0.3), np.sin(0.3)
    R_e = np.column_stack([np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]]), [0.0, 1, 0]])
    r, t = o.AngError(R_t, R_e)
    assert abs(r - np.degrees(0.3)) < 1e-12 and abs(t - 90.0) < 1e-12
    from oracle.reference_port import _matlab_abs_acos
    assert abs(_matlab_abs_acos(1 + 1e-12) - np.arccosh(1 + 1e-12)) < 1e-18


def test_transform_tft_roundtrip():
    rs = np.random.RandomState(2)
    T = rs.standard_normal((3, 3, 3)); T /= np.linalg.norm(T)
    M = [rs.standard_normal((3, 3)) + 3 * np.eye(3) for _ in range(3)]
    back = o.transform_TFT(o.transform_TFT(T, *M, 0), *M, 1)
    assert rel_frob_up_to_sign(T, back) < 1e-13


def test_triangulation_and_reprerror_forms():
    CalM, R_t0, C, X = o.generateSyntheticScene(30, 0.0, 4, 50, 0)
    K = CalM[:3]
    Ps = [K @ np.eye(3, 4), K @ R_t0[0], K @ R_t0[1]]
    X4 = o.triangulation3D(Ps, C)
    assert np.allclose(np.linalg.norm(X4, axis=0), 1.0)
    Xe = X4[:3] / X4[3]
    assert o.ReprError(Ps, C, Xe) < 1e-9
    assert o.ReprError(Ps, C, X4) < 1e-9
    assert o.ReprError(Ps, C) < 1e-9
    C3 = np.vstack([np.vstack([C[2 * v:2 * v + 2], np.ones(30)]) * (v + 2.0) for v in range(3)])
    assert o.ReprError(Ps, C3, Xe) < 1e-9
    assert np.allclose(o.project3Dpoints(Xe, Ps), C, atol=1e-8)
    assert o.triangulation3D(Ps[:1], C[:2]) is None and o.triangulation3D(Ps, C[:5]) is None


def test_epfl_fountain_top_triplet_prints(epfl_data):
    """experiments_real.m:94-101 prints 1360 valid correspondences with reprojection error 0.2586 (SURVEY.md 4)."""
    path = os.path.join(epfl_data, "fountain-P11")
    idx, cor, names = o.load_corresp_triplets(path)
    d = o.epfl_triplet(path, idx, cor, names, 1)
    assert d["triplet"] == (5, 6, 7)
    assert d["Corresp"].shape == (6, 1400) and d["Corresp_inliers"].shape == (6, 1360)
    assert abs(d["REr"] - 0.2586) < 5e-5
    K = d["CalM"][:3]
    assert abs(K[0, 0] - 2759.48) < 1e-9 and abs(K[1, 1] - 2764.16) < 1e-9
