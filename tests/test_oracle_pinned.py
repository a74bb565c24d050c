"""Pins the oracle restatement against the reference's own source.

tests/golden/*.npz hold `ref_*` arrays produced by executing the UNMODIFIED reference .m files
(TFT_methods, F_methods, auxiliar_functions of the original project) with oracle/mini_matlab.py, a
minimal MATLAB-subset interpreter whose built-ins are NumPy/LAPACK.  The oracle
(oracle/reference_port.py) must reproduce them."""
import os

import numpy as np
import pytest

import oracle as o
from conftest import ROOT, rel_frob_up_to_sign, votes8_equal

GOLDEN = os.path.join(ROOT, "tests", "golden")


def _load_golden(name):
    """A golden file together with its `_ref` companion (the ref_* arrays, kept apart where one file would exceed 1 MB)."""
    d = dict(np.load(os.path.join(GOLDEN, name)))
    ref = os.path.join(GOLDEN, name.replace(".npz", "_ref.npz"))
    if os.path.exists(ref):
        d.update(np.load(ref))
    return d


def _run_oracle(method, C, CalM):
    K = [CalM[0:3], CalM[3:6], CalM[6:9]]
    fn = o.LinearTFTPoseEstimation if method == "tft" else o.LinearFPoseEstimation
    R2, R3, Rec, T, it = fn(C, CalM)
    return R2, R3, Rec, T, o.ReprError([K[0] @ np.eye(3, 4), K[1] @ R2, K[2] @ R3], C, Rec)


@pytest.mark.parametrize("name,stride", [("sweep_n20.npz", 7), ("example_n100.npz", 1), ("epfl_triplets.npz", 3)])
@pytest.mark.parametrize("method", ["tft", "f"])
def test_oracle_reproduces_reference_source_outputs(name, stride, method):
    g = _load_golden(name)
    assert "ref_%s_T" % method in g, "golden file lacks interpreter outputs: regenerate with make_golden.py"
    for b in range(0, g["Corresp"].shape[0], stride):
        got = _run_oracle(method, g["Corresp"][b], g["CalM"][b])
        for k, key in enumerate(("Rt2", "Rt3", "Reconst", "T", "repr")):
            ref = g["ref_%s_%s" % (method, key)][b]
            # same LAPACK underneath: agreement to rounding, not merely to the parity tolerances
            scale = max(1.0, float(np.max(np.abs(ref))))
            assert np.max(np.abs(np.asarray(got[k]) - ref)) <= 1e-9 * scale, (name, method, b, key)
        # and the stored oracle outputs are the ones the GPU tests compare against
        assert rel_frob_up_to_sign(g["%s_T" % method][b], g["ref_%s_T" % method][b]) < 1e-12


@pytest.mark.parametrize("name,stride", [("optimf_n20.npz", 9), ("optimf_n12.npz", 5)])
def test_gauss_helmert_port_reproduces_reference_source_outputs(name, stride):
    """SURVEY 8 f4: oracle/gauss_helmert_port.py (Gauss_Helmert.m, optimF.m, OptimFPoseEstimation.m) against the
    outputs of the reference's unmodified .m files (ref_optf_*), iteration counts included."""
    g = np.load(os.path.join(GOLDEN, name))
    assert "ref_optf_T" in g.files, "golden file lacks interpreter outputs: regenerate with make_golden.py optimf"
    for b in range(0, g["Corresp"].shape[0], stride):
        C, CalM = g["Corresp"][b], g["CalM"][b]
        R2, R3, Rec, T, it = o.OptimFPoseEstimation(C, CalM)
        assert it == int(g["ref_optf_iter"][b])
        for got, key in ((R2, "Rt2"), (R3, "Rt3"), (Rec, "Reconst"), (T, "T")):
            ref = g["ref_optf_" + key][b]
            assert np.max(np.abs(got - ref)) <= 1e-9 * max(1.0, float(np.max(np.abs(ref)))), (name, b, key)
        F, it1 = o.optimF(C[0:2], C[2:4])
        assert it1 == int(g["ref_optf_iter_single"][b])
        assert rel_frob_up_to_sign(F, g["ref_optf_F_single"][b]) < 1e-11
    # all stored oracle outputs agree with the interpreter's
    assert np.array_equal(g["optf_iter"], g["ref_optf_iter"].astype(g["optf_iter"].dtype))
    for b in range(g["Corresp"].shape[0]):
        assert rel_frob_up_to_sign(g["optf_T"][b], g["ref_optf_T"][b]) < 1e-10


def test_faugpapa_constraint_jacobian_is_not_the_derivative():
    """SURVEY 8 f4, second step (FaugPapaTFTPoseEstimation): why the method has no well-defined oracle at the north-star
    tolerances.  The analytic Jacobian C of constraints 4..12 in the restated constrGH is not the derivative of its g
    (the minors are taken as if reshape([..],3,3) stacked the vectors as columns; MATLAB stacks them as rows), and the
    39 x 39 KKT matrix is rank deficient (12 constraints of rank 9) with pinv keeping the 1e-12-shifted singular
    values.  Two LAPACK-based executions of the same .m text then differ by ~1e-5 in T (DESIGN.md 8)."""
    from oracle.gauss_helmert_port import constrGH_FaugPapa
    rs = np.random.RandomState(1)
    obs = rs.standard_normal(30); x = rs.standard_normal(27)
    got = constrGH_FaugPapa(obs, x)
    eps = 1e-6
    Cfd = np.stack([(constrGH_FaugPapa(obs, x + eps * e)[1] - constrGH_FaugPapa(obs, x - eps * e)[1]) / (2 * eps)
                    for e in np.eye(27)], axis=1)
    assert np.abs(Cfd[:3] - got[4][:3]).max() < 1e-6            # det(T_i) rows: consistent
    assert np.abs(Cfd[3:] - got[4][3:]).max() > 1e-2            # rows 4..12: NOT the Jacobian of g


def test_matlab_pinv_definition():
    rs = np.random.RandomState(0)
    A = rs.standard_normal((7, 4)); A[:, 3] = A[:, 0] + A[:, 1]             # rank 3
    P = o.matlab_pinv(A)
    assert np.allclose(A @ P @ A, A, atol=1e-12) and np.allclose(P @ A @ P, P, atol=1e-12)
    assert np.linalg.matrix_rank(P) == 3
    D = np.diag([4.0, 1e-18, 2.0])
    assert np.array_equal(o.matlab_pinv(D), np.diag([0.25, 0.0, 0.5]))     # entries below max(size)*eps(norm) vanish
    assert o.matlab_pinv(np.zeros((0, 3))).shape == (3, 0)


def test_epfl_all_triplets_golden_is_pinned_by_the_reference_sources():
    """tests/golden/epfl_all_triplets.npz (all 70 + 50 triplets of experiments_real.m:31-36): the stored oracle
    outputs agree with what the reference's unmodified .m files produced (ref_*), tensor and the three error columns
    ([ReprError over all inliers, rot_err, t_err], experiments_real.m:130-136)."""
    g = np.load(os.path.join(GOLDEN, "epfl_all_triplets.npz"))
    assert g["Corresp"].shape[0] == 120 and list(np.bincount(g["dataset"])) == [70, 50]
    assert g["n_inliers"][0] == 1360 and abs(g["gt_repr"][0] - 0.2586) < 5e-5          # what experiments_real.m:101 prints
    for m in ("tft", "f"):
        for b in range(120):
            assert rel_frob_up_to_sign(g[m + "_T"][b], g["ref_" + m + "_T"][b]) < 1e-10, (m, b)
        assert np.max(np.abs(g["real_" + m][:, 0] - g["ref_real_" + m][:, 0])) < 1e-9
        assert np.max(np.abs(g["real_" + m][:, 1:] - g["ref_real_" + m][:, 1:])) < 1e-6
    # live: the oracle on the stored sample reproduces the stored tensor and votes (every 17th triplet)
    from make_golden_access import oracle_votes
    for b in range(0, 120, 17):
        ns = int(g["n_sample"][b])
        C, CalM = g["Corresp"][b][:, :ns], g["CalM"][b]
        assert rel_frob_up_to_sign(o.LinearTFTPoseEstimation(C, CalM)[3], g["tft_T"][b]) < 1e-12
        tv, fv = oracle_votes(C, CalM)
        assert votes8_equal(tv, g["tft_votes"][b]) and votes8_equal(fv, g["f_votes"][b])      # labels: see conftest


@pytest.mark.parametrize("name", ["sweep_n20.npz", "example_n100.npz", "epfl_triplets.npz"])
def test_votes_in_the_goldens_are_the_oracles(name):
    from make_golden_access import oracle_votes
    g = np.load(os.path.join(GOLDEN, name))
    assert "tft_votes" in g.files and "f_votes" in g.files
    n = g["Corresp"].shape[2]
    for b in range(0, g["Corresp"].shape[0], 23):
        tv, fv = oracle_votes(g["Corresp"][b], g["CalM"][b])
        assert votes8_equal(tv, g["tft_votes"][b]) and votes8_equal(fv, g["f_votes"][b])
    # SURVEY App. C: one candidate at +2n, one at -2n, two at 0 on regular data
    v = g["tft_votes"].reshape(-1, 4)
    assert np.all(np.sort(v, axis=1) == np.array([-2 * n, 0, 0, 2 * n]))
