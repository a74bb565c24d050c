"""The projected 15x15 Gram of linearTFT's second step, H = Up' G Up, formed straight from the 96 moments and the
epipoles as the stage-2 kernels do (form_h15 in tvf_core_kernels.cu, DESIGN.md §3.4), against the product through
the 27x27 Gram (tests/kernel_model.py).  CPU only."""
import os

import numpy as np
import pytest

import kernel_model as km
import oracle as o

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# the 15 pairs {a,b} in the order the kernel's lanes take them, and sym6 -> (i, i')
PAIRS = [(a, b) for a in range(5) for b in range(a, 5)]
SYM6_PAIRS = [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]


def cforms(p, q):
    """Quadratic forms p' N_g q of the four constant parts of M(x,y) = sum_g m4_g N_g."""
    return np.array([p[0] * q[0] + p[1] * q[1], p[0] * q[2] + p[2] * q[0], p[1] * q[2] + p[2] * q[1], p[2] * q[2]])


def projected_gram_from_moments(mom, e21, e31):
    """H[(i,a),(i',b)] = sum_{beta,gamma} mom[16 sym6(i,i') + 4 beta + gamma] c_beta(q_a,q_b) c_gamma(p_a,p_b):
    first the sum over gamma (view 2), then over beta (view 3)."""
    u1, u2 = km.onb(e21)
    v1, v2 = km.onb(e31)
    P = [e21, e21, e21, u1, u2]
    Q = [e31, v1, v2, e31, e31]
    M = np.asarray(mom).reshape(6, 4, 4)          # [sym6][beta][gamma]
    H = np.zeros((15, 15))
    for a, b in PAIRS:
        h = (M @ cforms(P[a], P[b])) @ cforms(Q[a], Q[b])
        for al, (i, i2) in enumerate(SYM6_PAIRS):
            for r, c in ((5 * i + a, 5 * i2 + b), (5 * i + b, 5 * i2 + a), (5 * i2 + a, 5 * i + b), (5 * i2 + b, 5 * i + a)):
                H[r, c] = h[al]
    return H


def projected_gram_via_gram27(mom, e21, e31):
    """Up' G Up with Up in the kernels' j + 3k + 9i order (kernel_model.constrained_tft)."""
    u1, u2 = km.onb(e21)
    v1, v2 = km.onb(e31)
    Bs = [np.outer(e21, e31), np.outer(e21, v1), np.outer(e21, v2), np.outer(u1, e31), np.outer(u2, e31)]
    Up = np.zeros((27, 15))
    for i in range(3):
        for a, B in enumerate(Bs):
            Up[9 * i:9 * i + 9, 5 * i + a] = B.reshape(9, order='F')
    return Up.T @ km.gram27_from_moments(mom) @ Up


def _moments_and_epipoles(C):
    xs = [o.Normalize2Ddata(C[2 * v:2 * v + 2])[0] for v in range(3)]
    mom = km.moments96(*xs)
    t, _ = km.smallest_eigvec_spd(km.gram27_from_moments(mom))
    e21, e31 = km.epipoles(t.reshape(3, 3, 3, order="F"))
    return mom, e21, e31


def _check(mom, e21, e31):
    Hf = projected_gram_from_moments(mom, e21, e31)
    Hg = projected_gram_via_gram27(mom, e21, e31)
    err = np.linalg.norm(Hf - Hg) / np.linalg.norm(Hg)
    assert err < 1e-14, err
    assert np.array_equal(Hf, Hf.T)
    return err


def test_projected_gram_golden_sweep():
    d = np.load(os.path.join(GOLDEN, "sweep_n20.npz"))
    worst = 0.0
    for C in d["Corresp"]:
        worst = max(worst, _check(*_moments_and_epipoles(C)))
    assert worst > 0.0          # the two routes round differently; identical results would mean one route was not taken


@pytest.mark.parametrize("n", [7, 8, 12, 100])
@pytest.mark.parametrize("noise", [0.0, 1.0])
def test_projected_gram_sizes(n, noise):
    for seed in (1, 2, 3):
        _, _, C, _ = o.experiments_subsample(n, noise, seed)
        _check(*_moments_and_epipoles(C))


def test_projected_gram_any_unit_epipoles():
    """The identity needs only unit e21, e31 (onb completes them), not epipoles of the data."""
    rng = np.random.default_rng(5)
    for _ in range(50):
        mom = km.moments96(*rng.normal(size=(3, 2, 30)))
        e21, e31 = (v / np.linalg.norm(v) for v in rng.normal(size=(2, 3)))
        _check(mom, e21, e31)
