"""Product scene generator (tft_vs_fund_b200/scene.py) == oracle restatement of
generateSyntheticScene.m / experiments.m:93-95, bit for bit (projected points, inside-image
compaction order and sub-sample indices are integer/bit-exact requirements of the north star)."""
import numpy as np
import pytest

import oracle as o
from tft_vs_fund_b200 import scene


@pytest.mark.parametrize("args", [(100, 1, 1, 50, 0), (120, 3, 7, 50, 0), (50, 2, 3, 20, 0), (300, 5, 2, 300, 175),
                                   (40, 0, 9, 100, 179.5)])
def test_generate_scene_bit_exact(args):
    a = o.generateSyntheticScene(*args)
    b = scene.generateSyntheticScene(*args)
    assert np.array_equal(a[0], b[0])
    assert all(np.array_equal(x, y) for x, y in zip(a[1], b[1]))
    assert np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
    assert a[2].min() >= 0 and a[2][0::2].max() <= 1800 and a[2][1::2].max() <= 1200


def test_example_config_geometry():
    """Config 1 (example.m:22-28): K, image bounds, P scaled to spectral norm sqrt(24)."""
    K, Ps, R_t = scene.scene_cameras(50, 0)
    assert np.array_equal(K, np.array([[2500.0, 0, 900], [0, 2500, 600], [0, 0, 1]]))
    for P in Ps:
        assert abs(np.linalg.norm(P, 2) - np.sqrt(24)) < 1e-12
    for Rt in R_t:
        assert abs(np.linalg.det(Rt[:, :3]) - 1) < 1e-12


def test_sweep_batch_matches_per_trial_oracle():
    d = scene.sweep_batch(13 * 6, 20)
    for j in range(0, 78, 5):
        CalM, R_t0, C, idx = o.experiments_subsample(20, 0.25 * (j % 13), j // 13 + 1)
        assert np.array_equal(C, d["Corresp"][j])
        assert d["noise"][j] == 0.25 * (j % 13) and d["seed"][j] == j // 13 + 1
    assert np.array_equal(d["CalM"], CalM)
    # any shard of the global trial index reproduces the same trials (multi-GPU sharding)
    s = scene.sweep_batch(20, 20, first_trial=31)
    assert np.array_equal(s["Corresp"], d["Corresp"][31:51])


def test_sweep_batch_workers_identical():
    a = scene.sweep_batch(5000, 20)
    b = scene.sweep_batch(5000, 20, workers=3)
    assert np.array_equal(a["Corresp"], b["Corresp"])


def test_epfl_loaders_match_oracle(epfl_data):
    """Product-side .camera / .mat loaders == oracle restatement, on files in the reference's format."""
    import os
    from tft_vs_fund_b200 import epfl
    path = os.path.join(epfl_data, "Herz-Jesu-P8")
    a = epfl.load_corresp_triplets(path); b = o.load_corresp_triplets(path)
    assert np.array_equal(a[0], b[0]) and a[2] == b[2]
    for name in a[2][:3]:
        x = epfl.readCalibrationOrientation_EPFL(path, name); y = o.readCalibrationOrientation_EPFL(path, name)
        assert all(np.array_equal(p, q) for p, q in zip(x, y))
