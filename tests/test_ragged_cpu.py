"""The ragged-batch layout in Python (api._pack / api._unpack, include/tvf.h): round trips, shapes, and the offsets
check, without a GPU."""
import numpy as np
import pytest


def test_pack_round_trip():
    from tft_vs_fund_b200 import api
    rs = np.random.RandomState(0)
    mats = [rs.rand(6, n) for n in (5, 0, 1, 17)]
    buf, offs = api._pack(mats, 6)
    assert offs.dtype == np.int64 and list(offs) == [0, 5, 5, 6, 23]
    assert buf.shape == (23, 6) and buf.flags.c_contiguous
    assert np.array_equal(buf[5], mats[2][:, 0])                  # 48 contiguous bytes per match
    back = api._unpack(buf, offs, (6,))
    assert all(a.shape == b.shape and np.array_equal(a, b) for a, b in zip(back, mats))


def test_unpack_per_match_shapes():
    from tft_vs_fund_b200 import api
    offs = np.array([0, 2, 2, 5])
    cov = np.arange(9 * 5, dtype=np.float64)
    out = api._unpack(cov, offs, (3, 3))
    assert [o.shape for o in out] == [(3, 3, 2), (3, 3, 0), (3, 3, 3)]
    assert out[0][1, 0, 0] == 1.0 and out[0][0, 1, 0] == 3.0 and out[2][0, 0, 0] == 18.0     # column-major per match
    flags = api._unpack(np.array([1, 0, 1, 1, 0], dtype=np.uint8), offs, ())
    assert [f.tolist() for f in flags] == [[1, 0], [], [1, 1, 0]]


def test_empty_batch():
    from tft_vs_fund_b200 import api
    buf, offs = api._pack([], 6)
    assert buf.shape == (0, 6) and list(offs) == [0]
    assert api._unpack(np.zeros(0), offs, (3,)) == []


@pytest.mark.parametrize("offs, B", [([0, 3, 2], 2), ([1, 3, 4], 2), ([0, 3], 2), ([0, 1, 2, 3], 2)])
def test_bad_offsets_are_rejected(offs, B):
    from tft_vs_fund_b200 import api
    with pytest.raises(ValueError):
        api._check_offsets(offs, B)


def test_pack_rejects_wrong_rows():
    from tft_vs_fund_b200 import api
    with pytest.raises(ValueError):
        api._pack([np.zeros((6, 3)), np.zeros((3, 3))], 6)
    with pytest.raises(ValueError):
        api._unpack(np.zeros(7), np.array([0, 2]), (3,))
