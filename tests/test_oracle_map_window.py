"""The CPU restatement of gm_map_evict / gm_map_merge (tests/map_window_oracle.py) on hand-made voxel sets: centre cells
of negative coordinates and of centres just below a cell face, the keep predicate at half_cells 0 and very large, the
GMM1 round trip, and merges with overlapping keys.  No device needed."""
import numpy as np
import pytest

import map_window_oracle as W


def _map(leaf, ijk, counts, sums):
    return W.make(leaf, W.pack(np.asarray(ijk, np.int64)), counts, sums)


def test_center_cell_floors_negative_coordinates():
    assert W.center_cell((0.0, 0.05, 0.15), 0.1).tolist() == [0, 0, 1]
    assert W.center_cell((-0.01, -0.1, -0.25), 0.1).tolist() == [-1, -1, -3]
    assert W.center_cell((-1e-30, 0.0, -0.0), 0.1).tolist() == [-1, 0, 0]


def test_center_cell_is_the_float_product_just_below_a_face():
    # -0.05 at a leaf of 0.1: float32(-0.05) * float32(10) rounds to -0.5 exactly -> -1; -0.1 lands on the face itself
    inv = W.inv_leaf(0.1)
    assert inv == np.float32(10.0)
    assert W.center_cell((-0.05, -0.1, np.nextafter(np.float32(-0.1), np.float32(0.0))), 0.1).tolist() == [-1, -1, -1]
    # a value whose float product rounds up onto the face: the float rule, not the real-number one, decides
    x = np.float32(0.3)                                      # 0.3f * 10.0f = 3.0000001... rounds to 3.0f
    assert np.float32(x * inv) == np.float32(3.0) and W.center_cell((x, 0, 0), 0.1)[0] == 3
    assert float(x) * 10.0 < 3.0 + 1e-6
    y = np.nextafter(np.float32(0.3), np.float32(0.0))       # just below: still a product that floors to 2
    assert W.center_cell((y, 0, 0), 0.1)[0] == int(np.floor(np.float32(y * inv)))


def test_center_cell_refuses_what_gm_map_evict_refuses():
    for c in ((np.nan, 0, 0), (0, np.inf, 0), (0, 0, -np.inf), (2.0e5, 0, 0), (0, -104857.7, 0)):
        assert W.center_cell(c, 0.1) is None, c
    assert W.center_cell((104857.5, 0, 0), 0.1) is not None  # cell 2^20 - 3: inside
    assert W.center_cell((-104857.6, 0, 0), 0.1).tolist()[0] == -(1 << 20)


def test_keep_predicate_is_a_chebyshev_cube():
    ijk = np.array([[0, 0, 0], [2, 0, 0], [-2, 2, -2], [3, 0, 0], [0, -3, 0], [0, 0, 3], [-5, 5, 5]], np.int64)
    assert W.keep(ijk, (0, 0, 0), 2).tolist() == [True, True, True, False, False, False, False]
    assert W.keep(ijk, (0, 0, 0), 0).tolist() == [True] + [False] * 6
    assert W.keep(ijk, (-3, 3, 3), 2).tolist() == [False] * 6 + [True]
    assert W.keep(ijk, (-3, 3, -1), 2).tolist() == [False, False, True, False, False, False, False]
    far = np.array([[-(1 << 20), -(1 << 20), -(1 << 20)], [(1 << 20) - 1] * 3], np.int64)
    assert W.keep(far, ((1 << 20) - 1, 0, 0), 2**31 - 1).all()                  # very large: everything
    assert W.keep(far, ((1 << 20) - 1,) * 3, (1 << 21) - 2).tolist() == [False, True]


def test_evict_splits_and_merge_gives_back_the_map():
    rng = np.random.default_rng(3)
    ijk = np.unique(rng.integers(-40, 40, (500, 3)), axis=0)
    cnt = rng.integers(1, 50, ijk.shape[0]).astype(np.int32)
    sums = rng.integers(-(1 << 40), 1 << 40, (ijk.shape[0], 3))
    m = _map(0.1, ijk, cnt, sums)
    for c, h in (((-0.05, 0.31, -2.0), 10), ((1.0, 1.0, 1.0), 0), ((0, 0, 0), 1000)):
        kept, gone = W.evict(m, c, h)
        assert kept["keys"].shape[0] + gone["keys"].shape[0] == m["keys"].shape[0]
        assert W.equal(W.merge(gone, kept), m) and W.equal(W.merge(kept, gone), m)
        cell = W.center_cell(c, 0.1)
        assert (np.abs(W.unpack(kept["keys"]) - cell).max(axis=1, initial=0) <= h).all()
    assert W.evict(m, (0, 0, 0), 1000)[1]["keys"].shape[0] == 0


def test_merge_with_overlapping_keys_adds_counts_and_sums():
    a = _map(0.1, [[0, 0, 0], [1, 0, 0], [-1, -1, -1]], [1, 2, 3], [[1, 2, 3], [4, 5, 6], [-7, -8, -9]])
    b = _map(0.1, [[1, 0, 0], [5, 5, 5], [-1, -1, -1]], [10, 20, 30], [[40, 50, 60], [1, 1, 1], [-70, 80, -90]])
    m = W.merge(a, b)
    assert W.unpack(m["keys"]).tolist() == [[-1, -1, -1], [0, 0, 0], [1, 0, 0], [5, 5, 5]]
    assert m["counts"].tolist() == [33, 1, 12, 20]
    assert m["sums"].tolist() == [[-77, 72, -99], [1, 2, 3], [44, 55, 66], [1, 1, 1]]
    assert W.equal(W.merge(b, a), m)
    e = W.make(0.1, np.zeros(0, np.uint64), np.zeros(0, np.int32), np.zeros((0, 3), np.int64))
    assert W.equal(W.merge(e, m), m) and W.equal(W.merge(m, e), m)


def test_gmm1_round_trip(tmp_path):
    m = _map(0.25, [[3, -2, 1], [-4, 0, 0]], [7, 9], [[1 << 40, -(1 << 41), 5], [0, 0, -1]])
    b = W.write_gmm1(m)
    assert len(b) == 24 + 36 * 2
    p = tmp_path / "m.gmm"
    p.write_bytes(b)
    r = W.read_gmm1(str(p))
    assert r["leaf"] == 0.25 and W.equal(r, m) and W.write_gmm1(r) == b
    assert np.array_equal(W.centroids(m), (m["sums"] / 1048576.0 / m["counts"][:, None]).astype(np.float32))
    with pytest.raises(AssertionError):
        W.read_gmm1(b[:-1])
