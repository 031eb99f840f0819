"""KeyFramePack.select (any keyframe list as a self-contained pack) and parallel.local_selection (a rank's part of a
global selection, in its local indices).  No GPU needed."""
import importlib
from dataclasses import fields

import numpy as np
import pytest

from conftest import PKG


@pytest.fixture(scope="module")
def pack(synth):
    return synth.generate(n_kf=5, seed=77, beams=8, az_steps=256, n_kp=300)[0]


def _equal(a, b):
    assert a.n_kf == b.n_kf and a.n_covis == b.n_covis
    for f in fields(a):
        x, y = getattr(a, f.name), getattr(b, f.name)
        if isinstance(x, np.ndarray):
            assert x.dtype == y.dtype and x.shape == y.shape, f.name
            assert np.array_equal(x, y, equal_nan=x.dtype.kind == "f"), f.name


@pytest.mark.parametrize("b,e", [(0, 5), (0, 1), (1, 4), (4, 5), (2, 2)])
def test_select_of_a_range_is_the_shard(pack, b, e):
    _equal(pack.select(range(b, e)), pack.shard(b, e))


def test_select_keeps_each_keyframes_rows(pack):
    kf = [0, 2, 3]
    s = pack.select(kf)
    for i, f in enumerate(kf):
        one = pack.shard(f, f + 1)
        so, ko = s.scan_offset, s.kp_offset
        assert np.array_equal(s.scan_xyz[so[i]:so[i + 1]], one.scan_xyz)
        assert np.array_equal(s.kp_xy[ko[i]:ko[i + 1]], one.kp_xy)
        assert np.array_equal(s.covis_uv[ko[i]:ko[i + 1]], one.covis_uv, equal_nan=True)
        for name in ("intrinsics", "image_wh", "Tcw", "covis_relpose", "covis_valid", "he_Tc", "he_Tl", "he_valid"):
            assert np.array_equal(getattr(s, name)[i], getattr(one, name)[0]), name
    # keyframe 0's hand-eye pair (0, 1) stays although keyframe 1 is not selected
    assert s.he_valid[0] == pack.he_valid[0]


def test_select_empty_and_numpy_input(pack):
    e = pack.select([])
    assert e.n_kf == 0 and e.scan_offset.tolist() == [0] and e.kp_offset.tolist() == [0]
    _equal(pack.select(np.array([1, 4], np.int32)), pack.select([1, 4]))


@pytest.mark.parametrize("kf,exc", [([2, 1], ValueError), ([1, 1], ValueError), ([-1, 2], ValueError), ([0, 5], ValueError),
                                    ([0.0, 1.0], TypeError), ([[0, 1]], TypeError)])
def test_select_validation(pack, kf, exc):
    with pytest.raises(exc):
        pack.select(kf)


def test_local_selection():
    par = importlib.import_module(PKG + ".parallel")
    g = [0, 3, 4, 9, 10, 17]
    bounds = [par.shard_bounds(18, 3, r) for r in range(3)]  # (0, 6), (6, 12), (12, 18)
    loc = [par.local_selection(g, b, e) for b, e in bounds]
    assert [x.tolist() for x in loc] == [[0, 3, 4], [3, 4], [5]]
    assert all(x.dtype == np.int32 for x in loc)
    assert sorted(int(v) + b for x, (b, _) in zip(loc, bounds) for v in x) == g
    assert par.local_selection([], 0, 6).tolist() == []
    assert par.local_selection([7, 8], 0, 6).tolist() == []        # the rank selects nothing and still makes the call
    for bad in ([3, 1], [2, 2], [-1, 0]):
        with pytest.raises(ValueError):
            par.local_selection(bad, 0, 6)
