"""Pins the oracle: the in-repo KD-tree restatement must reproduce the REFERENCE's own vendored
nanoflann v1.5.0 result for result — indices, squared distances, and the visit-order tie behaviour
(SURVEY.md F8).

Every test compares the port with the stored results of tests/golden/pin/pin_small.npz and pin_ties.npz
(made by tests/golden/pin/make_pin_golden.py, whose seeded inputs the tests rebuild; `backend` names what
produced them) and, where oracle/_ref is built from the reference's sources, with the real nanoflann as well."""
import os
import sys

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "pin")
sys.path.insert(0, GOLDEN)
import make_pin_golden as M  # noqa: E402


@pytest.fixture(scope="module")
def stored():
    g = np.load(os.path.join(GOLDEN, "pin_small.npz"))
    pack, X = M.pin_inputs()
    assert M.pack_digest(pack) == int(g["input_digest"]) and np.array_equal(X, g["X"]), "the seeded inputs changed"
    return g, pack


@pytest.fixture(scope="module")
def both(oracle_mod, stored):
    """(port, ref or None, pack): ref = the reference's nanoflann when oracle/_ref is built."""
    _, pack = stored
    ref = oracle_mod.Oracle(pack, kind="ref") if oracle_mod.have_ref() else None
    return oracle_mod.Oracle(pack, kind="port"), ref, pack


def test_backends_are_what_they_claim(both, stored):
    port, ref, _ = both
    assert port.kind == "port"
    assert str(stored[0]["backend"]) == "port" or str(stored[0]["backend"]).startswith("nanoflann-1.5.0")
    if ref is not None:
        assert ref.kind.startswith("nanoflann-1.5.0")


@pytest.mark.parametrize("k", M.KNN_K)
def test_knn_strict_identical_to_real_nanoflann(oracle_mod, both, stored, k):
    """strict = the reference's exact call; results must agree including visit-order ties."""
    g, _ = stored
    port, ref, pack = both
    q = M.knn_queries(pack.scan_xyz[: int(pack.scan_offset[1])].astype(np.float64), k)
    ia, da, ca, _ = port.knn3d(0, q, k, strict=True)
    assert oracle_mod.digest(q, ia, da, ca) == int(g[f"knn{k}"])
    if ref is not None:
        ib, db, cb, _ = ref.knn3d(0, q, k, strict=True)
        assert np.array_equal(ia, ib) and np.array_equal(da, db) and np.array_equal(ca, cb)


def test_knn_with_exact_ties_matches_real_nanoflann(oracle_mod):
    """Duplicated points => exact distance ties: the port must break them the same way (visit order)."""
    g = np.load(os.path.join(GOLDEN, "pin_ties.npz"))
    pack = M.tie_pack()
    assert M.pack_digest(pack) == int(g["input_digest"]), "the seeded inputs changed"
    port = oracle_mod.Oracle(pack, kind="port")
    ref = oracle_mod.Oracle(pack, kind="ref") if oracle_mod.have_ref() else None
    q = pack.scan_xyz[::7].astype(np.float64)
    for k in M.TIE_K:
        ia, da, _, _ = port.knn3d(0, q, k, strict=True)
        assert oracle_mod.digest(ia, da) == int(g[f"tie{k}"]), k
        if ref is not None:
            ib, db, _, _ = ref.knn3d(0, q, k, strict=True)
            assert np.array_equal(ia, ib) and np.array_equal(da, db), k
    # and the tie detector fires on such data
    _, _, _, ties = port.knn3d(0, q, 4)
    assert ties > 0


def test_ba_error_identical_with_real_nanoflann(both, stored):
    g, _ = stored
    port, ref, _ = both
    X = g["X"]
    sa, ta, ca = port.ba_error_sums(X, mode=0)
    assert np.array_equal(sa, g["sums"]) and np.array_equal(ca, g["counters"])
    assert ta.sum() == 0, "the synthetic data must be free of exact KNN ties (SURVEY.md H1)"
    # the reference's exact calls (no k+1 tie probe) give the same numbers when there is no tie
    assert np.array_equal(g["sums_strict"], g["sums"])
    assert np.array_equal(port.ba_error_sums(X, mode=0, strict=True)[0], g["sums_strict"])
    if ref is not None:
        sb, tb, cb = ref.ba_error_sums(X, mode=0)
        assert np.array_equal(sa, sb) and np.array_equal(ca, cb) and tb.sum() == 0
        assert np.array_equal(ref.ba_error_sums(X, mode=0, strict=True)[0], sb)


def test_frame_detail_identical_with_real_nanoflann(oracle_mod, both, stored):
    g, _ = stored
    port, ref, pack = both
    for kf in range(pack.n_kf):
        a = port.frame_debug(g["X"][1], kf)
        b = ref.frame_debug(g["X"][1], kf) if ref is not None else None
        for key in M.FRAME_KEYS:
            assert oracle_mod.digest(a[key]) == int(g[f"kf{kf}_{key}"]), (kf, key)
            if b is not None:
                assert np.array_equal(a[key], b[key]), (kf, key)


def test_lm_association_identical_with_real_nanoflann(both, stored):
    g, _ = stored
    port, ref, _ = both
    X = g["X"]
    na, _ = port.associate(X[0])
    keys, lin = port.block_keys(), port.linearize(X[:2])
    assert na.sum() > 100
    assert np.array_equal(na, g["lm_nblocks"]) and np.array_equal(keys, g["lm_keys"]) and np.array_equal(lin, g["lm_lin"])
    if ref is not None:
        nb, _ = ref.associate(X[0])
        assert np.array_equal(na, nb)
        assert np.array_equal(keys, ref.block_keys())
        assert np.array_equal(lin, ref.linearize(X[:2]))
