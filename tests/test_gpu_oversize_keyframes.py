"""Oversize keyframes (stl_allow_oversize_keyframes): keyframes whose K1 tables do not fit the one-kernel K1's shared memory
run on the banded three-kernel K1 and give what the one-kernel K1 would give with enough shared memory.

Shapes the one-kernel K1 cannot run are checked against the CPU oracle at the bar of test_gpu_camera_shapes.py (whose pack
builders and checks are reused); packs that fit are checked bit for bit against the one-kernel K1, with every keyframe routed
to the oversize path by STL_K1_OVERSIZE=all."""
import importlib

import numpy as np
import pytest

from conftest import PKG, has_cuda
from test_assoc2d_reference import project
from test_gpu_camera_shapes import (K1_KP_LIMIT, STL_ERR_CAPACITY, _concat, _gen, _params, _uploads, check_debug, check_eval,
                                    check_frames, check_lm)

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not has_cuda(), reason="no CUDA device")]

STL_ERR_STATE = 4
BIG_SCAN = dict(beams=64, az_steps=2000)  # ~128k points: larger than the SMALL_SCAN of the other keyframes


@pytest.fixture(scope="module")
def capi():
    return importlib.import_module(PKG + ".capi")


def _ctx(capi, monkeypatch, pack, params=None, allow=True, route_all=False):
    """A context holding `pack` with oversize keyframes allowed (or not); route_all sets STL_K1_OVERSIZE=all for the upload."""
    monkeypatch.delenv("STL_K1_SPLIT", raising=False)
    if route_all:
        monkeypatch.setenv("STL_K1_OVERSIZE", "all")
    else:
        monkeypatch.delenv("STL_K1_OVERSIZE", raising=False)
    c = capi.Context(params=params)
    c.allow_oversize_keyframes(allow)
    c.upload(pack)
    monkeypatch.delenv("STL_K1_OVERSIZE", raising=False)
    return c


def band_rows(W, H):
    """The band rule of DESIGN.md §3 "Oversize keyframes": bitmap rows of a band, rows of the bitmap."""
    wpr = ((W + 1) // 2 + 2 + 1 + 31) // 32
    return max(1, 4096 // wpr), (H + 1) // 2 + 3


def _corrsets(c, B, F):
    return [c.debug_corrset(b, f) for b in range(B) for f in range(F)]


def _same_corrsets(a, b):
    return len(a) == len(b) and all(np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1]) for x, y in zip(a, b))


# ------------------------------------------------------------------------------------------------------------------ 1. 4K
@pytest.fixture(scope="module")
def pack_4k(pkg, synth):
    """A 3840 x 2160 keyframe and a portrait 2160 x 3840 one, 2000 keypoints each."""
    a, x_gt = _gen(synth, 3840, 2160, n_kf=1, kf_begin=0, n_kf_total=2, n_kp=2000, seed=53)
    b, _ = _gen(synth, 2160, 3840, n_kf=1, kf_begin=1, n_kf_total=2, n_kp=2000, seed=53)
    return _concat(pkg, [a, b]), synth.candidates(x_gt, 3, 0.3, seed=54)


@pytest.mark.parametrize("plane_index", [1, 0])
def test_4k_keyframes(capi, pkg, oracle_mod, monkeypatch, pack_4k, plane_index):
    pack, X = pack_4k
    orc = oracle_mod.Oracle(pack, kind="best")
    with _ctx(capi, monkeypatch, pack, _params(pkg, plane_index=plane_index)) as c:
        assert c.oversize_keyframes().tolist() == [0, 1]
        got = check_eval(c, orc, X)
        assert c.work_counters()["k1_overflow_units"] == 0
        assert got[:, 11].sum() > 1000
        assert check_debug(c, orc, X, pack, (0, 2), plane_index) > 50
        check_frames(c, orc, X, pack)
        check_lm(c, orc, X, sample=150)


@pytest.mark.parametrize("plane_index", [1, 0])
def test_4k_keyframes_stable_variant(capi, pkg, oracle_mod, monkeypatch, pack_4k, plane_index):
    pack, X = pack_4k
    p = _params(pkg, variant=1, plane_index=plane_index, min_diff_dist=0.45)
    orc = oracle_mod.Oracle(pack, params=p, kind="best")
    with _ctx(capi, monkeypatch, pack, p) as c:
        assert c.oversize_keyframes().tolist() == [0, 1]
        check_eval(c, orc, X)
        check_debug(c, orc, X, pack, (0, 2), plane_index)
        check_frames(c, orc, X, pack)


# ------------------------------------------------------------------------------------------- 2. keypoints past the K1 limit
KP_PAST = [(1241, 376, K1_KP_LIMIT[(1241, 376)] + 1), (1241, 376, 12000), (1241, 376, 20000),
           (1920, 1080, K1_KP_LIMIT[(1920, 1080)] + 1), (1920, 1080, 8000)]


@pytest.mark.parametrize("plane_index", [1, 0])
@pytest.mark.parametrize("W,H,n", KP_PAST, ids=[f"{w}x{h}-{n}" for w, h, n in KP_PAST])
def test_keypoints_past_the_limit(capi, pkg, synth, oracle_mod, monkeypatch, W, H, n, plane_index):
    pack, x_gt = _gen(synth, W, H, n_kf=2, n_kp=n, seed=51)
    X = synth.candidates(x_gt, 2, 0.3, seed=52)
    with capi.Context() as c:
        assert _uploads(capi, c, pack) == STL_ERR_CAPACITY          # refused without the flag
    orc = oracle_mod.Oracle(pack, kind="best")
    with _ctx(capi, monkeypatch, pack, _params(pkg, plane_index=plane_index)) as c:
        assert c.oversize_keyframes().tolist() == [0, 1]
        check_eval(c, orc, X)
        assert c.work_counters()["k1_overflow_units"] == 0           # survivor capacity sized by the keypoints
        check_debug(c, orc, X, pack, (0,), plane_index)
        check_frames(c, orc, X, pack)
        check_lm(c, orc, X, sample=100)


# ------------------------------------------------------------------------------------------------------ 3. band boundaries
def _band_keypoints(pack, x, kf, seed=0):
    """Keypoints of keyframe kf (in place) at projected points moved onto every band boundary of the documented rule and to
    0.01, 0.75 and 1.5 px on either side of it, plus the image corners.  Returns (keypoints written, boundaries with points
    near them)."""
    rng = np.random.default_rng(seed)
    W, H = (int(v) for v in pack.image_wh[kf])
    R, rows = band_rows(W, H)
    u, v, _ = project(pack, x, kf)
    ok = (u >= 0) & (u < W) & (v >= 0) & (v < H)
    u, v = u[ok], v[ok]
    xy, hit = [], 0
    for r in range(R, rows, R):                                  # band boundary: bitmap row r, first pixel row 2 (r - 1)
        vb = 2.0 * (r - 1)
        near = np.flatnonzero(np.abs(v - vb) < 4.0)
        if len(near) == 0:
            continue
        hit += 1
        for i in rng.choice(near, min(5, len(near)), replace=False):
            for d in (-1.5, -0.75, -0.01, 0.0, 0.01, 0.75, 1.5):
                xy.append((u[i], vb + d))
    xy += [(0.0, 0.0), (W - 1e-3, 0.0), (0.0, H - 1e-3), (W - 1e-3, H - 1e-3)]
    xy = np.asarray(xy, np.float32)
    k0, k1 = int(pack.kp_offset[kf]), int(pack.kp_offset[kf + 1])
    n = min(len(xy), k1 - k0)
    pack.kp_xy[k0:k0 + n] = xy[:n]
    return n, hit


@pytest.mark.parametrize("plane_index", [1, 0])
def test_band_boundaries(capi, pkg, synth, oracle_mod, monkeypatch, plane_index):
    pack, x_gt = _gen(synth, 3840, 2160, n_kf=2, n_kp=2500, seed=57)
    X = synth.candidates(x_gt, 3, 0.2, seed=58)
    placed = [_band_keypoints(pack, X[0], f, seed=f) for f in range(2)]
    print("band boundaries with keypoints (of %d): %s" % (band_rows(3840, 2160)[1] // band_rows(3840, 2160)[0], placed))
    assert all(hit >= 2 for _, hit in placed), placed
    orc = oracle_mod.Oracle(pack, kind="best")
    with _ctx(capi, monkeypatch, pack, _params(pkg, plane_index=plane_index)) as c:
        check_eval(c, orc, X)
        assert check_debug(c, orc, X, pack, (0, 1, 2), plane_index) > 50
        check_frames(c, orc, X, pack)


# ------------------------------------------------------------------------------------------------------------- 4. mixed pack
@pytest.fixture(scope="module")
def mixed(pkg, synth):
    """Fitting and oversize keyframes interleaved: 1241 x 376 (fits), 3840 x 2160 (oversize), 1241 x 376 with the pack's
    largest scan (fits), 1920 x 1080 with 8000 keypoints (oversize)."""
    shapes = [(1241, 376, 2000, {}), (3840, 2160, 2000, {}), (1241, 376, 2000, BIG_SCAN), (1920, 1080, 8000, {})]
    parts, x_gt = [], None
    for i, (W, H, n, kw) in enumerate(shapes):
        p, x_gt = _gen(synth, W, H, n_kf=1, kf_begin=i, n_kf_total=len(shapes), n_kp=n, seed=61, **kw)
        parts.append(p)
    pack = _concat(pkg, parts)
    assert np.argmax(np.diff(pack.scan_offset)) == 2
    return pack, synth.candidates(x_gt, 3, 0.3, seed=62)


@pytest.mark.parametrize("plane_index", [1, 0])
def test_mixed_pack(capi, pkg, oracle_mod, monkeypatch, mixed, plane_index):
    pack, X = mixed
    p = _params(pkg, plane_index=plane_index)
    orc = oracle_mod.Oracle(pack, kind="best")
    with _ctx(capi, monkeypatch, pack, p) as c:
        assert c.oversize_keyframes().tolist() == [1, 3]
        check_eval(c, orc, X)
        rows = check_frames(c, orc, X, pack)
        c.eval_sums(X)
        corr = _corrsets(c, len(X), pack.n_kf)
        check_lm(c, orc, X, sample=100)
    for f in range(pack.n_kf):
        with _ctx(capi, monkeypatch, pack.select([f]), p) as c1:
            assert c1.oversize_keyframes().tolist() == ([0] if f in (1, 3) else [])
            assert np.array_equal(c1.eval_frames(X)[:, 0], rows[:, f]), f
            c1.eval_sums(X)
            assert _same_corrsets(_corrsets(c1, len(X), 1), corr[f::pack.n_kf]), f


# ------------------------------------------------------------------------------------------------------------ 5. route-all
@pytest.fixture(scope="module")
def kitti_pack(synth):
    pack, x_gt = _gen(synth, n_kf=3, seed=11)
    return pack, synth.candidates(x_gt, 4, 0.3, seed=12)


def _record(c, X, F):
    """Everything the K1 routing can change, from one context."""
    out = {"sums": c.eval_sums(X)}
    out["corr"] = _corrsets(c, len(X), F)
    out["frames"] = c.eval_frames(X)
    out["step"] = c.step(X, reassociate=True)
    out["blocks"] = c.associate(X[0])
    out["lin"] = c.linearize(X)
    out["multi"] = c.step_multi(X)
    c.select_keyframes([0, 2])
    out["sel_sums"] = c.eval_sums(X)
    out["sel_frames"] = c.eval_frames(X)
    out["sel_step"] = c.step(X[:1], reassociate=True)
    c.select_keyframes(None)
    return out


def _same_record(a, b):
    for k in a:
        if k == "corr":
            assert _same_corrsets(a[k], b[k]), k
        else:
            assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("plane_index", [1, 0])
def test_route_all_is_bit_identical(capi, pkg, monkeypatch, kitti_pack, plane_index):
    pack, X = kitti_pack
    p = _params(pkg, plane_index=plane_index)
    with _ctx(capi, monkeypatch, pack, p, allow=False) as c:
        assert c.oversize_keyframes().tolist() == []
        want = _record(c, X, pack.n_kf)
    with _ctx(capi, monkeypatch, pack, p, route_all=True) as c:
        assert c.oversize_keyframes().tolist() == list(range(pack.n_kf))
        got = _record(c, X, pack.n_kf)
        assert c.work_counters()["k1_overflow_units"] == 0
    _same_record(want, got)


def test_route_all_stable_variant(capi, pkg, monkeypatch, kitti_pack):
    pack, X = kitti_pack
    p = _params(pkg, variant=1, min_diff_dist=0.45)
    out = []
    for route_all in (False, True):
        with _ctx(capi, monkeypatch, pack, p, route_all=route_all) as c:
            out.append((c.eval_sums(X), _corrsets(c, len(X), pack.n_kf), c.eval_frames(X)))
    assert np.array_equal(out[0][0], out[1][0]) and _same_corrsets(out[0][1], out[1][1]) and np.array_equal(out[0][2], out[1][2])


# ------------------------------------------------------------------------------------------------------------- 6. selection
@pytest.mark.parametrize("sel", [[1, 3], [0, 2], [0, 1, 3], []], ids=["oversize", "fitting", "both", "none"])
def test_selection_on_mixed_pack(capi, pkg, monkeypatch, mixed, sel):
    pack, X = mixed
    with _ctx(capi, monkeypatch, pack) as c:
        c.eval_sums(X)
        c.associate(X[0])
        c.select_keyframes(sel)
        with pytest.raises(Exception) as e:                         # a selection drops the frozen problem
            c.linearize(X)
        assert getattr(e.value, "code", None) == STL_ERR_STATE
        got, rows = c.eval_sums(X), c.eval_frames(X)
        unsel = [f for f in range(pack.n_kf) if f not in sel]
        assert not rows[:, unsel].any()
        if not sel:
            assert not got.any()
            return
        corr = _corrsets(c, len(X), pack.n_kf)
        S = c.step(X, reassociate=True)
        assert c.oversize_keyframes().tolist() == [1, 3]           # the selection does not change the routing
    sub = pack.select(sel)
    with _ctx(capi, monkeypatch, sub) as c1:
        assert np.array_equal(c1.eval_sums(X), got)
        assert np.array_equal(c1.eval_frames(X), rows[:, sel])
        assert _same_corrsets(_corrsets(c1, len(X), len(sel)), [corr[b * pack.n_kf + f] for b in range(len(X)) for f in sel])
        assert np.array_equal(c1.step(X, reassociate=True), S)


# -------------------------------------------------------------------------------------------------------- 7. flag semantics
def test_flag_on_a_fitting_pack_changes_nothing(capi, pkg, monkeypatch, kitti_pack):
    pack, X = kitti_pack
    out = []
    for allow in (False, True):
        with _ctx(capi, monkeypatch, pack, allow=allow) as c:
            assert c.oversize_keyframes().tolist() == []
            c.eval_sums(X)
            l0 = c.work_counters()["launches"]
            r = (c.eval_sums(X), c.eval_frames(X), c.step(X, reassociate=True))
            out.append((r, c.work_counters()["launches"] - l0))
    assert all(np.array_equal(a, b) for a, b in zip(out[0][0], out[1][0]))
    assert out[0][1] == out[1][1]


def test_flag_is_read_at_upload(capi, pkg, monkeypatch, pack_4k, kitti_pack):
    pack, X = pack_4k
    with _ctx(capi, monkeypatch, pack) as c:
        before = c.eval_sums(X)
        c.allow_oversize_keyframes(False)                           # the resident pack keeps working
        assert np.array_equal(c.eval_sums(X), before)
        assert c.oversize_keyframes().tolist() == [0, 1]
        assert _uploads(capi, c, pack) == STL_ERR_CAPACITY          # ... and a re-upload is refused, the pack kept
        assert np.array_equal(c.eval_sums(X), before)
        assert c.oversize_keyframes().tolist() == [0, 1]
        c.upload(kitti_pack[0])
        assert c.oversize_keyframes().tolist() == []
        with pytest.raises(TypeError):
            c.allow_oversize_keyframes(2)
