"""GPU parity beyond the one KITTI-00 camera: fx != fy and an off-centre principal point, other image sizes and packs that mix
them, keypoint counts up to the K1 shared-memory limit, 0 and 10 covisible slots, and scan sizes at the layout boundaries.

Every case compares the CUDA path, through the C-ABI, with the CPU oracle on the same seeded pack, at the bar of
test_gpu_parity.py: counters and block counts exact, correspondence and alignment index lists bit-exact, eval sums to 1e-9,
LM cost to 1e-9, J^T r and J^T J to 1e-6 relative plus 1e-9 x the largest entry.  Per keyframe, the eval_frames row is compared
with the oracle's frame_sums, so that a failure names the keyframe and its camera."""
import importlib

import numpy as np
import pytest

from conftest import PKG, has_cuda
from test_assoc2d_reference import SIZES, border_keypoints, camera_for

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not has_cuda(), reason="no CUDA device")]

REL = 1e-9
COUNTERS = slice(3, 12)
NAMES = ("sum_3d2d", "valid_3d2d", "cnt_3d2d", "sum_he", "cnt_he", "kept", "n_corr", "n_queries",
         "sum_3d3d", "valid_3d3d", "cnt_3d3d", "valid_pl", "valid_pt")
STL_ERR_INVALID, STL_ERR_CAPACITY = 1, 5
SMALL_SCAN = dict(beams=32, az_steps=1200)      # ~38k points: the oracle keeps up with many keyframes and candidates


@pytest.fixture(scope="module")
def capi():
    return importlib.import_module(PKG + ".capi")


# ---------------------------------------------------------------------------------------------------------------- pack builders
def _gen(synth, W=1241, H=376, n_kf=2, kf_begin=0, n_kf_total=None, cam=None, seed=1000, **kw):
    fx, fy, cx, cy = cam if cam is not None else camera_for(W, H)
    kw = {**SMALL_SCAN, **kw}
    pack, x_gt, _ = synth.generate(n_kf=n_kf, kf_begin=kf_begin, n_kf_total=n_kf_total or kf_begin + n_kf, width=W, height=H,
                                   fx=fx, fy=fy, cx=cx, cy=cy, seed=seed, **kw)
    return pack, x_gt


def _concat(pkg, packs):
    """Keyframe by keyframe, offsets rebased.  Covisible and hand-eye data are baked per keyframe (as in KeyFramePack.select)."""
    assert len({p.n_covis for p in packs}) == 1

    def offsets(name):
        out, base = [np.zeros(1, np.int64)], 0
        for p in packs:
            o = getattr(p, name)
            out.append(o[1:] + base)
            base += int(o[-1])
        return np.concatenate(out)
    cat = lambda name: np.concatenate([getattr(p, name) for p in packs])
    return pkg.KeyFramePack(
        n_kf=sum(p.n_kf for p in packs), n_covis=packs[0].n_covis, scan_offset=offsets("scan_offset"), scan_xyz=cat("scan_xyz"),
        intrinsics=cat("intrinsics"), image_wh=cat("image_wh"), kp_offset=offsets("kp_offset"), kp_xy=cat("kp_xy"),
        kp_mappoint=cat("kp_mappoint"), Tcw=cat("Tcw"), covis_relpose=cat("covis_relpose"), covis_valid=cat("covis_valid"),
        covis_uv=cat("covis_uv"), he_Tc=cat("he_Tc"), he_Tl=cat("he_Tl"), he_valid=cat("he_valid"))


def _with_scans(pack, scans):
    """The pack with scan f replaced by scans[f] ([n,3] float32)."""
    so = np.concatenate([[0], np.cumsum([len(s) for s in scans])]).astype(np.int64)
    out = pack.select(np.arange(pack.n_kf))
    out.scan_offset, out.scan_xyz = so, np.ascontiguousarray(np.concatenate(scans).astype(np.float32).reshape(-1, 3))
    return out


def _scan(pack, f):
    return pack.scan_xyz[int(pack.scan_offset[f]): int(pack.scan_offset[f + 1])]


def _take_kp(pkg, pack, n):
    """Every keyframe of `pack` keeps its first n keypoints."""
    parts = []
    for f in range(pack.n_kf):
        p = pack.select([f])
        p.kp_offset = np.array([0, n], np.int64)
        p.kp_xy, p.kp_mappoint, p.covis_uv = p.kp_xy[:n].copy(), p.kp_mappoint[:n].copy(), p.covis_uv[:n].copy()
        parts.append(p)
    return _concat(pkg, parts)


def _params(pkg, **kw):
    p = pkg.default_params()
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def _ctx(capi, monkeypatch, pack, params, split=False):
    """A context holding `pack`, with the one-kernel K1 or the three-kernel K1 (STL_K1_SPLIT is read at upload)."""
    if split:
        monkeypatch.setenv("STL_K1_SPLIT", "1")
    else:
        monkeypatch.delenv("STL_K1_SPLIT", raising=False)
    c = capi.Context(params=params)
    c.upload(pack)
    monkeypatch.delenv("STL_K1_SPLIT", raising=False)
    return c


def _cam(pack, f):
    W, H = pack.image_wh[f]
    return "keyframe %d (%d x %d, fx %.4f fy %.4f cx %.4f cy %.4f)" % ((f, W, H) + tuple(float(v) for v in pack.intrinsics[f]))


# ------------------------------------------------------------------------------------------------------------------- checks
def check_eval(c, orc, X):
    want, ties, _ = orc.ba_error_sums(X, mode=0)
    assert ties.sum() == 0
    got = c.eval_sums(X)
    assert np.array_equal(got[:, COUNTERS], want[:, COUNTERS]), (got[:, COUNTERS], want[:, COUNTERS])
    assert np.allclose(got[:, :3], want[:, :3], rtol=REL, atol=0), (got[:, :3], want[:, :3])
    return got


def check_frames(c, orc, X, pack, bs=None):
    """eval_frames rows against the oracle's per-keyframe record; returns the rows."""
    F = c.eval_frames(X)
    for b in (range(len(X)) if bs is None else bs):
        for f in range(pack.n_kf):
            fo = orc.frame_sums(X[b], f)
            for i, key in enumerate(NAMES):
                if key.startswith("sum_"):
                    assert np.isclose(F[b, f, i], fo[key], rtol=REL, atol=0), (b, _cam(pack, f), key, F[b, f, i], fo[key])
                else:
                    assert F[b, f, i] == fo[key], (b, _cam(pack, f), key, F[b, f, i], fo[key])
    return F


def check_debug(c, orc, X, pack, bs, plane_index, kfs=None):
    """Correspondence and alignment lists of candidates `bs` (c.eval_sums(X) must be the last evaluation)."""
    n = 0
    for b in bs:
        for f in (range(pack.n_kf) if kfs is None else kfs):
            d = orc.frame_debug(X[b], f)
            kp, pt = c.debug_corrset(b, f)
            assert np.array_equal(kp, d["corr_kp"]) and np.array_equal(pt, d["corr_pt"]), (b, _cam(pack, f), len(kp), len(d["corr_kp"]))
            a = c.debug_align(b, f)
            assert np.array_equal(a["kp"], d["align_kp"]) and np.array_equal(a["nn"], d["align_nn"]), (b, _cam(pack, f))
            assert np.array_equal(a["m"], d["align_m"]) and np.array_equal(a["is_plane"], d["align_is_plane"]), (b, _cam(pack, f))
            assert np.allclose(a["dist"], d["align_dist"], rtol=1e-10, atol=1e-12), (b, _cam(pack, f))
            if not plane_index:
                for i in range(len(a["m"])):
                    assert np.array_equal(a["knn"][i][: a["m"][i]], d["align_knn"][i][: d["align_m"][i]]), (b, _cam(pack, f), i)
            n += len(kp)
    return n


def check_lin(L, L_o):
    """Block counts exact, cost to 1e-9, J^T r and J^T J to 1e-6 relative plus 1e-9 x the largest entry."""
    assert np.array_equal(L[:, 57:], L_o[:, 57:]), (L[:, 57:], L_o[:, 57:])
    assert np.allclose(L[:, 0], L_o[:, 0], rtol=REL, atol=0), (L[:, 0], L_o[:, 0])
    sg, sh = np.abs(L_o[:, 1:8]).max(), np.abs(L_o[:, 8:57]).max()
    assert np.allclose(L[:, 1:8], L_o[:, 1:8], rtol=1e-6, atol=1e-9 * sg)
    assert np.allclose(L[:, 8:57], L_o[:, 8:57], rtol=1e-6, atol=1e-9 * sh)


def check_lm(c, orc, X, blocks=True, sample=300):
    """associate / linearize / step against the oracle; eval_blocks against block_eval for every 2-D block and a sample of the
    others.  Returns the block counts."""
    nb_o, _ = orc.associate(X[0])
    nb = c.associate(X[0])
    assert np.array_equal(nb, nb_o), (nb, nb_o)
    L_o = orc.linearize(X)
    check_lin(c.linearize(X), L_o)
    S = c.step(X, reassociate=True)
    assert np.array_equal(c.block_counts(), nb_o)
    check_lin(S[:, 12:], L_o)
    if blocks and len(X) > 1:
        keys = orc.block_keys()
        B = c.eval_blocks(X[1])
        assert len(B["type"]) == len(keys) == nb_o.sum()
        gpu = {(int(t), int(f), int(k)): i for i, (t, f, k) in enumerate(zip(B["type"], B["kf"], B["kp"]))}
        assert set(gpu) == {tuple(int(v) for v in k) for k in keys}
        rng = np.random.default_rng(0)
        check = set(rng.choice(len(keys), min(sample, len(keys)), replace=False).tolist()) if len(keys) else set()
        check |= {i for i, k in enumerate(keys) if k[0] == 0}
        for i in sorted(check):
            key = tuple(int(v) for v in keys[i])
            j = gpu[key]
            nr = int(B["n_res"][j])
            eo, Jo = orc.block_eval(i, X[1])
            bt = 1e-5 if key[0] == 3 else 1e-9
            assert len(eo) == nr, key
            assert np.allclose(B["residuals"][j][:nr], eo, rtol=bt, atol=1e-12), key
            assert np.allclose(B["jacobians"][j][:nr], Jo, rtol=bt, atol=bt * max(np.abs(Jo).max(), 1e-300)), key
    return nb_o


# ----------------------------------------------------------------------------------------------------------- §1 camera model
@pytest.fixture(scope="module")
def camera_packs(pkg, synth):
    """fy = fx (the association's camera), fy = 0.97 fx and 1.03 fx (the same data), and an off-centre principal point."""
    base, x_gt = _gen(synth, n_kf=3, seed=11)
    out = {"base": base}
    for name, s in (("fy097", 0.97), ("fy103", 1.03)):
        p = base.select(np.arange(base.n_kf))
        p.intrinsics = p.intrinsics.copy()
        p.intrinsics[:, 1] = np.float32(p.intrinsics[:, 0] * np.float32(s))
        out[name] = p
    out["offcentre"], _ = _gen(synth, n_kf=3, seed=11, cam=(718.856, 718.856, 607.1928 + 43.5, 185.2157 - 27.25))
    X = synth.candidates(x_gt, 4, 0.3, seed=12)
    return out, X


@pytest.fixture(scope="module")
def camera_oracles(oracle_mod, camera_packs):
    packs, _ = camera_packs
    return {k: oracle_mod.Oracle(p, kind="best") for k, p in packs.items()}


@pytest.mark.parametrize("split", [0, 1], ids=["k1", "k1-split"])
@pytest.mark.parametrize("plane_index", [1, 0])
@pytest.mark.parametrize("kind", ["fy097", "fy103", "offcentre"])
def test_camera_model(capi, pkg, monkeypatch, camera_packs, camera_oracles, kind, plane_index, split):
    packs, X = camera_packs
    pack, orc = packs[kind], camera_oracles[kind]
    p = _params(pkg, plane_index=plane_index)
    with _ctx(capi, monkeypatch, pack, p, split) as c:
        got = check_eval(c, orc, X)
        assert check_debug(c, orc, X, pack, (0, 2), plane_index) > 300
        rows = check_frames(c, orc, X, pack)
        if kind != "offcentre":
            # the data can tell fx from fy: the association reads fx only, the covisible term reads fy
            with _ctx(capi, monkeypatch, packs["base"], p, split) as cb:
                base = cb.eval_sums(X)
                base_corr = [cb.debug_corrset(b, f) for b in range(len(X)) for f in range(pack.n_kf)]
            c.eval_sums(X)
            corr = [c.debug_corrset(b, f) for b in range(len(X)) for f in range(pack.n_kf)]
            assert all(np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) for a, b in zip(corr, base_corr))
            assert np.array_equal(got[:, 11], base[:, 11])                     # same correspondence counts
            assert (got[:, 0] != base[:, 0]).all()                             # ... a different 3-D/2-D cost
            assert (got[:, 5] != base[:, 5]).any()                             # ... and different valid counts
        check_lm(c, orc, X)


@pytest.mark.parametrize("kind", ["fy097", "offcentre"])
def test_camera_model_gpr(capi, pkg, oracle_mod, monkeypatch, camera_packs, kind):
    """use_gpr = 1: the GPR blocks' training pixels use fy (k_linearize_gpr); 1e-6 bar of test_gpr_factor_blocks."""
    packs, X = camera_packs
    p = _params(pkg, use_gpr=1)
    orc = oracle_mod.Oracle(packs[kind], params=p, kind="best")
    with _ctx(capi, monkeypatch, packs[kind], p) as c:
        nb = c.associate(X[0])
        nb_o, _ = orc.associate(X[0])
        assert np.array_equal(nb, nb_o) and nb_o[3] > 20
        got, want = c.linearize(X[:3]), orc.linearize(X[:3])
    assert np.array_equal(got[:, 57:], want[:, 57:])
    sg = np.abs(want[:, 1:8]).max(axis=1, keepdims=True); sh = np.abs(want[:, 8:57]).max(axis=1, keepdims=True)
    assert np.allclose(got[:, 0], want[:, 0], rtol=1e-6, atol=0)
    assert np.allclose(got[:, 1:8], want[:, 1:8], rtol=1e-6, atol=1e-6 * sg)
    assert np.allclose(got[:, 8:57], want[:, 8:57], rtol=1e-6, atol=1e-6 * sh)


@pytest.mark.parametrize("plane_index", [1, 0])
@pytest.mark.parametrize("kind", ["fy097", "fy103", "offcentre"])
def test_camera_model_stable_variant(capi, pkg, oracle_mod, monkeypatch, camera_packs, kind, plane_index):
    """variant = 1: the query pixel of a keypoint is its map point re-projected with fx AND fy."""
    packs, X = camera_packs
    p = _params(pkg, variant=1, plane_index=plane_index, min_diff_dist=0.45)
    orc = oracle_mod.Oracle(packs[kind], params=p, kind="best")
    with _ctx(capi, monkeypatch, packs[kind], p) as c:
        got = check_eval(c, orc, X)
        assert (got[:, 11] > 50).any()                  # re-projected queries still find correspondences
        check_debug(c, orc, X, packs[kind], (0, 3), plane_index)
        check_frames(c, orc, X, packs[kind])


def test_calib_edges_with_fx_ne_fy(capi, oracle_mod):
    """calibEdge (calibmath.hpp, used by calib.cu) projects with fx for u and fy for v."""
    rng = np.random.default_rng(4)
    x_gt = np.array([1.21, -1.19, 1.2, 0.05, -0.08, -0.27, 9.0])
    n_kf, per_kf = 4, 150
    intr = np.array([[718.856, 718.856 * 0.97, 607.1928 + 30.0, 185.2157 - 20.0], [718.856, 718.856 * 1.03, 607.1928, 185.2157],
                     [650.0, 690.0, 320.0, 240.0], [720.0, 700.0, 188.0, 620.0]], np.float32)
    Tq, Xw, obs, off = [], [], [], [0]
    for f in range(n_kf):
        Tq.append(np.concatenate([rng.normal(0, 0.05, 3), [0.8 * f, 0.02 * f, 0.0]]))
        for _ in range(per_kf):
            Xw.append(np.array([rng.uniform(-6, 6), rng.uniform(-2, 2), rng.uniform(4, 30)]) / x_gt[6])
            obs.append(-oracle_mod.calib_edge(x_gt, Xw[-1], Tq[-1], intr[f], np.zeros(2)) + rng.normal(0, 0.3, 2))
        off.append(len(Xw))
    ed = capi.CalibBAEdges(off, np.asarray(Tq), intr, np.asarray(Xw), np.asarray(obs), np.full(len(Xw), 0.694, np.float32))
    X = x_gt + rng.normal(0, 0.02, (4, 7))
    X[3, :3] = 0.0
    with capi.Context() as c:
        got, chi_g = c.calib_linearize(ed, X, want_chi2=True)
    want, chi_o = oracle_mod.calib_linearize(ed, X)
    assert np.array_equal(got[:, 57:], want[:, 57:])
    assert np.allclose(chi_g, chi_o, rtol=1e-9, atol=1e-12) and np.allclose(got[:, 0], want[:, 0], rtol=1e-10)
    sg = np.abs(want[:, 1:8]).max(axis=1, keepdims=True); sh = np.abs(want[:, 8:57]).max(axis=1, keepdims=True)
    assert np.allclose(got[:, 1:8], want[:, 1:8], rtol=1e-8, atol=1e-10 * sg)
    assert np.allclose(got[:, 8:57], want[:, 8:57], rtol=1e-8, atol=1e-10 * sh)
    # the observations were made with fy: with fy replaced by fx the same edges cost more
    ed.intrinsics = ed.intrinsics.copy(); ed.intrinsics[:, 1] = ed.intrinsics[:, 0]
    assert oracle_mod.calib_linearize(ed, x_gt)[0][0, 0] > 10 * oracle_mod.calib_linearize(
        capi.CalibBAEdges(off, np.asarray(Tq), intr, np.asarray(Xw), np.asarray(obs), np.full(len(Xw), 0.694, np.float32)), x_gt)[0][0, 0]


# ------------------------------------------------------------------------------------------------------------ §2 image sizes
@pytest.fixture(scope="module")
def size_packs(pkg, synth):
    """Two keyframes per image size, generated as consecutive ranges of one 16-keyframe sequence (one world frame), and all of
    them in one pack.  The KITTI-sized part carries keypoints on cell edges and on / just outside the image border."""
    parts = []
    x_gt = None
    for i, (W, H) in enumerate(SIZES):
        p, x_gt = _gen(synth, W, H, n_kf=2, kf_begin=2 * i, n_kf_total=2 * len(SIZES), seed=21)
        parts.append(p)
    X = synth.candidates(x_gt, 64, 0.3, seed=22)
    for f in range(2):
        border_keypoints(parts[0], X[0], f, seed=f)
    return parts, _concat(pkg, parts), X


@pytest.fixture(scope="module")
def mixed_oracle(oracle_mod, size_packs):
    return oracle_mod.Oracle(size_packs[1], kind="best")


@pytest.mark.parametrize("split", [0, 1], ids=["k1", "k1-split"])
@pytest.mark.parametrize("i", range(len(SIZES)), ids=[f"{w}x{h}" for w, h in SIZES])
def test_single_size_pack(capi, pkg, oracle_mod, monkeypatch, size_packs, i, split):
    pack = size_packs[0][i]
    X = size_packs[2][:3]
    orc = oracle_mod.Oracle(pack, kind="best")
    with _ctx(capi, monkeypatch, pack, pkg.default_params(), split) as c:
        check_eval(c, orc, X)
        assert check_debug(c, orc, X, pack, (0, 2), 1) > 100
        check_frames(c, orc, X, pack)


@pytest.mark.parametrize("split", [0, 1], ids=["k1", "k1-split"])
@pytest.mark.parametrize("B", [1, 16, 64])
def test_mixed_camera_pack(capi, pkg, monkeypatch, size_packs, mixed_oracle, B, split):
    """All sizes in one pack: B = 16 and 64 take K1's 4- and 8-candidate chunks, so a table blob is reused and then replaced by
    one of another size.  Every keyframe's row and correspondences are bit-identical to its own single-camera pack."""
    parts, pack, Xall = size_packs
    X = Xall[:B]
    with _ctx(capi, monkeypatch, pack, pkg.default_params(), split) as c:
        check_eval(c, mixed_oracle, X)
        rows = check_frames(c, mixed_oracle, X, pack, bs=sorted({0, B - 1}))
        bs = sorted({0, B // 2, B - 1})
        c.eval_sums(X)
        corr = {(b, f): c.debug_corrset(b, f) for b in bs for f in range(pack.n_kf)}
        check_debug(c, mixed_oracle, X, pack, bs[:1], 1)
    for i, part in enumerate(parts):
        with _ctx(capi, monkeypatch, part, pkg.default_params(), split) as c:
            own = c.eval_frames(X)
            assert np.array_equal(own, rows[:, 2 * i: 2 * i + 2]), _cam(pack, 2 * i)
            c.eval_sums(X)
            for b in bs:
                for f in range(2):
                    kp, pt = c.debug_corrset(b, f)
                    assert np.array_equal(kp, corr[(b, 2 * i + f)][0]) and np.array_equal(pt, corr[(b, 2 * i + f)][1]), (b, _cam(pack, 2 * i + f))


@pytest.mark.parametrize("plane_index", [1, 0])
def test_mixed_camera_pack_lm(capi, pkg, monkeypatch, size_packs, mixed_oracle, plane_index):
    _, pack, Xall = size_packs
    with _ctx(capi, monkeypatch, pack, _params(pkg, plane_index=plane_index)) as c:
        nb = check_lm(c, mixed_oracle, Xall[:3])
    assert nb[0] > 0 and nb[1] + nb[2] > 0


def test_large_then_small_then_large_tables(capi, pkg, monkeypatch, size_packs):
    """The K1 shared-memory attribute is only ever raised: a small pack after a large one, and the large one again, give what a
    fresh context gives."""
    parts, _, Xall = size_packs
    large, small = parts[SIZES.index((1920, 1080))], parts[SIZES.index((640, 480))]
    X = Xall[:4]
    fresh = {}
    for name, p in (("large", large), ("small", small)):
        with _ctx(capi, monkeypatch, p, pkg.default_params()) as c:
            fresh[name] = (c.eval_frames(X), c.step(X, reassociate=True))
    with capi.Context() as c:
        for name, p in (("large", large), ("small", small), ("large", large)):
            c.upload(p)
            assert np.array_equal(c.eval_frames(X), fresh[name][0]), name
            assert np.array_equal(c.step(X, reassociate=True), fresh[name][1]), name


# ------------------------------------------------------------------------------------------------ §3 keypoints and the K1 limit
KP_COUNTS = [0, 1, 31, 32, 33, 511, 512, 513, 2000, 6000]


@pytest.mark.parametrize("split", [0, 1], ids=["k1", "k1-split"])
@pytest.mark.parametrize("plane_index", [1, 0])
def test_keypoint_counts(capi, pkg, synth, oracle_mod, monkeypatch, plane_index, split):
    parts, x_gt = [], None
    for i, n in enumerate(KP_COUNTS):
        p, x_gt = _gen(synth, n_kf=1, kf_begin=i, n_kf_total=len(KP_COUNTS), n_kp=n, seed=31)
        parts.append(p)
    pack = _concat(pkg, parts)
    assert np.array_equal(np.diff(pack.kp_offset), KP_COUNTS)
    X = synth.candidates(x_gt, 3, 0.3, seed=32)
    orc = oracle_mod.Oracle(pack, kind="best")
    with _ctx(capi, monkeypatch, pack, _params(pkg, plane_index=plane_index), split) as c:
        got = check_eval(c, orc, X)
        check_debug(c, orc, X, pack, (0, 2), plane_index)
        rows = check_frames(c, orc, X, pack)
        assert (rows[:, 0, 5] == 0).all()                 # no keypoint: the frame is skipped by the num_min_corr gate
        assert (rows[:, -2:, 5] == 1).all()
        check_lm(c, orc, X)
    assert (got[:, 10] < len(KP_COUNTS)).all()


def test_no_map_point_anywhere(capi, pkg, synth, oracle_mod):
    pack, x_gt = _gen(synth, n_kf=3, seed=41)
    pack.kp_mappoint = np.full_like(pack.kp_mappoint, np.nan)
    X = synth.candidates(x_gt, 3, 0.3, seed=42)
    orc = oracle_mod.Oracle(pack, kind="best")
    with capi.Context() as c:
        c.upload(pack)
        check_eval(c, orc, X)
        check_frames(c, orc, X, pack)
        nb_o, _ = orc.associate(X[0])
        nb = c.associate(X[0])
        assert nb.sum() == 0 and np.array_equal(nb, nb_o)
        L = c.linearize(X)
        assert not L.any() and not orc.linearize(X).any()
        S = c.step(X, reassociate=True)
        assert not S[:, 12:].any() and np.array_equal(S[:, :12], c.eval_sums(X))
        B = c.eval_blocks(X[1])
        assert len(B["type"]) == 0


def _uploads(capi, ctx, pack):
    try:
        ctx.upload(pack)
        return 0
    except Exception as e:                                 # StlError: the code says why
        return getattr(e, "code", -1)


# Largest keypoint count of a keyframe that upload accepts, for a 2-keyframe pack of ~38k-point scans (the 2 B per 128 scan
# points of K1's group list count too), measured on an NVIDIA B200 (227 KB opt-in shared memory per block).
K1_KP_LIMIT = {(1241, 376): 7694, (1920, 1080): 3782}


@pytest.mark.parametrize("W,H", list(K1_KP_LIMIT), ids=[f"{w}x{h}" for w, h in K1_KP_LIMIT])
def test_k1_keypoint_limit(capi, pkg, synth, oracle_mod, W, H):
    """Bisects the largest keypoint count upload accepts.  The rule is that a keyframe's K1 tables (keypoints, 2 px bitmap,
    8 px grid, map-point bits) and per-keypoint scratch fit the opt-in shared memory; count + 1 is refused with
    STL_ERR_CAPACITY and leaves the uploaded pack as it was."""
    import torch
    big, x_gt = _gen(synth, W, H, n_kf=2, n_kp=9000, seed=51)
    X = synth.candidates(x_gt, 2, 0.3, seed=52)
    with capi.Context() as c:
        lo, hi = 1, 9000
        assert _uploads(capi, c, _take_kp(pkg, big, lo)) == 0
        assert _uploads(capi, c, _take_kp(pkg, big, hi)) == STL_ERR_CAPACITY
        while hi - lo > 1:
            mid = (lo + hi) // 2
            code = _uploads(capi, c, _take_kp(pkg, big, mid))
            assert code in (0, STL_ERR_CAPACITY), (mid, code)
            lo, hi = (mid, hi) if code == 0 else (lo, mid)
        print("K1 keypoint limit at %d x %d: %d" % (W, H, lo))
        if torch.cuda.get_device_properties(0).shared_memory_per_block_optin == 232448:
            assert lo == K1_KP_LIMIT[(W, H)]
        pack = _take_kp(pkg, big, lo)
        orc = oracle_mod.Oracle(pack, kind="best")
        c.upload(pack)
        before = check_eval(c, orc, X)
        check_debug(c, orc, X, pack, (0,), 1)
        check_frames(c, orc, X, pack)
        check_lm(c, orc, X, sample=100)
        before = c.eval_sums(X)
        assert _uploads(capi, c, _take_kp(pkg, big, lo + 1)) == STL_ERR_CAPACITY
        assert np.array_equal(c.eval_sums(X), before)


def test_4k_keyframe_is_refused(capi, synth):
    """3840 x 2160: the 2 px bitmap alone (61 words x 1083 rows, 264 KB) exceeds the shared memory."""
    pack, _ = _gen(synth, 3840, 2160, n_kf=1, n_kp=2000, seed=53)
    with capi.Context() as c:
        assert _uploads(capi, c, pack) == STL_ERR_CAPACITY


# ----------------------------------------------------------------------------------------------------------- §4 covisible slots
@pytest.mark.parametrize("mask", ["all", "random"])
@pytest.mark.parametrize("split", [0, 1], ids=["k1", "k1-split"])
def test_ten_covisible_slots(capi, pkg, synth, oracle_mod, monkeypatch, split, mask):
    pack, x_gt = _gen(synth, n_kf=2, kf_begin=5, n_kf_total=16, n_covis=10, seed=61)
    assert pack.covis_valid.all()
    if mask == "random":
        pack.covis_valid = (np.random.default_rng(62).uniform(size=pack.covis_valid.shape) < 0.5).astype(np.uint8)
        assert 0 < pack.covis_valid.sum() < pack.covis_valid.size
    X = synth.candidates(x_gt, 3, 0.3, seed=63)
    orc = oracle_mod.Oracle(pack, kind="best")
    with _ctx(capi, monkeypatch, pack, pkg.default_params(), split) as c:
        check_eval(c, orc, X)
        check_debug(c, orc, X, pack, (0, 2), 1)
        check_frames(c, orc, X, pack)
        nb = check_lm(c, orc, X)
        assert nb[0] > 0
        B = c.eval_blocks(X[1])
        assert B["residuals"].shape[1] == 20 and B["n_res"].max() == (20 if mask == "all" else B["n_res"].max())
        assert B["n_res"].max() <= 20
        with pytest.raises(pkg._abi.StlError) as ei:
            c.eval_blocks(X[1], rmax=19)
        assert ei.value.code == STL_ERR_INVALID


@pytest.mark.parametrize("plane_index", [1, 0])
def test_no_covisible_slot(capi, pkg, synth, oracle_mod, plane_index):
    """n_covis = 0: no 3-D/2-D term.  BAError keeps its 3-D/3-D term; BuildProblem skips a correspondence without a covisible
    observation before it reaches the 3-D/3-D term (the `continue` at iba_local.cpp:259), so the problem has no block at all."""
    pack, x_gt = _gen(synth, n_kf=3, n_covis=0, seed=71)
    X = synth.candidates(x_gt, 3, 0.3, seed=72)
    orc = oracle_mod.Oracle(pack, kind="best")
    with capi.Context(params=_params(pkg, plane_index=plane_index)) as c:
        c.upload(pack)
        got = check_eval(c, orc, X)
        assert (got[:, 0] == 0).all() and (got[:, 11] > 0).all() and (got[:, 1] > 0).all()
        check_debug(c, orc, X, pack, (0,), plane_index)
        check_frames(c, orc, X, pack)
        nb = check_lm(c, orc, X)
        assert nb.sum() == 0 and not c.linearize(X).any()


# ------------------------------------------------------------------------------------------------------------ §5 scan sizes
SCAN_SIZES = [1, 31, 32, 33, 127, 128, 129, 1023, 1024, 1025, 8191, 8192, 8193, 32767, 32768, 32769]


@pytest.fixture(scope="module")
def scan_size_pack(synth):
    pack, x_gt = _gen(synth, n_kf=len(SCAN_SIZES), seed=81, beams=64, az_steps=1875)
    rng = np.random.default_rng(82)
    scans = [_scan(pack, f)[np.sort(rng.choice(len(_scan(pack, f)), n, replace=False))] for f, n in enumerate(SCAN_SIZES)]
    return _with_scans(pack, scans), synth.candidates(x_gt, 2, 0.3, seed=83)


@pytest.mark.parametrize("plane_index", [1, 0])
def test_scan_sizes(capi, pkg, oracle_mod, scan_size_pack, plane_index):
    pack, X = scan_size_pack
    assert np.array_equal(np.diff(pack.scan_offset), SCAN_SIZES)
    p = _params(pkg, plane_index=plane_index, num_min_corr=1)
    orc = oracle_mod.Oracle(pack, params=p, kind="best")
    with capi.Context(params=p) as c:
        c.upload(pack)
        check_eval(c, orc, X)
        check_debug(c, orc, X, pack, (0, 1), plane_index)
        rows = check_frames(c, orc, X, pack)
        assert rows[:, 7:, 5].all() and rows[:, :7, 5].any()   # tiny scans pass the gate too and reach the 3-D stage
        check_lm(c, orc, X)
        rng = np.random.default_rng(84)
        for f in range(pack.n_kf):
            P = _scan(pack, f).astype(np.float64)
            q = np.concatenate([P[rng.choice(len(P), 50)] + rng.normal(0, 0.05, (50, 3)), P[rng.choice(len(P), 20)],
                                rng.uniform(-60, 60, (10, 3))])
            io, do, co, ties = orc.knn3d(f, q, 30, 0.0)
            assert ties == 0
            ig, dg, cg = c.knn3d(f, q, 30, 0.0)
            assert np.array_equal(cg, co) and (cg == min(30, len(P))).all(), f
            for i in range(len(q)):
                assert np.array_equal(ig[i, :cg[i]], io[i, :co[i]]) and np.array_equal(dg[i, :cg[i]], do[i, :co[i]]), (f, i)


def test_largest_scan(capi, pkg, synth, oracle_mod):
    """2^20 points (a scan replicated with 1 mm jitter) upload and match the oracle; 2^20 + 1 are refused."""
    pack, x_gt = _gen(synth, n_kf=1, seed=91, beams=64, az_steps=1875)
    P = _scan(pack, 0)
    rng = np.random.default_rng(92)
    reps = -(-(1 << 20) // len(P))
    big = np.concatenate([P] + [P + rng.normal(0, 1e-3, P.shape).astype(np.float32) for _ in range(reps)])
    X = synth.candidates(x_gt, 1, 0.3, seed=93)
    full = _with_scans(pack, [big[: 1 << 20]])
    orc = oracle_mod.Oracle(full, kind="best")
    with capi.Context() as c:
        c.upload(full)
        check_eval(c, orc, X)
        check_debug(c, orc, X, full, (0,), 1)
        want = c.eval_sums(X)
        assert _uploads(capi, c, _with_scans(pack, [big[: (1 << 20) + 1]])) == STL_ERR_CAPACITY
        assert np.array_equal(c.eval_sums(X), want)


def test_far_outlier(capi, pkg, synth, oracle_mod, monkeypatch):
    """One point 2 km away raises pmax, which widens the thin slab that bypasses K1's float32 pre-cull."""
    pack, x_gt = _gen(synth, n_kf=2, seed=95)
    scans = [_scan(pack, 0), np.concatenate([_scan(pack, 1), [[2000.0, 35.0, -4.0]]]).astype(np.float32)]
    pack = _with_scans(pack, scans)
    X = synth.candidates(x_gt, 2, 0.3, seed=96)
    orc = oracle_mod.Oracle(pack, kind="best")
    for split in (0, 1):
        with _ctx(capi, monkeypatch, pack, pkg.default_params(), split) as c:
            check_eval(c, orc, X)
            if not split:
                assert c.work_counters()["k1_overflow_units"] > 0    # the exact path really ran
            check_debug(c, orc, X, pack, (0, 1), 1)
            check_frames(c, orc, X, pack)
            check_lm(c, orc, X)


@pytest.mark.parametrize("plane_index", [1, 0])
def test_coplanar_and_collinear_patches(capi, pkg, synth, oracle_mod, plane_index):
    """A patch flattened exactly to z = const and one squashed onto a line: repeated eigenvalues, the gates decide."""
    pack, x_gt = _gen(synth, n_kf=2, seed=97)
    scans = []
    for f in range(2):
        P = _scan(pack, f).copy()
        r = np.hypot(P[:, 0], P[:, 1])
        ang = np.arctan2(P[:, 1], P[:, 0])
        plane = (r > 8) & (r < 14) & (np.abs(ang) < 0.25)
        line = (r > 14) & (r < 30) & (np.abs(ang - 0.3) < 0.15)
        P[plane, 2] = np.float32(-1.5)
        P[line, 1] = np.float32(P[line, 0] * np.float32(np.tan(0.3)))
        P[line, 2] = np.float32(-1.0)
        assert plane.sum() > 500 and line.sum() > 100
        scans.append(P)
    pack = _with_scans(pack, scans)
    X = synth.candidates(x_gt, 3, 0.3, seed=98)
    orc = oracle_mod.Oracle(pack, kind="best")
    with capi.Context(params=_params(pkg, plane_index=plane_index)) as c:
        c.upload(pack)
        check_eval(c, orc, X)
        check_debug(c, orc, X, pack, (0, 1, 2), plane_index)
        check_frames(c, orc, X, pack)
        check_lm(c, orc, X)
