"""Keyframe selection on a resident pack (stl_select_keyframes) and the per-keyframe BAError (stl_eval_frames): a context
that selects S computes, bit for bit, what a fresh context holding pack.select(S) computes.  Every test makes its own
contexts, so that no other file sees a context with a selection."""
import importlib

import numpy as np
import pytest

from conftest import PKG, has_cuda

pytestmark = pytest.mark.gpu

ROT_TOL, TRANS_TOL = np.deg2rad(0.01), 1e-3
LB = np.array([-0.1, -0.1, -0.1, -0.3, -0.3, -0.3, -1.0])

# the 6-keyframe small_pack: all (as a list), every 2nd, the first, the last, a contiguous run, a non-contiguous set, none
SELECTIONS = {"all": [0, 1, 2, 3, 4, 5], "every2": [0, 2, 4], "first": [0], "last": [5], "run": [1, 2, 3], "sparse": [0, 3, 4],
              "none": []}


@pytest.fixture(scope="module")
def capi():
    if not has_cuda():
        pytest.skip("no CUDA device")
    return importlib.import_module(PKG + ".capi")


@pytest.fixture(scope="module")
def pack(small_pack):
    return small_pack[0]


@pytest.fixture(scope="module")
def X(synth, small_pack):
    return synth.candidates(small_pack[1], 4, spread=0.5)


@pytest.fixture(params=[1, 0], ids=["plane-index", "plane-fit"])
def params(request, pkg):
    p = pkg.default_params()
    p.plane_index = request.param
    return p


def _ctx(capi, params, pack, sel=None):
    c = capi.Context(params=params)
    c.upload(pack)
    if sel is not None:
        c.select_keyframes(sel)
    return c


def _run(c, X):
    """eval record, block counts, per-block output and linearisation at X[1], step record of X[:2] (re-associating at X[0])"""
    ev = c.eval_sums(X)
    nb = c.associate(X[1])
    lin = c.linearize(X[:3])
    blocks = c.eval_blocks(X[2])
    step = c.step(X[:2])
    return ev, nb, lin, blocks, step


@pytest.mark.parametrize("name", list(SELECTIONS))
def test_selection_equals_sliced_pack(capi, params, pack, X, name):
    S = SELECTIONS[name]
    with _ctx(capi, params, pack, S) as c:
        got = _run(c, X)
    if not S:  # no keyframe: nothing is counted and nothing is frozen
        ev, nb, lin, blocks, step = got
        assert not ev.any() and not nb.any() and not lin.any() and not step.any() and len(blocks["type"]) == 0
        return
    with _ctx(capi, params, pack.select(S)) as c:
        want = _run(c, X)
    for i, what in ((0, "eval"), (1, "block counts"), (2, "linearisation"), (4, "step")):
        assert np.array_equal(got[i], want[i]), what
    assert got[1].sum() > 0
    gb, wb = got[3], want[3]
    assert np.array_equal(gb["kf"], np.asarray(S)[wb["kf"]])  # the pack's own keyframe indices
    for k in ("type", "kp", "n_res", "residuals", "jacobians"):
        assert np.array_equal(gb[k], wb[k]), k


@pytest.mark.parametrize("name", ["every2", "sparse"])
def test_selection_multi_and_oracle(capi, params, pack, X, oracle_mod, name):
    S = SELECTIONS[name]
    starts = X[:3]
    with _ctx(capi, params, pack, S) as c:
        nb = c.associate_multi(starts)
        lin = c.linearize_multi(starts)
        step = c.step_multi(starts)
    sliced = pack.select(S)
    with _ctx(capi, params, sliced) as c:
        assert np.array_equal(nb, c.associate_multi(starts))
        assert np.array_equal(lin, c.linearize_multi(starts))
        assert np.array_equal(step, c.step_multi(starts))
    orc = oracle_mod.Oracle(sliced, kind="best")
    for p, x in enumerate(starts):
        nb_o, _ = orc.associate(x)
        want = orc.linearize(x[None])
        assert np.array_equal(nb[p], nb_o)
        assert np.array_equal(lin[p, 57:], want[0, 57:])
        assert np.allclose(lin[p, 0], want[0, 0], rtol=1e-9, atol=0)
        sg, sh = np.abs(want[0, 1:8]).max(), np.abs(want[0, 8:57]).max()
        assert np.allclose(lin[p, 1:8], want[0, 1:8], rtol=1e-6, atol=1e-9 * sg)
        assert np.allclose(lin[p, 8:57], want[0, 8:57], rtol=1e-6, atol=1e-9 * sh)


def test_selection_gpr(capi, pkg, pack, X):
    p = pkg.default_params(); p.use_gpr = 1
    S = SELECTIONS["sparse"]
    with _ctx(capi, p, pack, S) as c:
        got = (c.associate(X[0]), c.linearize(X[:2]), c.step(X[:2]))
    with _ctx(capi, p, pack.select(S)) as c:
        want = (c.associate(X[0]), c.linearize(X[:2]), c.step(X[:2]))
    assert got[0][3] > 0
    for g, w in zip(got, want):
        assert np.array_equal(g, w)


def test_null_selection_restores_the_pack(capi, params, pack, X):
    with _ctx(capi, params, pack) as c:
        want = _run(c, X)
    with _ctx(capi, params, pack, SELECTIONS["sparse"]) as c:
        _run(c, X)
        c.select_keyframes(None)
        got = _run(c, X)
    for g, w in zip(got, want):
        if isinstance(g, dict):
            assert all(np.array_equal(g[k], w[k]) for k in g)
        else:
            assert np.array_equal(g, w)


def test_state_rules(capi, pkg, pack, X):
    p = pkg.default_params()
    E = capi._abi.StlError

    def code(f):
        with pytest.raises(E) as e:
            f()
        return e.value.code

    with capi.Context(params=p) as c:
        assert code(lambda: c.select_keyframes([0])) == 4           # no pack yet
        c.upload(pack)
        c.eval_sums(X[:1])
        c.associate(X[0])
        c.linearize(X[0])
        c.select_keyframes([0, 2])
        for call in (lambda: c.linearize(X[0]), c.block_counts, lambda: c.eval_blocks(X[0]), lambda: c.step(X[:1], reassociate=False),
                     lambda: c.linearize_multi(X[:1])):
            assert code(call) == 4
        c.associate(X[0])                                          # a new association lifts the refusal
        lin = c.linearize(X[0])
        # invalid lists are refused and leave the selection (and the frozen problem) in place
        for bad in ([2, 0], [1, 1], [0, 6], [-1, 2]):
            assert code(lambda: c.select_keyframes(bad)) == 1
        for bad in ([0.7, 2.2], [[0, 2]]):                         # not truncated to integers: refused before the call
            with pytest.raises(TypeError):
                c.select_keyframes(bad)
        k = np.array([0, 2], np.int32)
        assert c.lib.stl_select_keyframes(c.h, k.ctypes.data_as(capi._abi._i32p), -1) == 1
        assert np.array_equal(c.linearize(X[0]), lin)
        ev = c.eval_sums(X)
        # the points K1 streamed are those of the selected scans
        pts = sum(int(pack.scan_offset[f + 1] - pack.scan_offset[f]) for f in (0, 2))
        assert c.work_counters()["points"] == pts * len(X)
        with _ctx(capi, p, pack.select([0, 2])) as s:
            assert np.array_equal(ev, s.eval_sums(X))
            s.eval_sums(X)
            want_frame = s.debug_frame(1, 1)
        # unselected keyframes read as empty through the debug getters
        assert not any(c.debug_frame(1, 1).values()) and not any(c.debug_frame(1, 3).values())
        assert len(c.debug_corrset(1, 1)[0]) == 0 and len(c.debug_align(1, 1)["nn"]) == 0
        assert c.debug_frame(1, 2) == want_frame
        # an upload selects every keyframe again
        c.upload(pack)
        with _ctx(capi, p, pack) as full:
            assert np.array_equal(c.eval_sums(X), full.eval_sums(X))
        assert c.work_counters()["points"] == int(pack.scan_offset[-1]) * len(X)


def test_split_k1_honours_the_selection(capi, params, pack, X, monkeypatch):
    """the three-kernel K1 walks the selection as the one-kernel K1 does, and (a diagnostic switch) changes no bit: its
    covisible term is summed in the one-kernel K1's order"""
    S = SELECTIONS["sparse"]
    with _ctx(capi, params, pack.select(S)) as c:
        want = (c.eval_sums(X), c.step(X[:2]))
    with _ctx(capi, params, pack) as c:
        full = (c.eval_sums(X), c.step(X[:2]))
    monkeypatch.setenv("STL_K1_SPLIT", "1")  # read when the pack is uploaded
    with _ctx(capi, params, pack, S) as c:
        got = (c.eval_sums(X), c.step(X[:2]))
    with _ctx(capi, params, pack) as c:
        got_full = (c.eval_sums(X), c.step(X[:2]))
    monkeypatch.delenv("STL_K1_SPLIT")
    for g, w in zip(got + got_full, want + full):
        assert np.array_equal(g, w)


@pytest.mark.parametrize("name", ["all", "sparse"])
def test_eval_frames(capi, params, pack, X, name):
    S = SELECTIONS[name]
    with _ctx(capi, params, pack, None if name == "all" else S) as c:
        fr = c.eval_frames(X)
        wf = c.work_counters()
        ev = c.eval_sums(X)
        we = c.work_counters()
        for k in ("points", "q2d", "q3d_nn", "q3d_knn", "k1_bytes"):  # eval_frames counts what stl_eval_batch counts
            assert wf[k] == we[k], k
        assert we["q3d_nn"] > 0
        assert fr.shape == (len(X), pack.n_kf, 13)
        for b in range(len(X)):
            for f in range(pack.n_kf):
                d = np.array(list(c.debug_frame(b, f).values()))
                assert np.array_equal(fr[b, f], d), (b, f)
    off = [f for f in range(pack.n_kf) if f not in S]
    assert not fr[:, off].any()
    assert fr[:, S, 5].sum() > 0
    tot = fr.sum(axis=1)
    # columns of the record: sum_3d2d, sum_3d3d, sum_he, cnt_he, cnt_3d2d, valid_3d2d, cnt_3d3d, valid_3d3d, valid_pl, valid_pt, kept, n_corr
    cols = [0, 8, 3, 4, 2, 1, 10, 9, 11, 12, 5, 6]
    rec = tot[:, cols]
    counts = [3, 4, 5, 6, 7, 8, 9, 10, 11]
    assert np.array_equal(rec[:, counts], ev[:, counts])
    for j in (0, 1, 2):
        assert np.allclose(rec[:, j], ev[:, j], rtol=1e-13, atol=0)


def test_eval_frames_chunks_and_unit_3d_weight(capi, pkg, pack, synth, small_pack, monkeypatch):
    X5 = synth.candidates(small_pack[1], 5, spread=0.4)
    S = SELECTIONS["every2"]
    p = pkg.default_params()
    with _ctx(capi, p, pack, S) as c:
        want = c.eval_frames(X5)
    monkeypatch.setenv("STL_MAX_CHUNK", "2")
    with _ctx(capi, p, pack, S) as c:
        got = c.eval_frames(X5)
        assert c.eval_sums(X5).shape == (5, 12)
    monkeypatch.delenv("STL_MAX_CHUNK")
    assert np.array_equal(got, want)
    # err_weight[1] = 0: the record counts one valid 3-D term per kept frame, and so do the rows
    p.err_weight[1] = 0.0
    with _ctx(capi, p, pack, S) as c:
        fr = c.eval_frames(X5)
        ev = c.eval_sums(X5)
    assert np.array_equal(fr[..., 9], fr[..., 5]) and np.array_equal(fr[..., 10], fr[..., 5]) and not fr[..., [8, 11, 12]].any()
    assert np.array_equal(fr.sum(axis=1)[:, [9, 10]], ev[:, [7, 6]])


def test_eval_frames_leaves_the_association_to_reuse(capi, params, pack, X):
    with _ctx(capi, params, pack, SELECTIONS["run"]) as c:
        c.eval_frames(X)
        before = c.work_counters()["assoc_reused"]
        nb = c.associate(X[2])
        assert c.work_counters()["assoc_reused"] == before + 1
        lin = c.linearize(X[2])
    with _ctx(capi, params, pack.select(SELECTIONS["run"])) as c:
        assert np.array_equal(nb, c.associate(X[2])) and np.array_equal(lin, c.linearize(X[2]))


def test_poll_search_on_a_selection(capi, pkg, pack, small_pack, small_candidates):
    host = importlib.import_module(PKG + ".host")
    optim = importlib.import_module(PKG + ".optim")
    x_gt, x0 = small_pack[1], small_candidates[2]
    lb, ub = x_gt + LB, x_gt - LB
    kw = dict(max_bb_eval=41, init_frame=0.5 * (-LB))
    S = SELECTIONS["every2"]
    p = pkg.default_params()
    with _ctx(capi, p, pack, S) as c:
        xs, bs, ns, hs = optim.poll_search(host.BALoss(c), x0, lb, ub, **kw)
    with _ctx(capi, p, pack.select(S)) as c:
        xw, bw, nw, hw = optim.poll_search(host.BALoss(c), x0, lb, ub, **kw)
    assert np.array_equal(xs, xw) and ns == nw and np.array_equal(np.asarray(bs), np.asarray(bw))
