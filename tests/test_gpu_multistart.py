"""Problem sets on the LM path (stl_associate_multi / stl_linearize_multi / stl_step_multi): problem p gives, bit for bit,
what a fresh stl_associate(x0[p]) + stl_linearize_batch gives, whatever else shares the call.  Every test makes its own
contexts, so that no other file ever sees a context holding a set of several problems."""
import importlib

import numpy as np
import pytest

from conftest import PKG, has_cuda

pytestmark = pytest.mark.gpu

ROT_TOL, TRANS_TOL = np.deg2rad(0.01), 1e-3


@pytest.fixture(scope="module")
def capi():
    if not has_cuda():
        pytest.skip("no CUDA device")
    return importlib.import_module(PKG + ".capi")


@pytest.fixture(scope="module")
def pack(small_pack):
    return small_pack[0].shard(0, 3)


@pytest.fixture(scope="module")
def starts(synth, small_pack):
    return synth.candidates(small_pack[1], 5, spread=0.5)


@pytest.fixture(params=[1, 0], ids=["plane-index", "plane-fit"])
def params(request, pkg):
    p = pkg.default_params()
    p.plane_index = request.param
    return p


def _ctx(capi, params, pack):
    c = capi.Context(params=params)
    c.upload(pack)
    return c


def _single(capi, params, pack, x0, X):
    """block counts and [B,62] of a fresh single association at x0, linearised at the rows of X"""
    with _ctx(capi, params, pack) as c:
        return c.associate(x0), c.linearize(np.atleast_2d(X))


def test_set_equals_single_associations_and_oracle(capi, params, pack, starts, oracle_mod):
    with _ctx(capi, params, pack) as c:
        nb = c.associate_multi(starts)
        lin = c.linearize_multi(starts)
        assert np.array_equal(c.block_counts_multi(), nb)
    orc = oracle_mod.Oracle(pack, kind="best")
    for p, x in enumerate(starts):
        nb1, lin1 = _single(capi, params, pack, x, x)
        assert np.array_equal(nb[p], nb1), p
        assert np.array_equal(lin[p], lin1[0]), p
        nb_o, ties = orc.associate(x)
        want = orc.linearize(x[None])
        assert np.array_equal(nb[p], nb_o)
        assert np.array_equal(lin[p, 57:], want[0, 57:])
        assert np.allclose(lin[p, 0], want[0, 0], rtol=1e-9, atol=0)
        sg, sh = np.abs(want[0, 1:8]).max(), np.abs(want[0, 8:57]).max()
        assert np.allclose(lin[p, 1:8], want[0, 1:8], rtol=1e-6, atol=1e-9 * sg)
        assert np.allclose(lin[p, 8:57], want[0, 8:57], rtol=1e-6, atol=1e-9 * sh)


def test_problem_index_mapping(capi, params, pack, starts):
    rng = np.random.default_rng(3)
    prob = np.repeat(np.arange(len(starts)), 3)
    rng.shuffle(prob)
    X = starts[prob] + rng.normal(scale=1e-3, size=(len(prob), 7))
    with _ctx(capi, params, pack) as c:
        c.associate_multi(starts)
        got = c.linearize_multi(X, prob)
    for p, x0 in enumerate(starts):
        _, want = _single(capi, params, pack, x0, X[prob == p])
        assert np.array_equal(got[prob == p], want), p


def test_rebuild_mask(capi, params, pack, starts, synth, small_pack):
    moved = synth.candidates(small_pack[1], 5, spread=0.3) + 1e-3
    mask = np.array([1, 0, 1, 0, 0], np.uint8)
    X1 = np.where(mask[:, None] == 1, moved, np.nan)  # the rows of untouched problems are not read
    with _ctx(capi, params, pack) as c:
        nb0 = c.associate_multi(starts)
        lin0 = c.linearize_multi(starts)
        nb1 = c.associate_multi(X1, rebuild=mask)
        xs = np.where(mask[:, None] == 1, moved, starts)
        lin1 = c.linearize_multi(xs)
    for p in range(5):
        if mask[p]:
            nbs, lins = _single(capi, params, pack, moved[p], moved[p])
            assert np.array_equal(nb1[p], nbs) and np.array_equal(lin1[p], lins[0]), p
        else:
            assert np.array_equal(nb1[p], nb0[p]) and np.array_equal(lin1[p], lin0[p]), p


def test_step_multi_equals_the_three_calls(capi, params, pack, starts):
    with _ctx(capi, params, pack) as c:
        step = c.step_multi(starts)
        step_again = c.step_multi(starts, rebuild=np.ones(5))
    with _ctx(capi, params, pack) as c:  # after an evaluation at the same starts: the correspondences are reused
        ev = c.eval_sums(starts)
        c.associate_multi(starts)
        lin = c.linearize_multi(starts)
        assert c.work_counters()["assoc_reused"] >= 5
    with _ctx(capi, params, pack) as c:  # no evaluation before: the association runs K1 itself
        c.associate_multi(starts)
        lin_cold = c.linearize_multi(starts)
    assert np.array_equal(step[:, :12], ev)
    assert np.array_equal(step[:, 12:], lin)
    assert np.array_equal(lin_cold, lin)
    assert np.array_equal(step_again, step)


def test_workspace_chunks(capi, params, pack, starts, monkeypatch):
    monkeypatch.setenv("STL_MAX_CHUNK", "2")  # read when the context sizes its workspace
    with _ctx(capi, params, pack) as c:
        c.eval_sums(starts[:1])
        nb = c.associate_multi(starts)
        lin = c.linearize_multi(starts)
        step = c.step_multi(starts)
    monkeypatch.delenv("STL_MAX_CHUNK")
    for p, x in enumerate(starts):
        nb1, lin1 = _single(capi, params, pack, x, x)
        assert np.array_equal(nb[p], nb1) and np.array_equal(lin[p], lin1[0]), p
    assert np.array_equal(step[:, 12:], lin)


def test_workspace_chunks_with_rebuild_mask(capi, params, pack, starts, synth, small_pack, monkeypatch):
    """a rebuild mask under a workspace of two candidates: the re-associated problems are a sparse list spread over chunks"""
    moved = synth.candidates(small_pack[1], 5, spread=0.3) + 1e-3
    mask = np.array([1, 0, 1, 1, 0], np.uint8)
    monkeypatch.setenv("STL_MAX_CHUNK", "2")
    with _ctx(capi, params, pack) as c:
        c.associate_multi(starts)
        nb = c.associate_multi(np.where(mask[:, None] == 1, moved, starts), rebuild=mask)
        lin = c.linearize_multi(moved)
    with _ctx(capi, params, pack) as c:
        c.step_multi(starts)
        step = c.step_multi(moved, rebuild=mask)
        ev = c.eval_sums(moved)
    monkeypatch.delenv("STL_MAX_CHUNK")
    for p in range(5):
        nb1, lin1 = _single(capi, params, pack, moved[p] if mask[p] else starts[p], moved[p])
        assert np.array_equal(nb[p], nb1) and np.array_equal(lin[p], lin1[0]), p
    assert np.array_equal(step[:, 12:], lin) and np.array_equal(step[:, :12], ev)


def test_gpr_blocks(capi, pkg, pack, starts):
    p = pkg.default_params(); p.use_gpr = 1
    with _ctx(capi, p, pack) as c:
        nb = c.associate_multi(starts[:3])
        lin = c.linearize_multi(starts[:3])
    assert nb[:, 3].sum() > 0
    for q in range(3):
        nb1, lin1 = _single(capi, p, pack, starts[q], starts[q])
        assert np.array_equal(nb[q], nb1) and np.array_equal(lin[q], lin1[0]), q


def test_single_calls_on_a_set(capi, params, pack, starts):
    with _ctx(capi, params, pack) as c:
        nb1 = c.associate_multi(starts[:1])           # a set of one is what stl_associate makes
        assert np.array_equal(c.block_counts(), nb1[0])
        l1 = c.linearize(starts[0])
        c.associate_multi(starts)
        for call in (lambda: c.linearize(starts[0]), c.block_counts, lambda: c.eval_blocks(starts[0]),
                     lambda: c.step(starts[:1], reassociate=False), c.gpr_hyper):
            with pytest.raises(capi._abi.StlError) as e:
                call()
            assert e.value.code == 4
        c.associate(starts[0])
        assert np.array_equal(c.linearize(starts[0]), l1)
        assert np.array_equal(c.block_counts(), nb1[0])


def test_error_codes(capi, pkg, pack, starts):
    with _ctx(capi, pkg.default_params(), pack) as c:
        def code(f):
            with pytest.raises(capi._abi.StlError) as e:
                f()
            return e.value.code
        assert code(lambda: c.associate_multi(np.zeros((0, 7)))) == 1
        assert code(lambda: c.associate_multi(np.repeat(starts[:1], 257, axis=0))) == 5
        assert code(lambda: c.step_multi(np.repeat(starts[:1], 257, axis=0))) == 5
        c.associate_multi(starts)
        assert code(lambda: c.linearize_multi(starts[:2], [0, 5])) == 1
        assert code(lambda: c.linearize_multi(starts[:2], [-1, 0])) == 1
        assert code(lambda: c.linearize_multi(starts[:2])) == 1          # problem = NULL needs B == P
        assert code(lambda: c.associate_multi(starts[:4], rebuild=np.ones(4))) == 1
        assert code(lambda: c.step_multi(starts[:4], rebuild=np.ones(4))) == 1
        assert c.linearize_multi(starts).shape == (5, 62)               # the set survived the refusals
    p = pkg.default_params(); p.variant = 1
    with _ctx(capi, p, pack) as c:
        assert code(lambda: c.associate_multi(starts)) == 4


def test_lm_refine_multi(capi, pkg, pack, starts, oracle_mod):
    host = importlib.import_module(PKG + ".host")
    optim = importlib.import_module(PKG + ".optim")
    kw = dict(max_iba_iter=3, max_num_iterations=8)
    X0 = starts[:3]
    with _ctx(capi, pkg.default_params(), pack) as c:
        X, costs = optim.lm_refine_multi(host.LMProblemSet(c), X0, **kw)
    orc = oracle_mod.Oracle(pack, kind="best")

    class OracleProblem:
        def build(self, x):
            return orc.associate(x)[0]

        def evaluate(self, x):
            s = orc.linearize(np.asarray(x, dtype=np.float64).reshape(1, 7))
            return float(s[0, 0]), s[0, 1:8].copy(), s[0, 8:57].reshape(7, 7).copy()

    with _ctx(capi, pkg.default_params(), pack) as c:
        for p in range(len(X0)):
            x1, c1 = optim.lm_refine(host.LMProblem(c), X0[p], **kw)
            assert np.array_equal(X[p], x1) and costs[p] == c1, p
            xo, co = optim.lm_refine(OracleProblem(), X0[p], **kw)
            assert len(co) == len(c1) and np.allclose(c1, co, rtol=1e-6)
            assert np.abs(x1[:3] - xo[:3]).max() < ROT_TOL and np.abs(x1[3:6] - xo[3:6]).max() < TRANS_TOL
