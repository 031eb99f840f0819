"""Per-keyframe normal equations on the LM path (stl_linearize_frames): the rows of a candidate sum to its record, row f is
what a context holding keyframe f alone computes (and what the oracle computes for it), and a row is bit for bit the same
whatever the batch, the selection, the problem set or the keyframe shard around it.  Every test makes its own contexts."""
import importlib
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from conftest import PKG, ROOT, has_cuda

pytestmark = pytest.mark.gpu

F = 6  # keyframes of small_pack
STATE, INVALID = 4, 1


@pytest.fixture(scope="module")
def capi():
    if not has_cuda():
        pytest.skip("no CUDA device")
    return importlib.import_module(PKG + ".capi")


@pytest.fixture(scope="module")
def pack(small_pack):
    return small_pack[0]


@pytest.fixture(scope="module")
def X(small_candidates):
    return small_candidates  # 4 candidates; X[0] is the association point x0


@pytest.fixture(params=[1, 0], ids=["plane-index", "plane-fit"])
def params(request, pkg):
    p = pkg.default_params()
    p.plane_index = request.param
    return p


@pytest.fixture(scope="module")
def gpr_params(pkg):
    p = pkg.default_params()
    p.use_gpr = 1
    return p


def _ctx(capi, params, pack, sel=None):
    c = capi.Context(params=params)
    c.upload(pack)
    if sel is not None:
        c.select_keyframes(sel)
    return c


def _near(got, want, tol=1e-13):
    """counts ([57:62]) exactly; cost, J^T r and J^T J within tol x the largest of them, per record"""
    got, want = np.atleast_2d(got), np.atleast_2d(want)
    assert np.array_equal(got[:, 57:], want[:, 57:]), (got[:, 57:], want[:, 57:])
    scale = np.abs(want[:, :57]).max(axis=1, keepdims=True)
    err = np.abs(got[:, :57] - want[:, :57])
    assert (err <= tol * scale).all(), (err / np.maximum(scale, 1e-300)).max()


def _oracle_bar(got, want, tol_cost, tol_atol):
    """the bar of test_gpu_lm.py: counts exactly, cost relative, J^T r / J^T J 1e-6 relative + tol_atol x the largest entry"""
    got, want = np.atleast_2d(got), np.atleast_2d(want)
    assert np.array_equal(got[:, 57:], want[:, 57:])
    assert np.allclose(got[:, 0], want[:, 0], rtol=tol_cost, atol=0)
    sg = np.abs(want[:, 1:8]).max(axis=1, keepdims=True)
    sh = np.abs(want[:, 8:57]).max(axis=1, keepdims=True)
    assert np.allclose(got[:, 1:8], want[:, 1:8], rtol=1e-6, atol=tol_atol * sg)
    assert np.allclose(got[:, 8:57], want[:, 8:57], rtol=1e-6, atol=tol_atol * sh)


# ---- 1. the rows of a candidate sum to its record
@pytest.mark.parametrize("B", [1, 4])
def test_rows_sum_to_the_record(capi, params, pack, X, B):
    with _ctx(capi, params, pack) as c:
        c.associate(X[0])
        rows = c.linearize_frames(X[:B])
        rec = c.linearize_multi(X[:B], problem=np.zeros(B, np.int32))
    assert rows.shape == (B, F, 62)
    assert rec[:, 57].min() > 0 and (rec[:, 58] + rec[:, 59]).min() > 0 and (rows[:, :, 57] > 0).sum() > 1  # both kinds, several keyframes
    _near(rows.sum(axis=1), rec)


def test_rows_sum_to_the_record_of_a_problem_set(capi, params, pack, X):
    problem = np.array([2, 0, 2, 1], np.int32)
    with _ctx(capi, params, pack) as c:
        c.associate_multi(X[:3])
        rows = c.linearize_frames(X, problem=problem)
        rec = c.linearize_multi(X, problem=problem)
    _near(rows.sum(axis=1), rec)


# ---- 2. / 3. row f is keyframe f alone: a fresh association of it, and the oracle on it
def test_row_equals_a_context_holding_the_keyframe_alone(capi, params, pack, X):
    with _ctx(capi, params, pack) as c:
        c.associate(X[0])
        rows = c.linearize_frames(X)
    for f in range(F):
        with _ctx(capi, params, pack, [f]) as c:
            c.associate(X[0])
            _near(rows[:, f], c.linearize(X))


def test_row_against_the_oracle(capi, params, pack, X, oracle_mod):
    with _ctx(capi, params, pack) as c:
        c.associate(X[0])
        rows = c.linearize_frames(X)
    for f in range(F):
        orc = oracle_mod.Oracle(pack.select([f]), kind="best")
        orc.associate(X[0])
        _oracle_bar(rows[:, f], orc.linearize(X), 1e-9, 1e-9)


# ---- 4. block counts against the per-block output
def test_counts_equal_the_per_block_histogram(capi, params, pack, X):
    with _ctx(capi, params, pack) as c:
        c.associate(X[0])
        rows = c.linearize_frames(X[1])
        blk = c.eval_blocks(X[1])
    for f in range(F):
        on = blk["kf"] == f
        want = [np.sum(on & (blk["type"] == t)) for t in (0, 1, 2)] + [blk["n_res"][on].sum(), np.sum(on & (blk["type"] == 3))]
        assert rows[0, f, 57:].tolist() == want, f


# ---- 5. bitwise invariance
def test_row_alone_and_in_a_batch(capi, params, pack, X):
    with _ctx(capi, params, pack) as c:
        c.associate(X[0])
        rows = c.linearize_frames(X)
        for b in range(len(X)):
            assert np.array_equal(c.linearize_frames(X[b:b + 1])[0], rows[b])
        assert np.array_equal(c.linearize_frames(X[::-1]), rows[::-1])


@pytest.mark.parametrize("sel", [[0, 3, 4], [5], [1, 2, 3, 4, 5]])
def test_row_under_a_selection(capi, params, pack, X, sel):
    with _ctx(capi, params, pack) as c:
        c.associate(X[0])
        rows = c.linearize_frames(X)
        c.select_keyframes(sel)
        c.associate(X[0])
        got = c.linearize_frames(X)
    out = [f for f in range(F) if f not in sel]
    assert np.array_equal(got[:, sel], rows[:, sel])
    assert not got[:, out].any()


def test_empty_selection_gives_zero_rows(capi, params, pack, X):
    with _ctx(capi, params, pack, []) as c:
        c.associate(X[0])
        got = c.linearize_frames(X)
    assert got.shape == (len(X), F, 62) and not got.any()


def test_row_in_a_problem_set_and_in_a_set_of_one(capi, params, pack, X):
    problem = [2, 0, 2, 1]
    with _ctx(capi, params, pack) as c:
        c.associate_multi(X[:3])
        rows = c.linearize_frames(X, problem=problem)
        for p in range(3):
            c.associate(X[p])
            for b in np.flatnonzero(np.asarray(problem) == p):
                assert np.array_equal(c.linearize_frames(X[b:b + 1])[0], rows[b]), (p, b)


# ---- 6. leave one keyframe out, end to end
def test_leave_one_out(capi, params, pack, X):
    with _ctx(capi, params, pack) as c:
        c.associate(X[0])
        rows = c.linearize_frames(X)
    total = rows.sum(axis=1)
    for f in range(F):
        with _ctx(capi, params, pack, [k for k in range(F) if k != f]) as c:
            c.associate(X[0])
            _near(total - rows[:, f], c.linearize(X))


# ---- 7. with IBA_GPRFactor blocks
def test_gpr_rows(capi, gpr_params, pack, X, oracle_mod):
    sub = pack.shard(0, 3)
    with _ctx(capi, gpr_params, sub) as c:
        c.associate(X[0])
        rows = c.linearize_frames(X)
        rec = c.linearize(X)
        assert np.array_equal(c.linearize_frames(X[2:3])[0], rows[2])
    assert rec[:, 61].min() > 0 and (rows[:, :, 61] > 0).sum() > 1
    _near(rows.sum(axis=1), rec)
    for f in range(3):
        with _ctx(capi, gpr_params, sub, [f]) as c:
            c.associate(X[0])
            _near(rows[:, f], c.linearize(X))
            assert np.array_equal(c.linearize_frames(X)[:, f], rows[:, f])
        orc = oracle_mod.Oracle(sub.select([f]), params=gpr_params, kind="best")
        orc.associate(X[0])
        _oracle_bar(rows[:, f], orc.linearize(X), 1e-6, 1e-6)


# ---- 8. error codes; the set survives every refusal
def test_error_codes(capi, pkg, pack, X):
    def code(f):
        with pytest.raises(capi._abi.StlError) as e:
            f()
        return e.value.code

    with _ctx(capi, pkg.default_params(), pack) as c:
        assert code(lambda: c.linearize_frames(X)) == STATE                      # no association
        c.associate(X[0])
        c.select_keyframes(None)
        assert code(lambda: c.linearize_frames(X)) == STATE                      # a selection call since
        problem = [2, 0, 2, 1]
        c.associate_multi(X[:3])
        want = c.linearize_frames(X, problem=problem)
        out = np.zeros((1, 62))
        refusals = [lambda: code(lambda: c.linearize_frames(X, problem=[0, 3, 0, 0])) == INVALID,
                    lambda: code(lambda: c.linearize_frames(X, problem=[0, -1, 0, 0])) == INVALID,
                    lambda: code(lambda: c.linearize_frames(X)) == STATE,       # NULL problem on a set of 3
                    lambda: c.lib.stl_linearize_frames(c.h, X.ctypes.data_as(capi._dp), 0, None,  # B = 0
                                                       out.ctypes.data_as(capi.C.POINTER(capi._abi.LinSums))) == INVALID]
        for i, refused in enumerate(refusals):
            assert refused(), i
            assert np.array_equal(c.linearize_frames(X, problem=problem), want), i
    p = pkg.default_params()
    p.variant = 1
    with _ctx(capi, p, pack) as c:
        assert code(lambda: c.associate(X[0])) == STATE
        assert code(lambda: c.linearize_frames(X)) == STATE


# ---- 9. keyframe shards on two GPUs: each rank's rows are the single-GPU rows of its keyframes
def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


_WORKER = textwrap.dedent("""
    import importlib, sys
    import numpy as np
    sys.path.insert(0, {root!r})
    PKG = {pkg!r}
    rank, world, idf, outf = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3], sys.argv[4]
    capi = importlib.import_module(PKG + ".capi")
    par = importlib.import_module(PKG + ".parallel")
    synth = importlib.import_module(PKG + ".synth")
    F = 6
    b, e = par.shard_bounds(F, world, rank)
    pack, x_gt, _ = synth.generate(n_kf=e - b, kf_begin=b, n_kf_total=F, seed=1000)
    X = synth.candidates(x_gt, 4, 0.4)
    with capi.Context(device=rank) as c:
        par.attach_communicator(c, rank, world, id_file=idf)
        c.upload(pack)
        c.associate(X[0])
        fr = c.linearize_frames(X)
        c.associate_multi(X[:3])
        fm = c.linearize_frames(X, problem=[2, 0, 2, 1])
        np.savez(outf, fr=fr, fm=fm)
""")


@pytest.mark.skipif(not has_cuda() or _n_gpus() < 2, reason="needs two GPUs")
def test_rows_over_keyframe_shards(tmp_path, synth):
    capi = importlib.import_module(PKG + ".capi")
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT, pkg=PKG))
    idf = str(tmp_path / "nccl_id.bin")
    env = dict(os.environ, OMP_NUM_THREADS="4")
    procs = [subprocess.Popen([sys.executable, str(script), str(r), "2", idf, str(tmp_path / f"out{r}.npz")],
                              stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env) for r in range(2)]
    outs = [p.communicate(timeout=600) for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    r0, r1 = (np.load(str(tmp_path / f"out{r}.npz")) for r in range(2))
    pack, x_gt, _ = synth.generate(n_kf=6, seed=1000)
    X = synth.candidates(x_gt, 4, 0.4)
    with capi.Context(device=0) as c:
        c.upload(pack)
        c.associate(X[0])
        fr = c.linearize_frames(X)
        c.associate_multi(X[:3])
        fm = c.linearize_frames(X, problem=[2, 0, 2, 1])
    for key, want in (("fr", fr), ("fm", fm)):
        assert np.array_equal(np.concatenate([r0[key], r1[key]], axis=1), want), key
