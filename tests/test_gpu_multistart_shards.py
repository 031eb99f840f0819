"""Problem sets over keyframe shards on two GPUs: the [P][62] / [P][74] records of stl_linearize_multi / stl_step_multi are
exchanged once (peer memory or NCCL) and every rank returns what one GPU holding all keyframes returns; block counts are per
shard and sum to the one-GPU counts.  Worker pattern of test_gpu_multi.py; skipped with fewer than two GPUs."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from conftest import PKG, ROOT, has_cuda

pytestmark = pytest.mark.gpu


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


_WORKER = textwrap.dedent("""
    import importlib, os, sys
    import numpy as np
    sys.path.insert(0, {root!r})
    PKG = {pkg!r}
    rank, world, idf, outf = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3], sys.argv[4]
    capi = importlib.import_module(PKG + ".capi")
    par = importlib.import_module(PKG + ".parallel")
    synth = importlib.import_module(PKG + ".synth")
    F = 6
    b, e = par.shard_bounds(F, world, rank)
    pack, x_gt, _ = synth.generate(n_kf=e - b, kf_begin=b, n_kf_total=F, seed=1000)   # this rank's keyframes only
    X = synth.candidates(x_gt, 4, 0.4)
    prob = np.array([2, 0, 3, 1, 2, 0], np.int32)
    with capi.Context(device=rank) as c:
        par.attach_communicator(c, rank, world, id_file=idf)
        c.upload(pack)
        st = c.step_multi(X)
        nb_st = c.block_counts_multi()
        nb = c.associate_multi(X)
        lin = c.linearize_multi(X[prob] + 1e-4, prob)
        cs = c.comm_stats()
        np.savez(outf, st=st, nb_st=nb_st, nb=nb, lin=lin, p2p=np.array([cs["p2p"], cs["p2p_exchanges"], cs["nccl_exchanges"]]))
""")


@pytest.mark.skipif(not has_cuda() or _n_gpus() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("exchange", ["peer-memory", "nccl"])
def test_problem_set_over_keyframe_shards(tmp_path, synth, exchange):
    import importlib
    capi = importlib.import_module(PKG + ".capi")
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT, pkg=PKG))
    idf = str(tmp_path / "nccl_id.bin")
    env = dict(os.environ, OMP_NUM_THREADS="4")
    if exchange == "nccl":
        env["STL_NO_P2P"] = "1"
    procs = [subprocess.Popen([sys.executable, str(script), str(r), "2", idf, str(tmp_path / f"out{r}.npz")],
                              stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env) for r in range(2)]
    outs = [p.communicate(timeout=600) for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    r0, r1 = (np.load(str(tmp_path / f"out{r}.npz")) for r in range(2))
    for key in ("st", "lin"):
        assert np.array_equal(r0[key], r1[key]), key                    # every rank holds the same totals
    if exchange == "nccl":
        assert r0["p2p"][0] == 0 and r0["p2p"][1] == 0 and r0["p2p"][2] >= 2, r0["p2p"]
    else:   # the finishing kernels exchanged the records themselves
        assert r0["p2p"][0] == 1 and r0["p2p"][1] >= 2 and r0["p2p"][2] == 0, r0["p2p"]
    pack, x_gt, _ = synth.generate(n_kf=6, seed=1000)
    X = synth.candidates(x_gt, 4, 0.4)
    prob = np.array([2, 0, 3, 1, 2, 0], np.int32)
    with capi.Context(device=0) as c:
        c.upload(pack)
        st = c.step_multi(X)
        nb_st = c.block_counts_multi()
        nb = c.associate_multi(X)
        lin = c.linearize_multi(X[prob] + 1e-4, prob)
    assert np.array_equal(r0["nb_st"] + r1["nb_st"], nb_st) and np.array_equal(r0["nb"] + r1["nb"], nb)  # per shard
    assert np.array_equal(r0["st"][:, 3:12], st[:, 3:12]) and np.allclose(r0["st"][:, :3], st[:, :3], rtol=1e-12, atol=0)
    assert np.array_equal(r0["st"][:, 12 + 57:], st[:, 12 + 57:])            # block / residual counts summed in the record
    sc = np.abs(st[:, 12:12 + 57]).max()
    assert np.allclose(r0["st"][:, 12:12 + 57], st[:, 12:12 + 57], rtol=1e-10, atol=1e-12 * sc)
    assert np.array_equal(r0["lin"][:, 57:], lin[:, 57:])
    sl = np.abs(lin[:, :57]).max()
    assert np.allclose(r0["lin"][:, :57], lin[:, :57], rtol=1e-10, atol=1e-12 * sl)
