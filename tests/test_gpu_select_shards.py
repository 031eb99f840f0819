"""Keyframe selection over keyframe shards on two GPUs: every rank selects its part of one global selection in local indices
(rank 0 none, rank 1 a subset of its shard), every rank still makes every call, and the exchanged records equal those of one
GPU holding all keyframes with the same global selection.  Worker pattern of test_gpu_multi.py; skipped with fewer than two
GPUs."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from conftest import PKG, ROOT, has_cuda

pytestmark = pytest.mark.gpu

GLOBAL_SEL = [3, 5]  # shard bounds of 6 keyframes over 2 ranks: (0, 3), (3, 6) -> rank 0 selects nothing


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
    with capi.Context(device=rank) as c:
        par.attach_communicator(c, rank, world, id_file=idf)
        c.upload(pack)
        c.select_keyframes(par.local_selection({sel!r}, b, e))
        ev = c.eval_sums(X)
        st = c.step(X[:2])
        ms = c.step_multi(X[:3])
        fr = c.eval_frames(X)
        np.savez(outf, ev=ev, st=st, ms=ms, fr=fr)
""")


@pytest.mark.skipif(not has_cuda() or _n_gpus() < 2, reason="needs two GPUs")
def test_selection_over_keyframe_shards(tmp_path, synth):
    import importlib
    capi = importlib.import_module(PKG + ".capi")
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT, pkg=PKG, sel=GLOBAL_SEL))
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
        c.select_keyframes(GLOBAL_SEL)
        ev, st, ms, fr = c.eval_sums(X), c.step(X[:2]), c.step_multi(X[:3]), c.eval_frames(X)
    # rank 0 holds no selected keyframe: its records are rank 1's alone, exchanged; every rank returns the totals
    for r in (r0, r1):
        assert np.array_equal(r["ev"], ev)
        assert np.array_equal(r["st"], st)
        assert np.array_equal(r["ms"], ms)
    # no exchange for the per-keyframe rows: each rank returns its own keyframes
    assert not r0["fr"].any()
    assert np.array_equal(np.concatenate([r0["fr"], r1["fr"]], axis=1), fr)
