"""Keyframe sharding across the GPUs of a node (SURVEY.md §8e): one process per GPU.

Every (candidate, keyframe) pair is independent up to the final sums
(iba_global.cpp:243-250,322-325,274-275), and everything a keyframe needs from its covisible
keyframes is baked into its own pack rows, so a contiguous block of keyframes per rank needs no
halo.  The only exchange is ONE fp64 sum all-reduce of the per-candidate record
([B,12] evaluation, [B,62] linearisation, [B,74] fused step); counters travel as doubles (exact
< 2^53).  On GPUs the all-reduce is issued by the LIBRARY on its compute stream, over an NCCL
communicator the context owns (``stl_comm_init``): this module only decides who holds which
keyframes and carries the 128-byte communicator id between the processes.  A batch of
candidates larger than the work-buffer chunk is walked chunk by chunk inside the library, so
with B >= G the tiling is (candidate chunk) x (keyframe shard) with a single all-reduce at the end.
``SumAllReduce`` is the host-side equivalent over ``torch.distributed`` (gloo in the CPU tests).
"""
from __future__ import annotations

import os
import time

import numpy as np


def shard_bounds(n_kf: int, world: int, rank: int) -> tuple[int, int]:
    """Contiguous keyframe block of `rank`: sizes differ by at most one."""
    base, rem = divmod(n_kf, world)
    begin = rank * base + min(rank, rem)
    return begin, begin + base + (1 if rank < rem else 0)


def local_selection(global_kf, begin: int, end: int) -> np.ndarray:
    """The part of a global keyframe selection that falls in the shard [begin, end), as the LOCAL indices
    ``Context.select_keyframes`` takes on that rank (empty where the rank holds none of it: the rank still makes the call)."""
    g = np.asarray(global_kf)
    if g.size == 0:
        g = g.astype(np.int64).reshape(0)
    if g.ndim != 1 or g.dtype.kind not in "iu":
        raise TypeError("local_selection: global_kf must be a 1-D list of integer keyframe indices")
    g = g.astype(np.int64)
    if np.any(np.diff(g) <= 0) or (g.size and g[0] < 0):
        raise ValueError("local_selection: global keyframe indices must be non-negative and strictly increasing")
    return (g[(g >= begin) & (g < end)] - begin).astype(np.int32)


def attach_communicator(ctx, rank: int, world: int, exchange=None, id_file: str | None = None, timeout_s: float = 120.0):
    """Attaches an NCCL communicator of `world` ranks to `ctx` (which must hold keyframe shard `rank`).

    Rank 0 draws the id (``stl_comm_unique_id``); it reaches the other ranks either through
    ``exchange`` — a callable ``bytes | None -> bytes`` (e.g. a torch.distributed / MPI broadcast) —
    or through ``id_file`` (rank 0 writes it atomically, the others wait for it): no framework is
    needed to bring the library's own collective up."""
    if world <= 1:
        return
    if exchange is not None:
        uid = exchange(ctx.comm_unique_id() if rank == 0 else None)
    elif id_file is not None:
        if rank == 0:
            uid = ctx.comm_unique_id()
            tmp = id_file + ".tmp"
            with open(tmp, "wb") as f:
                f.write(uid)
            os.replace(tmp, id_file)
        else:
            t0 = time.time()
            while not os.path.exists(id_file):
                if time.time() - t0 > timeout_s:
                    raise TimeoutError(f"communicator id file {id_file} did not appear")
                time.sleep(0.01)
            with open(id_file, "rb") as f:
                uid = f.read()
    else:
        raise ValueError("attach_communicator needs `exchange` or `id_file`")
    ctx.comm_init(uid, rank, world)


def torch_exchange(src: int = 0):
    """`exchange` callable for :func:`attach_communicator` over the default torch.distributed group."""
    import torch.distributed as dist

    def ex(uid):
        box = [uid]
        dist.broadcast_object_list(box, src=src)
        return box[0]
    return ex


class SumAllReduce:
    """Callable that all-reduces a host [B, n] fp64 array over the default process group."""

    def __init__(self, device=None):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.device = device
        self.enabled = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1

    def __call__(self, arr: np.ndarray) -> np.ndarray:
        if not self.enabled:
            return arr
        t = self.torch.from_numpy(np.ascontiguousarray(arr, dtype=np.float64))
        if self.device is not None:
            t = t.to(self.device)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return t.cpu().numpy()
