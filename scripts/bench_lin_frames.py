#!/usr/bin/env python3
"""Per-keyframe normal equations (stl_linearize_frames) against the record (stl_linearize_multi) on ONE GPU, same frozen problem.

Workload: the KITTI-00 shape of bench.py (config c2: 1500 synthetic keyframes, 64 beams x 1875 azimuth steps, generator seed
1000), default params, BuildProblem at the first of synth.candidates(x_gt, 257, 0.2, seed = 42)[1:] (bench.py's candidate stream);
the B candidates are the first B of that stream, B in --B.  Also use_gpr = 1 at B = 1 (--gpr-B).
For each B and call, over --rounds interleaved rounds (record, then frames, in every round), each after --warmup untimed calls:
  stage: the STL_STAGE_LINEARIZE stage (the library's CUDA events, profiling on) per call, averaged over --iters calls;
  wall:  host clock around --iters host calls (profiling off), which includes the copy of the [B][62] / [B][n_kf][62] rows.
Reports median and min-max over the rounds.  Checks, in the same run, that the rows of every candidate sum to its record:
counts exactly, cost / J^T r / J^T J within 1e-13 of the record's largest entry.  Writes JSON with the card's name, power limit
and max SM clock (read in the same run) to --out."""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = "spatial-temporal-lidar-camera-calibration_b200"
LIN = 3  # STAGE_NAMES index of "linearize"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # the measurement still stands; say that the card could not be read
        return f"unavailable ({e})"


def sum_check(rows, rec):
    """(counters exact, max |sum - record| over the record's largest cost / J^T r / J^T J entry)"""
    s = rows.sum(axis=1)
    exact = bool(np.array_equal(s[:, 57:], rec[:, 57:]))
    scale = np.abs(rec[:, :57]).max(axis=1)
    rel = float((np.abs(s[:, :57] - rec[:, :57]).max(axis=1) / np.maximum(scale, 1e-300)).max())
    return exact, rel


def stats(v):
    v = np.asarray(v)
    return dict(median=float(np.median(v)), min=float(v.min()), max=float(v.max()))


def measure(ctx, X, B, args):
    Xb = X[:B]
    prob = np.zeros(B, np.int32)
    calls = {"record": lambda: ctx.linearize_multi(Xb, problem=prob), "frames": lambda: ctx.linearize_frames(Xb)}
    st = {k: [] for k in calls}
    wall = {k: [] for k in calls}
    for r in range(args.rounds):
        for name, f in calls.items():
            for _ in range(args.warmup):
                f()
            ctx.set_profiling(True)
            ctx.stage_stats()  # reset
            for _ in range(args.iters):
                f()
            ms, n = ctx.stage_stats()["linearize"]
            ctx.set_profiling(False)
            st[name].append(ms / args.iters)
            t0 = time.perf_counter()
            for _ in range(args.iters):
                f()
            wall[name].append((time.perf_counter() - t0) * 1e3 / args.iters)
    exact, rel = sum_check(calls["frames"](), calls["record"]())
    res = dict(B=B, stage_ms={k: stats(v) for k, v in st.items()}, wall_ms={k: stats(v) for k, v in wall.items()},
               stage_ratio_frames_over_record=float(np.median(st["frames"]) / np.median(st["record"])),
               wall_ratio_frames_over_record=float(np.median(wall["frames"]) / np.median(wall["record"])),
               sum_counters_exact=exact, sum_max_rel_err=rel, sum_ok=bool(exact and rel <= 1e-13))
    log(json.dumps(res))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nkf", type=int, default=1500)
    ap.add_argument("--B", default="1,16,256")
    ap.add_argument("--gpr-B", default="1", help="B values measured with use_gpr = 1 (empty: none)")
    ap.add_argument("--iters", type=int, default=10, help="timed calls per round")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seed", type=int, default=1000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_lin_frames.json"))
    args = ap.parse_args()
    Bs = [int(v) for v in args.B.split(",") if v]
    gBs = [int(v) for v in args.gpr_B.split(",") if v]
    import torch  # before the library: its NCCL must be the one torch resolves
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU")
    pkg = importlib.import_module(PKG)
    synth = importlib.import_module(PKG + ".synth")
    capi = importlib.import_module(PKG + ".capi")
    card = gpu_info()
    log("card:", card)
    t0 = time.perf_counter()
    pack, x_gt, _ = synth.generate(n_kf=args.nkf, beams=64, az_steps=1875, seed=args.seed)
    log(f"pack: {args.nkf} keyframes in {time.perf_counter() - t0:.1f}s")
    X = synth.candidates(x_gt, max(Bs + gBs) + 1, 0.2, seed=42)[1:]
    out = dict(what=__doc__.split("\n")[0], gpu=card, keyframes=args.nkf, seed=args.seed, iters=args.iters, rounds=args.rounds,
               warmup=args.warmup, results=[], results_gpr=[])
    ok = True
    for use_gpr, Bl, key in ((0, Bs, "results"), (1, gBs, "results_gpr")):
        if not Bl:
            continue
        params = pkg.default_params()
        params.use_gpr = use_gpr
        with capi.Context(params=params) as ctx:
            ctx.upload(pack)
            ctx.eval_sums(X[:1])
            nb = ctx.associate(X[0])
            out["blocks" if not use_gpr else "blocks_gpr"] = nb.tolist()
            for B in Bl:
                r = measure(ctx, X, B, args)
                ok &= r["sum_ok"]
                out[key].append(r)
    out["ok"] = bool(ok)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))
    return 0 if ok else 3


if __name__ == "__main__":
    sys.exit(main())
