#!/usr/bin/env python3
"""Multi-start LM refinement on ONE GPU (keyframe shards over several GPUs are not measured here): a problem set (stl_step_multi / stl_linearize_multi) against the only way there was
before it, P successive stl_step_batch(x[p], reassociate = 1) calls on one context.

Workload: the KITTI-00 shape of bench.py (config c2: 1500 synthetic keyframes, 64 beams x 1875 azimuth steps, k = 30, generator
seed 1000); the P starts are synth.candidates(x_gt, 65, 0.2, seed = 42)[1:P+1] (bench.py's candidate stream).  For every P it
times, interleaved over --rounds rounds (the spread is over those rounds), each with --warmup untimed calls first:
  (a) stl_step_multi(X[:P])                  every problem re-associated at its start: one LM iteration of P starts
  (b) stl_linearize_multi(X[:P])             the P problems frozen: one inner LM evaluation of P starts
  (c) P x stl_step_batch(X[p], 1, 1)         the single-problem context re-associating at every switch of start
The _device twins of the three calls are enqueued back to back on one stream and timed with CUDA events around --iters of
them (the host staging of a call overlaps the device work of the previous one).  Every timed
record is checked: row p of (a) and (b) equals (c)'s record of start p bit for bit, and one start is compared with the CPU
oracle (--oracle-sample, counters exact, sums within 1e-6).  Resident bytes of the set: computed from the allocation sizes
(per-problem arrays x P + association lanes x min(P, workspace chunk), at most P lanes); a device-wide free-memory difference is no measure on
a GPU other processes share.  Writes JSON (GPU name and power limit read in the same run) to --out."""
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


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # the measurement still stands; say that the card could not be read
        return f"unavailable ({e})"


def set_bytes(n_slots, P, lanes):
    """device bytes of a set of P problems with `lanes` association lanes, from the allocation sizes of lm_reserve (csrc/lm.cu)"""
    stride = (n_slots + 15) // 16 * 16
    per_problem = stride * (4 + 4 + 4 + 48 + 72 + 4 + 4) + 16   # slot_kf, slot_kp, 4 flags, geo2d, geo3d, 2-D / GPR lists; counts
    per_lane = n_slots * (1 + 32 + 4 + 4 * 32 + 16 * 32 + 4 + 8)  # stage, plane_a, nnb_pos, nbb, nbbx, nbb_m, nbb_last
    return per_problem, per_lane, per_problem * P + per_lane * lanes + 4 * n_slots  # + idx3d (problem 0)


def timed(torch, stream, f, n):
    """CUDA events on `stream` around n back-to-back enqueues of f (the _device calls): device ms per call"""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(n):
        f()
    b.record(stream)
    b.synchronize()
    return a.elapsed_time(b) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nkf", type=int, default=1500)
    ap.add_argument("--P", default="1,4,16,64")
    ap.add_argument("--iters", type=int, default=5, help="timed calls per round")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seed", type=int, default=1000)
    ap.add_argument("--oracle-sample", type=int, default=1, help="starts compared with the CPU oracle (0: none)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_lm_multistart.json"))
    args = ap.parse_args()
    Ps = [int(v) for v in args.P.split(",")]
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
    X = synth.candidates(x_gt, max(Ps) + 1, 0.2, seed=42)[1:]
    params = pkg.default_params()
    ctx = capi.Context(params=params)
    ctx.upload(pack)
    ctx.eval_sums(X[:1])
    ctx.associate(X[0])
    n_slots = int(np.count_nonzero(~np.isnan(np.asarray(pack.kp_mappoint).reshape(-1, 3)[:, 0])))
    out = dict(what=__doc__.split("\n")[0], gpu=card, keyframes=args.nkf, seed=args.seed, iters=args.iters, rounds=args.rounds,
               warmup=args.warmup, clock="CUDA events on the calls' stream around --iters back-to-back _device calls", results=[])
    stream = torch.cuda.Stream()
    sp = stream.cuda_stream
    d_out = torch.empty((max(Ps), 74), dtype=torch.float64, device="cuda")
    ptr, row = d_out.data_ptr(), 74 * 8
    ok_all = True
    for P in Ps:
        Xp = X[:P]
        ref = np.stack([ctx.step(Xp[p:p + 1], reassociate=True)[0] for p in range(P)])  # (c)'s records, also the yardstick

        def run_a():
            ctx.step_multi_device(Xp, ptr, stream_ptr=sp)

        def run_b():
            ctx.linearize_multi_device(Xp, ptr, stream_ptr=sp)

        def run_c():
            for p in range(P):
                ctx.step_device(Xp[p:p + 1], ptr + p * row, stream_ptr=sp, reassociate=True)

        def rec():
            stream.synchronize()
            return d_out[:P].cpu().numpy().copy()
        ta, tb, tc = [], [], []
        ok = True
        for r in range(args.rounds):
            for _ in range(args.warmup):
                run_a()
            ta.append(timed(torch, stream, run_a, args.iters))
            ok &= bool(np.array_equal(rec(), ref))
            ctx.associate_multi(Xp)
            for _ in range(args.warmup):
                run_b()
            tb.append(timed(torch, stream, run_b, args.iters))
            stream.synchronize()
            ok &= bool(np.array_equal(d_out.view(-1)[:P * 62].cpu().numpy().reshape(P, 62), ref[:, 12:]))
            for _ in range(args.warmup):
                run_c()
            tc.append(timed(torch, stream, run_c, args.iters))
            ok &= bool(np.array_equal(rec(), ref))
        ok_all &= ok

        def per(ts):
            v = np.asarray(ts) / P
            return dict(median=float(np.median(v)), min=float(v.min()), max=float(v.max()))
        res = dict(P=P, a_step_multi_ms_per_problem_iter=per(ta), b_linearize_multi_ms_per_problem_iter=per(tb),
                   c_sequential_step_batch_ms_per_problem_iter=per(tc), speedup_a_over_c=float(np.median(tc) / np.median(ta)),
                   set_bytes_at_most=set_bytes(n_slots, P, P)[2], bitwise_equal_to_single=ok)
        out["results"].append(res)
        log(json.dumps(res))
    pp, pl, _ = set_bytes(n_slots, 1, 1)
    out.update(map_point_slots=n_slots, bytes_per_problem=pp, bytes_per_association_lane=pl,
               bytes_note="from the sizes lm_reserve allocates: per-problem arrays x P + association lanes x min(P, workspace chunk); "
                          "set_bytes_at_most counts P lanes")
    if args.oracle_sample > 0:
        from oracle import oracle as O
        orc = O.Oracle(pack, params=params, kind="ref" if O.have_ref() else "port", nthreads=os.cpu_count())
        rec = ctx.step_multi(X[:max(Ps)])
        errs, exact = 0.0, True
        for p in range(min(args.oracle_sample, max(Ps))):
            s = orc.ba_error_sums(X[p:p + 1], mode=1, strict=True, nthreads=os.cpu_count())[0]
            orc.associate(X[p], strict=True)
            lo = orc.linearize(X[p:p + 1], nthreads=os.cpu_count())
            g = rec[p]
            exact &= bool(np.array_equal(g[3:12], s[0, 3:12]) and np.array_equal(g[12 + 57:], lo[0, 57:]))
            errs = max(errs, float(abs(g[12] - lo[0, 0]) / abs(lo[0, 0])),
                       float(np.abs(g[13:20] - lo[0, 1:8]).max() / np.abs(lo[0, 1:8]).max()),
                       float(np.abs(g[20:69] - lo[0, 8:57]).max() / np.abs(lo[0, 8:57]).max()))
        out["oracle_check"] = dict(starts=min(args.oracle_sample, max(Ps)), counters_exact=exact, max_rel_err=errs, ok=bool(exact and errs < 1e-6))
        ok_all &= out["oracle_check"]["ok"]
        log("oracle:", out["oracle_check"])
    out["ok"] = bool(ok_all)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))
    ctx.close()
    return 0 if ok_all else 3


if __name__ == "__main__":
    sys.exit(main())
