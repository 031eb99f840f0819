#!/usr/bin/env python3
"""Keyframe selection on ONE GPU: a context holding the whole pack that selects S (stl_select_keyframes) against a context
holding only pack.select(S), on the same calls.

Workload: the KITTI-00 shape of bench.py (config c2: 1500 synthetic keyframes, 64 beams x 1875 azimuth steps, k = 30, generator
seed 1000); candidates synth.candidates(x_gt, 257, 0.2, seed = 42)[1:] (bench.py's candidate stream).  Selections: none (the
whole pack), every 2nd, every 8th, a contiguous 188, every 32nd and a single keyframe.  For every selection it times,
interleaved over --rounds rounds (the spread is over those rounds), each with --warmup untimed calls first:
  step  stl_step_batch_device(X[0], B = 1, reassociate = 1)       one LM iteration
  eval  stl_eval_batch_device(X[:256])                            one 256-candidate NOMAD poll
on the selecting context and on the sliced one.  The _device calls are enqueued back to back on one stream and timed with CUDA
events around --iters of them.  Every timed record is compared with the sliced context's, bit for bit.  Writes JSON (GPU name
and power limit read in the same run) to --out."""
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


def timed(torch, stream, f, n):
    """CUDA events on `stream` around n back-to-back enqueues of f (the _device calls): device ms per call"""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(n):
        f()
    b.record(stream)
    b.synchronize()
    return a.elapsed_time(b) / n


def selections(F):
    return {"none": None, "every_2nd": list(range(0, F, 2)), "every_8th": list(range(0, F, 8)),
            "contiguous_188": list(range(F // 2, F // 2 + 188)), "every_32nd": list(range(0, F, 32)), "single": [F // 2]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nkf", type=int, default=1500)
    ap.add_argument("--B", type=int, default=256, help="candidates of the timed evaluation")
    ap.add_argument("--iters", type=int, default=10, help="timed calls per round")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seed", type=int, default=1000)
    ap.add_argument("--only", default="", help="comma-separated subset of the selections")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_keyframe_select.json"))
    args = ap.parse_args()
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
    X = synth.candidates(x_gt, args.B + 1, 0.2, seed=42)[1:]
    params = pkg.default_params()
    full = capi.Context(params=params)
    full.upload(pack)
    out = dict(what=__doc__.split("\n")[0], gpu=card, keyframes=args.nkf, seed=args.seed, B=args.B, iters=args.iters, rounds=args.rounds,
               warmup=args.warmup, clock="CUDA events on the calls' stream around --iters back-to-back _device calls", results=[])
    stream = torch.cuda.Stream()
    sp = stream.cuda_stream
    d_step = torch.empty((2, 74), dtype=torch.float64, device="cuda")
    d_eval = torch.empty((2, args.B, 12), dtype=torch.float64, device="cuda")
    ok_all = True
    sels = selections(args.nkf)
    if args.only:
        sels = {k: v for k, v in sels.items() if k in args.only.split(",")}
    for name, S in sels.items():
        full.select_keyframes(S)
        if S is None:
            sliced, n_sel = full, args.nkf
        else:
            t0 = time.perf_counter()
            sliced = capi.Context(params=params)
            sliced.upload(pack.select(S))
            n_sel = len(S)
            log(f"{name}: {n_sel} keyframes, sliced pack uploaded in {time.perf_counter() - t0:.2f}s")
        ctxs = (full, sliced)
        calls = {
            "step": [lambda c=c, i=i: c.step_device(X[:1], d_step[i].data_ptr(), stream_ptr=sp, reassociate=True) for i, c in enumerate(ctxs)],
            "eval": [lambda c=c, i=i: c.eval_sums_device(X, d_eval[i].data_ptr(), stream_ptr=sp) for i, c in enumerate(ctxs)],
        }
        res = dict(selection=name, keyframes=n_sel)
        for what, (f_sel, f_sliced) in calls.items():
            ts, tw = [], []
            same = True
            for _ in range(args.rounds):
                for f, acc in ((f_sel, ts), (f_sliced, tw)):
                    for _ in range(args.warmup):
                        f()
                    acc.append(timed(torch, stream, f, args.iters))
                stream.synchronize()
                d = d_step if what == "step" else d_eval
                same &= bool(torch.equal(d[0], d[1]))
            ok_all &= same

            def st(v):
                v = np.asarray(v)
                return dict(median=float(np.median(v)), min=float(v.min()), max=float(v.max()))
            res[what] = dict(selected_ms=st(ts), sliced_ms=st(tw), ratio=float(np.median(ts) / np.median(tw)), bitwise_equal=same)
        out["results"].append(res)
        log(json.dumps(res))
        if sliced is not full:
            sliced.close()
    full.close()
    out["ok"] = bool(ok_all)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))
    return 0 if ok_all else 3


if __name__ == "__main__":
    sys.exit(main())
