#!/usr/bin/env python3
"""Oversize keyframes on ONE GPU: what stl_allow_oversize_keyframes costs on a pack that fits, what the banded three-kernel K1
costs per keyframe where both K1 forms can run, and what packs the one-kernel K1 cannot hold take.

Workloads (synthetic, 64 beams x 1875 azimuth steps per scan, k = 30, generator seed 1000, candidates
synth.candidates(x_gt, 257, 0.2, seed = 42)[1:] as in bench.py):
  kitti   the KITTI-00 shape of bench.py (config c2: 1500 keyframes of 1241 x 376, 2000 keypoints), on three contexts:
          flag off, flag on (no keyframe is oversize: the same launches), and STL_K1_OVERSIZE=all (every keyframe on the
          banded K1).  Every timed record of the last two is compared with the first, bit for bit.
  4k      --nkf-big keyframes of 3840 x 2160 with 2000 keypoints (17 bands each), flag on
  12k     --nkf-big keyframes of 1241 x 376 with 12000 keypoints, flag on
For every context it times, interleaved over --rounds rounds (the spread is over those rounds), each with --warmup untimed
calls first:
  step  stl_step_batch_device(X[0], B = 1, reassociate = 1)       one LM iteration
  eval  stl_eval_batch_device(X[:256])                            one 256-candidate NOMAD poll
The _device calls are enqueued back to back on one stream and timed with CUDA events around --iters of them.  Work counter
[6] (units whose survivors overflowed into the exact pass over every point) is reported after the evaluations.  Writes JSON
(GPU name and power limit read in the same run) to --out."""
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


def stats(v):
    v = np.asarray(v)
    return dict(median=float(np.median(v)), min=float(v.min()), max=float(v.max()))


def context(capi, params, pack, allow, route_all=False):
    os.environ.pop("STL_K1_OVERSIZE", None)
    if route_all:
        os.environ["STL_K1_OVERSIZE"] = "all"  # read at upload
    c = capi.Context(params=params)
    c.allow_oversize_keyframes(allow)
    t0 = time.perf_counter()
    c.upload(pack)
    os.environ.pop("STL_K1_OVERSIZE", None)
    return c, time.perf_counter() - t0


def measure(torch, args, ctxs, X, names):
    """Interleaved rounds of step and eval over the contexts; records of contexts 1.. compared with context 0's."""
    stream = torch.cuda.Stream()
    sp = stream.cuda_stream
    n = len(ctxs)
    d_step = torch.empty((n, 74), dtype=torch.float64, device="cuda")
    d_eval = torch.empty((n, args.B, 12), dtype=torch.float64, device="cuda")
    calls = {
        "step": [lambda c=c, i=i: c.step_device(X[:1], d_step[i].data_ptr(), stream_ptr=sp, reassociate=True) for i, c in enumerate(ctxs)],
        "eval": [lambda c=c, i=i: c.eval_sums_device(X, d_eval[i].data_ptr(), stream_ptr=sp) for i, c in enumerate(ctxs)],
    }
    res = {}
    for what, fs in calls.items():
        t = [[] for _ in fs]
        same = [True] * n
        for _ in range(args.rounds):
            for i, f in enumerate(fs):
                for _ in range(args.warmup):
                    f()
                t[i].append(timed(torch, stream, f, args.iters))
            stream.synchronize()
            d = d_step if what == "step" else d_eval
            for i in range(1, n):
                same[i] &= bool(torch.equal(d[0], d[i]))
        res[what] = {names[i]: dict(ms=stats(t[i]), **({"bitwise_equal_to_" + names[0]: same[i]} if i else {})) for i in range(n)}
        for i in range(1, n):
            res[what][names[i]]["ratio_to_" + names[0]] = float(np.median(t[i]) / np.median(t[0]))
    for i, c in enumerate(ctxs):
        c.eval_sums(X)  # the work counters of one evaluation
        w = c.work_counters()
        res.setdefault("counters", {})[names[i]] = dict(k1_overflow_units=float(w["k1_overflow_units"]),
                                                        oversize_keyframes=int(len(c.oversize_keyframes())))
    ok = all(v.get("bitwise_equal_to_" + names[0], True) for what in ("step", "eval") for v in res[what].values())
    return res, ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nkf", type=int, default=1500, help="keyframes of the KITTI-00-shaped pack")
    ap.add_argument("--nkf-big", type=int, default=188, help="keyframes of the 4K and 12k-keypoint packs")
    ap.add_argument("--B", type=int, default=256, help="candidates of the timed evaluation")
    ap.add_argument("--iters", type=int, default=10, help="timed calls per round")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seed", type=int, default=1000)
    ap.add_argument("--only", default="", help="comma-separated subset of kitti,4k,12k")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_oversize_keyframes.json"))
    args = ap.parse_args()
    import torch  # before the library: its NCCL must be the one torch resolves
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU")
    pkg = importlib.import_module(PKG)
    synth = importlib.import_module(PKG + ".synth")
    capi = importlib.import_module(PKG + ".capi")
    card = gpu_info()
    log("card:", card)
    params = pkg.default_params()
    out = dict(what=__doc__.split("\n")[0], gpu=card, seed=args.seed, B=args.B, iters=args.iters, rounds=args.rounds, warmup=args.warmup,
               clock="CUDA events on the calls' stream around --iters back-to-back _device calls", results={})
    only = set(args.only.split(",")) if args.only else {"kitti", "4k", "12k"}
    ok_all = True
    if "kitti" in only:
        t0 = time.perf_counter()
        pack, x_gt, _ = synth.generate(n_kf=args.nkf, beams=64, az_steps=1875, seed=args.seed)
        log(f"kitti pack: {args.nkf} keyframes in {time.perf_counter() - t0:.1f}s")
        X = synth.candidates(x_gt, args.B + 1, 0.2, seed=42)[1:]
        ctxs, up = [], {}
        for name, allow, ra in (("flag_off", False, False), ("flag_on", True, False), ("route_all", True, True)):
            c, t = context(capi, params, pack, allow, ra)
            ctxs.append(c)
            up[name] = t
        res, ok = measure(torch, args, ctxs, X, ["flag_off", "flag_on", "route_all"])
        res.update(keyframes=args.nkf, image="1241x376", keypoints=2000, upload_s=up)
        out["results"]["kitti"] = res
        ok_all &= ok
        log(json.dumps(res))
        for c in ctxs:
            c.close()
        del pack
    for name, W, H, nkp in (("4k", 3840, 2160, 2000), ("12k", 1241, 376, 12000)):
        if name not in only:
            continue
        t0 = time.perf_counter()
        f = 718.856 * max(W, H) / 1241  # KITTI-00's focal length scaled to the longer side (as the GPU tests' packs)
        cam = dict(fx=718.856, fy=718.856, cx=607.1928, cy=185.2157) if W == 1241 else dict(fx=f, fy=f, cx=W / 2 - 0.35, cy=H / 2 + 0.15)
        pack, x_gt, _ = synth.generate(n_kf=args.nkf_big, beams=64, az_steps=1875, seed=args.seed, width=W, height=H, n_kp=nkp, **cam)
        log(f"{name} pack: {args.nkf_big} keyframes in {time.perf_counter() - t0:.1f}s")
        X = synth.candidates(x_gt, args.B + 1, 0.2, seed=42)[1:]
        c, t = context(capi, params, pack, True)
        res, _ = measure(torch, args, [c], X, ["flag_on"])
        res.update(keyframes=args.nkf_big, image=f"{W}x{H}", keypoints=nkp, upload_s=t)
        out["results"][name] = res
        log(json.dumps(res))
        c.close()
        del pack
    out["ok"] = bool(ok_all)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))
    return 0 if ok_all else 3


if __name__ == "__main__":
    sys.exit(main())
