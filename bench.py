#!/usr/bin/env python
"""bench.py — extrinsic cost evaluations / s at KITTI-00 shape (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config c1|c2|c3|c4|c5] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

BASELINE.json configs -> `--config` (default c2, the one the metric is quoted on):
  c1  50 keyframes, 1 candidate / step:   BAError cost                          (stl_eval_batch)
  c2  1500 keyframes, 1 candidate / step: BAError cost + BuildProblem at x + cost / J^T r / 7x7 J^T J
                                          (one LM / g2o iteration, stl_step_batch with reassociate)
  c3  as c2 with k = 20 neighbours for the local-plane PCA (>= 150 k map-point queries per evaluation)
  c4  1500 keyframes, 256 candidates / step (a NOMAD MADS poll): BAError sums + cost / J^T J of every
      candidate on the frozen association (stl_step_batch without reassociate)
  c5  4000 keyframes, 128-beam ~250 k-point scans, GPR depth factor enabled, step as c2
`value`  : evaluations / s with the pack resident in HBM, results left on the device, timed with CUDA
           events on the launching stream (max over ranks).
`e2e`    : the same step through the host-facing C-ABI call (host x in, host record out; H2D / D2H
           copies and the synchronisation inside the timed region).
N > 1    : one process per GPU; keyframes are sharded over the ranks and every call ends with ONE NCCL
           fp64 all-reduce of the [B,74] record, issued by the library on its compute stream
           (stl_comm_init) — the north-star layout, strong scaling.  `--shard candidates` keeps the
           round-1 replica layout (every rank holds the whole pack and evaluates its own candidates).
The CPU arm (`cpu_baseline`, and the whole `--impl reference` arm) is the oracle — the reference's
vendored nanoflann (oracle/_ref) when built, else the in-repo port — on all host cores: OpenMP over
keyframes for BAError and BuildProblem (iba_func.cpp:203, iba_local.cpp:162) and over residual blocks
for the linearisation (ceres num_threads, iba_local.cpp:439), on the SAME workload, unextrapolated for
c1-c3 and on a stated bounded sample for c4 / c5.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
PKG = "spatial-temporal-lidar-camera-calibration_b200"
METRIC = "extrinsic_cost_evals_per_s"
UNIT = "evals/s"

# workload definitions (BASELINE.json configs[0..4]); `mode`: what one step computes
CONFIGS = {
    "c1": dict(nkf=50, beams=64, az=1875, B=1, k=30, gpr=0, mode="eval",
               what="BAError cost (BASELINE configs[0])"),
    "c2": dict(nkf=1500, beams=64, az=1875, B=1, k=30, gpr=0, mode="step",
               what="BAError cost + association + cost/JtJ (BASELINE configs[1])"),
    "c3": dict(nkf=1500, beams=64, az=1875, B=1, k=20, gpr=0, mode="step",
               what="k=20 local-plane variant: BAError cost + association + cost/JtJ (BASELINE configs[2])"),
    "c4": dict(nkf=1500, beams=64, az=1875, B=256, k=30, gpr=0, mode="poll",
               what="NOMAD poll batch: BAError sums + cost/JtJ of 256 candidates on the frozen association (BASELINE configs[3])"),
    "c5": dict(nkf=4000, beams=128, az=2048, B=1, k=30, gpr=1, mode="step",
               what="GPR depth-factor variant on 128-beam scans: BAError cost + association + cost/JtJ (BASELINE configs[4])"),
}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--nkf", type=int, default=0, help="override the keyframe count of the config (diagnostics)")
    ap.add_argument("--shard", default="keyframes", choices=["candidates", "keyframes"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the side measurements (poll batch, per-query plane fit)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--seed", type=int, default=1000)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy (rank 0's record; with "
                         "--shard candidates that covers only rank 0's candidates)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


def dump_outputs(d, eval_sums, lin_sums):
    """The record of the last timed step as float64 arrays: DIR/eval_sums.npy, the [B,12] BAError sums
    (stl_eval_sums_t), and DIR/lin_sums.npy, the [B,62] cost / J^T r / J^T J (stl_lin_sums_t) when the step
    linearises.  The inputs follow from the arguments alone (seeded generator and candidates), so two builds run
    with the same arguments can be compared array for array.  Rank 0 writes its record: with keyframes sharded that is
    the whole step, with `--shard candidates` only rank 0's B candidates."""
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "eval_sums.npy"), np.ascontiguousarray(eval_sums, dtype=np.float64))
    if lin_sums is not None:
        np.save(os.path.join(d, "lin_sums.npy"), np.ascontiguousarray(lin_sums, dtype=np.float64))


def workload_config(args):
    """The `config` object — identical, byte for byte, in both arms (it only names the workload)."""
    c = CONFIGS[args.config]
    F = args.nkf or c["nkf"]
    pts = c["beams"] * c["az"]
    return {
        "workload": f"{args.config}: {F} keyframes x ~{pts // 1000}k-ray {c['beams']}-beam scans x 2000 keypoints, "
                    f"{c['B']} candidate(s)/step: {c['what']}",
        "config_id": args.config, "keyframes": F, "beams": c["beams"], "rays_per_scan": pts, "keypoints_per_keyframe": 2000,
        "candidates_per_step": c["B"], "knn_k": c["k"], "gpr_factor": bool(c["gpr"]), "step": c["mode"], "seed": args.seed,
        "l2_policy": f"inputs larger than L2 (~{12e-9 * pts * 0.976 * F:.2f} GB of scans streamed per candidate)",
    }


def make_params(pkgmod, args):
    c = CONFIGS[args.config]
    p = pkgmod.default_params()
    p.norm_max_pts = c["k"]
    p.use_gpr = c["gpr"]
    return p


def gen_kwargs(args):
    c = CONFIGS[args.config]
    kw = dict(beams=c["beams"], az_steps=c["az"], seed=args.seed)
    if c["beams"] == 128:
        kw.update(elev_top_deg=15.0, elev_bottom_deg=-25.0)
    return kw


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md recipe).  NVML is polled
    from a thread every 2 ms (the timed region is ~0.1 s, too short for `nvidia-smi -lms`); nvidia-smi
    is the fallback when the NVML binding is missing."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []
        self.nvml, self.h, self.stop_flag, self.sm, self.mask = None, None, False, [], 0
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self.nvml = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
                self.mask |= int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nvml is not None:
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.t.join(timeout=1.0)
            try:
                mx = float(self.nvml.nvmlDeviceGetMaxClockInfo(self.h, self.nvml.NVML_CLOCK_SM))
            except Exception:
                mx = None
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": mx,
                    "reasons": sorted(v for b, v in self.BITS.items() if self.mask & b), "samples": len(self.sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


# ------------------------------------------------------------------------------------------------ CPU arm
class CpuArm:
    """The reference's CPU path for one workload: the oracle on all host cores."""

    def __init__(self, pack, params, mode, cores):
        from oracle import oracle as O
        self.kind = "ref" if O.have_ref() else "port"
        self.cores = cores
        self.mode = mode
        self.orc = O.Oracle(pack, params=params, kind=self.kind, nthreads=cores)
        self.build_s = self.orc.build_seconds
        self.frozen = False

    def freeze(self, x0):
        self.orc.associate(x0, strict=True)
        self.frozen = True

    def step(self, X):
        """One step on candidates X [B,7]; returns ([B,12] sums, [B,62] linearisation or None)."""
        o, n = self.orc, self.cores
        X = np.atleast_2d(X)
        if self.mode == "eval":
            return o.ba_error_sums(X, mode=1, strict=True, nthreads=n)[0], None
        if self.mode == "step":     # BAError (OpenMP over keyframes, iba_func.cpp:203) + BuildProblem + Evaluate (ceres threads)
            s = o.ba_error_sums(X, mode=1, strict=True, nthreads=n)[0]
            o.associate(X[0], strict=True)
            return s, o.linearize(X, nthreads=n)
        # poll: candidates in parallel, each serial over keyframes (NOMAD evaluation threads, iba_global.cpp:385)
        s = o.ba_error_sums(X, mode=2, strict=True, nthreads=n)[0]
        return s, o.linearize(X, nthreads=n)

    def describe(self):
        return "reference nanoflann v1.5.0 (oracle/_ref)" if self.kind == "ref" else "in-repo nanoflann port"


def run_reference(args, rank):
    """--impl reference: the reference's CPU path on the host cores, same workload, same config object."""
    if rank != 0:
        return
    pkgmod = importlib.import_module(PKG)
    synth = importlib.import_module(PKG + ".synth")
    c = CONFIGS[args.config]
    F = args.nkf or c["nkf"]
    cores = os.cpu_count() or 1
    # bounded sample: c1-c3 run the whole workload; c4 a slice of the poll batch; c5 a slice of the keyframes
    nkf_s = F if args.config != "c5" else min(F, 384)
    B_s = c["B"] if args.config != "c4" else min(c["B"], max(cores, 8))
    pack, x_gt, _ = synth.generate(n_kf=nkf_s, n_kf_total=F, **gen_kwargs(args))
    nsteps = args.steps + args.warmup
    Xall = synth.candidates(x_gt, nsteps * c["B"] + 1, 0.2, seed=42)[1:]
    arm = CpuArm(pack, make_params(pkgmod, args), c["mode"], cores)
    if c["mode"] == "poll":
        arm.freeze(Xall[0])

    def cands(i):
        return Xall[i * c["B"]: i * c["B"] + B_s]
    for i in range(args.warmup):
        arm.step(cands(i))
    t0 = time.perf_counter()
    for i in range(args.steps):
        last = arm.step(cands(args.warmup + i))
    dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *last)
    frac = (nkf_s / F) * (B_s / c["B"])          # share of one step's work the sample covers
    val = c["B"] * frac / dt
    sample = (f"{nkf_s} of {F} keyframes x {B_s} of {c['B']} candidates per step"
              + (" (the whole workload, no extrapolation)" if frac == 1.0 else f" (extrapolated linearly, x{1 / frac:.1f})")
              + f"; {cores} threads: OpenMP over keyframes (BAError, BuildProblem), over residual blocks (linearisation); KNN = {arm.describe()}; "
              f"one-off KD-tree build {arm.build_s:.2f}s excluded")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3 / frac, "higher_is_better": True, "scaling": "strong" if args.shard == "keyframes" else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(args),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "reference" if arm.kind == "ref" else "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    ncpu = os.cpu_count() or 8
    if args.impl == "reference":
        # torchrun exports OMP_NUM_THREADS=1; the CPU arm is entitled to every host core (rank 0 runs alone)
        os.environ["OMP_NUM_THREADS"] = str(ncpu)
        run_reference(args, rank)
        return
    os.environ["OMP_NUM_THREADS"] = str(max(1, ncpu // max(world, 1)))  # host-side generator / pack preparation only

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the cost-evaluation path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    pkgmod = importlib.import_module(PKG)
    synth = importlib.import_module(PKG + ".synth")
    capi = importlib.import_module(PKG + ".capi")
    par = importlib.import_module(PKG + ".parallel")
    _abi = importlib.import_module(PKG + "._abi")

    cfg = CONFIGS[args.config]
    F = args.nkf or cfg["nkf"]
    B = cfg["B"]
    mode = cfg["mode"]
    by_kf = world > 1 and args.shard == "keyframes"
    params = make_params(pkgmod, args)
    t0 = time.time()
    if by_kf:
        kb, ke = par.shard_bounds(F, world, rank)
        pack, x_gt, _ = synth.generate(n_kf=ke - kb, kf_begin=kb, n_kf_total=F, **gen_kwargs(args))
    else:
        pack, x_gt, _ = synth.generate(n_kf=F, **gen_kwargs(args))
    t_gen = time.time() - t0
    nsteps = args.steps + args.warmup
    # every step gets its own candidates; row 0 of the list is the ground truth and is not used
    if by_kf or world == 1:
        Xall = synth.candidates(x_gt, nsteps * B + 1, 0.2, seed=42)[1:]
        units_per_step = B

        def cands(i):
            return Xall[i * B: (i + 1) * B]
    else:   # replicas: every rank draws its own candidates
        Xall = synth.candidates(x_gt, nsteps * B * world + 1, 0.2, seed=42)[1:]
        units_per_step = B * world

        def cands(i):
            return Xall[(i * world + rank) * B: (i * world + rank + 1) * B]

    ctx = capi.Context(params=params, device=local_rank)
    if by_kf:   # the library owns the communicator; torch.distributed only carries the 128-byte id
        par.attach_communicator(ctx, rank, world, exchange=par.torch_exchange())
    # a few keyframes first: loads the CUDA modules of the build (lazy loading would otherwise be timed as "K0")
    ctx.upload(pack.shard(0, min(4, pack.n_kf)))
    ctx.stage_stats()
    free0 = torch.cuda.mem_get_info()[0]
    t0 = time.time()
    ctx.upload(pack)
    torch.cuda.synchronize()
    t_upload = time.time() - t0
    st0 = ctx.stage_stats()
    build_ms, pidx_ms = st0["build"][0], st0["plane_index"][0]
    # a stream of our own: the handle of torch's default stream is 0, which the C-ABI reads as "the context's own
    # stream" — events recorded on the legacy default stream would then not be ordered with the library's work
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    ctx.set_stream(stream.cuda_stream)
    W = _abi.STL_STEP_NSUMS if mode != "eval" else _abi.STL_EVAL_NSUMS
    d_out = torch.zeros((max(args.steps, 1), B, W), dtype=torch.float64, device=dev)   # one record row per timed step
    d_tmp = torch.zeros((B, W), dtype=torch.float64, device=dev)

    def step_device(X, out):
        if mode == "eval":
            ctx.eval_sums_device(X, out.data_ptr(), stream.cuda_stream)
        else:
            ctx.step_device(X, out.data_ptr(), stream.cuda_stream, reassociate=(mode == "step"))

    def step_host(X):
        if mode == "eval":
            return ctx.eval_sums(X)
        return ctx.step(X, reassociate=(mode == "step"))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if mode == "poll":
        ctx.associate(cands(0)[0])            # BuildProblem once at the poll centre; the polls below keep it frozen
    for i in range(args.warmup):
        step_device(cands(i), d_tmp)
    barrier()
    mem_used = free0 - torch.cuda.mem_get_info()[0]
    launches0 = ctx.work_counters()["launches"]
    ctx.set_profiling(True)
    ctx.stage_stats()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for i in range(args.steps):
        step_device(cands(args.warmup + i), d_out[i])
    ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop()
    stats = ctx.stage_stats()
    ctx.set_profiling(False)
    wc = ctx.work_counters()
    exch = ctx.comm_stats() if (by_kf and world > 1) else {}
    launches = int(wc["launches"] - launches0)
    rec = d_out.cpu().numpy()                  # [steps, B, W]
    if args.dump_outputs and rank == 0:
        E = _abi.STL_EVAL_NSUMS
        dump_outputs(args.dump_outputs, rec[args.steps - 1][:, :E], rec[args.steps - 1][:, E:] if mode != "eval" else None)

    # ---- end to end through the host-facing C-ABI (host buffers in and out)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        r_host = step_host(cands(args.warmup + i))
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert np.array_equal(r_host, rec[args.steps - 1]), "host-facing call and device-resident call disagree"

    # ---- side measurements (single configuration each, device-timed, reported beside `value`, never as it)
    extras = {}
    if not args.no_extras and args.config == "c2":
        # (a) BASELINE configs[3] shape on this layout: one 256-candidate poll on the frozen association
        Xp = synth.candidates(x_gt, 257, 0.2, seed=43)[1:]
        Xp = Xp if (by_kf or world == 1) else Xp[rank::world]
        d_p = torch.zeros((len(Xp), _abi.STL_STEP_NSUMS), dtype=torch.float64, device=dev)
        ctx.associate(Xp[0])
        ctx.step_device(Xp, d_p.data_ptr(), stream.cuda_stream, reassociate=False)   # untimed: sizes the batch buffers
        barrier()
        ctx.set_profiling(True); ctx.stage_stats()
        q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        q0.record(stream)
        for _ in range(2):
            ctx.step_device(Xp, d_p.data_ptr(), stream.cuda_stream, reassociate=False)
        q1.record(stream)
        barrier()
        pst = ctx.stage_stats(); ctx.set_profiling(False)
        extras["poll_ms"] = q0.elapsed_time(q1) / 2
        extras["poll_stage_ms"] = {k: round(v[0] / 2, 3) for k, v in pst.items() if v[1]}
        # (b) the same step with the plane fitted per query at evaluation time (the reference's order of work)
        ctx.close()
        p0 = make_params(pkgmod, args)
        p0.plane_index = 0
        ctx = capi.Context(params=p0, device=local_rank)
        if by_kf:
            par.attach_communicator(ctx, rank, world, exchange=par.torch_exchange())
        t0 = time.time()
        ctx.upload(pack)
        torch.cuda.synchronize()
        extras["fit_upload_s"] = time.time() - t0
        ctx.set_stream(stream.cuda_stream)
        for i in range(args.warmup):
            step_device(cands(i), d_tmp)
        barrier()
        p0e, p1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0e.record(stream)
        for i in range(args.steps):
            step_device(cands(args.warmup + i), d_tmp)
        p1e.record(stream)
        barrier()
        extras["fit_ms"] = p0e.elapsed_time(p1e)
        extras["fit_same"] = bool(np.array_equal(d_tmp.cpu().numpy(), rec[args.steps - 1]))

    tmax = torch.tensor([ms, e2e_s * 1e3, extras.get("poll_ms", 0.0), extras.get("fit_ms", 0.0)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_max, e2e_ms_max, poll_ms_max, fit_ms_max = (float(v) for v in tmax)
    value = units_per_step * args.steps / (ms_max * 1e-3)
    e2e_value = units_per_step * args.steps / (e2e_ms_max * 1e-3)

    rc = 0
    if rank == 0:
        peak, peak_src = peaks()
        k1_ms, k1_n = stats["assoc2d"]
        k1_avg = k1_ms / max(k1_n, 1)
        n_pts, n_kp = pack.n_points, pack.n_keypoints
        # algorithmic bytes of one K1 launch = one chunk of `per_launch` candidates over this rank's keyframes: the
        # scan is read once per chunk (12 B / point; candidates 2.. of the chunk are served by L2), keypoints in
        # and correspondences out per candidate (16 B / keypoint)
        launches_per_step = max(1, round(k1_n / max(args.steps, 1)))
        per_launch = B / launches_per_step
        k1_bytes = 12.0 * n_pts + 16.0 * n_kp * per_launch
        achieved = k1_bytes / (k1_avg * 1e-3) / 1e9 if k1_avg > 0 else 0.0
        tot_stage = sum(v[0] for k, v in stats.items() if k not in ("build", "plane_index"))
        share = {k: round(v[0] / tot_stage, 4) for k, v in stats.items() if v[1] and k not in ("build", "plane_index")}
        k2_ms, k2_n = stats["knn3d"]
        last = rec[args.steps - 1]
        q3 = float(last[:, 6].mean())                # 3-D queries of one candidate (all keyframes: the record is all-reduced)
        knn_q_eval = 2000.0 * F + 2.0 * q3           # findNeighbors calls of one BAError (iba_global.cpp:92,120,129)
        x_bytes = 56 * B
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "strong" if (by_kf or world == 1) else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args),
            "layout": {
                "sharding": (("keyframes sharded over the ranks + ONE fp64 sum of the [B,%d] record per step, issued by the library: " % W) +
                             ("inside the finishing kernel over NVLink peer memory (cudaIpc)" if exch.get("p2p") else "ncclAllReduce on the compute stream")
                             if by_kf else ("candidates (pack replicated per GPU, no collective)" if world > 1 else "single GPU")),
                "keyframes_this_rank": int(pack.n_kf), "points_this_rank": int(n_pts), "keypoints_this_rank": int(n_kp),
                "plane_index": bool(params.plane_index), "candidates_per_step_all_ranks": units_per_step,
                "exchange": exch,
            },
            "setup": {"upload_s": round(t_upload, 3), "k0_index_build_device_ms": round(build_ms, 1), "plane_index_build_ms": round(pidx_ms, 1),
                      "synth_s": round(t_gen, 2), "hbm_bytes_resident": int(mem_used)},
            # per step: candidates in (x, 56 B each; the library stages them as 208-B + 1608-B prepared records), record out
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": (208 + (1608 if mode != "eval" else 0)) * B,
                    "d2h_bytes_per_step": 8 * W * B, "x_bytes_per_step": x_bytes},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": {
                "kernel": "k_assoc2d (K1: transform + project + 2-D association)", "bound": "hbm", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": k1_bytes, "avg_launch_ms": k1_avg, "launches": k1_n,
                "candidates_per_launch": per_launch,
            },
            "roofline_k0": {
                "kernel": "K0 index build (k_bbox, k_morton, radix sort, k_scatter, k_kd_refine, AABBs, k_leaf_adj), once per pack",
                "bound": "hbm", "algorithmic_bytes": 28.0 * n_pts, "device_ms": build_ms,
                "achieved": (28.0 * n_pts / (build_ms * 1e-3) / 1e9) if build_ms > 0 else None, "peak": peak, "unit": "GB/s",
                "frac": (28.0 * n_pts / (build_ms * 1e-3) / 1e9 / peak) if build_ms > 0 else None,
                "note": "12 B read + 16 B written per point; dominated by the shared-memory KD refinement (bitonic networks), not by HBM",
            },
            "stage_share": share,
            "stage_note": "device time per stage from CUDA events on the stream each stage runs on; in the step the association chain (assoc_lm, linearize) runs on a second stream beside knn3d / reduce, so the stages overlap and do not add up to ms_per_step (STL_NO_OVERLAP=1 serialises them)",
            "stage_ms_per_launch": {k: round(v[0] / v[1], 4) for k, v in stats.items() if v[1] and k not in ("build", "plane_index")},
            "knn": {"queries_per_eval": knn_q_eval, "queries_per_s_whole_step": knn_q_eval * value,
                    "k2_pairs_per_s": (q3 * B / (world if by_kf else 1) / (k2_ms / max(k2_n, 1) * 1e-3)) if k2_ms > 0 else None},
            "k1_point_transforms_per_s": (float(n_pts) * per_launch / (k1_avg * 1e-3)) if k1_avg > 0 else None,
            "assoc_reused": wc["assoc_reused"],
            "result_check": {"f_sums": [float(last[0, 0]), float(last[0, 1])], "frames_kept": float(last[0, 10]),
                             "lm_cost": float(last[0, 12]) if mode != "eval" else None},
        }
        if "poll_ms" in extras:
            line["poll_batch"] = {
                "candidates": 256, "ms": poll_ms_max, "evals_per_s": 256 / (poll_ms_max * 1e-3), "unit": UNIT, "stage_ms": extras["poll_stage_ms"],
                "k1_point_transforms_per_s": 256.0 * n_pts / (extras["poll_stage_ms"].get("assoc2d", float("nan")) * 1e-3),
                "note": "BASELINE configs[3] shape (bench.py --config c4 is the full run): one stl_step_batch over 256 candidates on the frozen "
                        "association; device-timed mean of 2 polls after one untimed poll, max over ranks"}
        if "fit_ms" in extras:
            line["plane_fit_per_query"] = {
                "value": units_per_step * args.steps / (fit_ms_max * 1e-3), "unit": UNIT, "ms_per_step": fit_ms_max / args.steps,
                "upload_s": round(extras["fit_upload_s"], 3), "identical_record": extras["fit_same"],
                "note": "params.plane_index=0: the local plane is fitted per query inside every evaluation (the reference's order of work) "
                        "instead of being looked up in the index built at upload; same record bit for bit"}
        # the ncu traffic figure of K1 (a static capture: DRAM counters cannot be read in-run)
        tp = os.path.join(ROOT, "profiles", "k1_traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                line["roofline"]["traffic"] = tj["dram_bytes_per_launch"] * (pack.n_kf / float(tj.get("keyframes", pack.n_kf))) if per_launch == 1 else None
                line["roofline"]["traffic_source"] = "static: " + tj.get("source", "profiles/k1_traffic.json") + " (ncu --set full, scaled to this launch's units)"
            except Exception:
                pass
        if world == 1 and not args.no_cpu_baseline:
            # The reference's CPU path on this box's host cores, on a bounded sample of the SAME candidates — and the
            # parity check of the timed GPU records against it (counters exact, sums 1e-9, normal equations 1e-6).
            cores = ncpu
            nkf_s = F if args.config not in ("c5",) else min(F, 256)
            B_s = B if mode != "poll" else min(B, max(cores, 8))
            cpack = pack if nkf_s == F else pack.shard(0, nkf_s)
            arm = CpuArm(cpack, params, mode, cores)
            if mode == "poll":
                arm.freeze(cands(0)[0])
            t_tot, reps, ok, checked = 0.0, 0, True, 0
            errs = {"sum_3d2d": 0.0, "sum_3d3d": 0.0, "sum_he": 0.0, "lm_cost": 0.0, "lm_JtR": 0.0, "lm_JtJ": 0.0}
            while reps < args.steps and (t_tot < args.cpu_seconds or reps < 2):
                Xs = cands(args.warmup + reps)[:B_s]
                t0 = time.perf_counter()
                s_cpu, l_cpu = arm.step(Xs)
                t_tot += time.perf_counter() - t0
                if nkf_s == F:          # full keyframe set: the GPU record of this very step must match
                    g = rec[reps][:B_s]
                    ok &= bool(np.array_equal(g[:, 3:12], s_cpu[:, 3:12]))
                    for j, name in enumerate(("sum_3d2d", "sum_3d3d", "sum_he")):
                        den = np.maximum(np.abs(s_cpu[:, j]), 1e-300)
                        errs[name] = max(errs[name], float((np.abs(g[:, j] - s_cpu[:, j]) / den).max()))
                    if l_cpu is not None:
                        gl = g[:, 12:]
                        ok &= bool(np.array_equal(gl[:, 57:], l_cpu[:, 57:]))
                        errs["lm_cost"] = max(errs["lm_cost"], float((np.abs(gl[:, 0] - l_cpu[:, 0]) / np.abs(l_cpu[:, 0])).max()))
                        sg = np.abs(l_cpu[:, 1:8]).max(axis=1, keepdims=True)
                        sh = np.abs(l_cpu[:, 8:57]).max(axis=1, keepdims=True)
                        errs["lm_JtR"] = max(errs["lm_JtR"], float((np.abs(gl[:, 1:8] - l_cpu[:, 1:8]) / sg).max()))
                        errs["lm_JtJ"] = max(errs["lm_JtJ"], float((np.abs(gl[:, 8:57] - l_cpu[:, 8:57]) / sh).max()))
                    checked += 1
                reps += 1
            worst = max(errs.values())
            ok &= worst < 1e-6
            frac = (nkf_s / F) * (B_s / B)
            cpu_val = B * frac / (t_tot / reps)
            line["cpu_baseline"] = {
                "value": cpu_val, "unit": UNIT, "cores": cores, "kind": "reference" if arm.kind == "ref" else "port",
                "sample": f"{reps} steps of {nkf_s} of {F} keyframes x {B_s} of {B} candidates"
                          + (" (the whole workload, no extrapolation)" if frac == 1.0 else f" (extrapolated linearly, x{1 / frac:.1f})")
                          + f"; OpenMP over keyframes / residual blocks, {cores} threads; KNN = {arm.describe()}; KD-tree build {arm.build_s:.2f}s excluded",
            }
            line["oracle_check"] = {"steps_checked": checked, "ok": bool(ok) if checked else None, "max_rel_err": worst, "rel_err": errs,
                                    "what": "timed GPU records vs the CPU oracle on the same candidates: counters and block counts exact; sums, cost, "
                                            "J^T r, J^T J (relative to their largest entry) within 1e-6"}
            if checked and not ok:
                rc = 3
            if args.config == "c2":
                # SURVEY 8d: both CPU modes of the BAError cost alone next to the composite — M1 = OpenMP over keyframes, one
                # candidate at a time (iba_func.cpp:203,463); M2 = candidates in parallel, each serial over keyframes (NOMAD)
                try:
                    Xc = np.stack([cands(args.warmup + (i % args.steps))[0] for i in range(cores)])
                    t0 = time.perf_counter(); arm.orc.ba_error_sums(Xc[:4], mode=1, strict=True, nthreads=cores); t_m1 = (time.perf_counter() - t0) / 4
                    t0 = time.perf_counter(); arm.orc.ba_error_sums(Xc, mode=2, strict=True, nthreads=cores); t_m2 = (time.perf_counter() - t0) / len(Xc)
                    gpu_bae_ms = sum(stats[k][0] / max(stats[k][1], 1) for k in ("assoc2d", "knn3d", "reduce"))
                    line["cpu_baseline"]["bae_only"] = {
                        "m1_keyframe_parallel_evals_per_s": 1.0 / t_m1, "m2_candidate_parallel_evals_per_s": 1.0 / t_m2,
                        "gpu_bae_only_evals_per_s": 1e3 / gpu_bae_ms if gpu_bae_ms > 0 else None,
                        "sample": f"BAError only, all {F} keyframes: M1 4 candidates one after another, M2 {len(Xc)} candidates at once; {cores} threads"}
                except Exception as e:  # the headline baseline above stands on its own
                    line["cpu_baseline"]["bae_only"] = {"error": str(e)[:200]}
        print(json.dumps(line), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    if rc:
        log("bench.py: the GPU records DISAGREE with the CPU oracle (oracle_check.ok = false)")
        sys.exit(rc)


if __name__ == "__main__":
    main()
