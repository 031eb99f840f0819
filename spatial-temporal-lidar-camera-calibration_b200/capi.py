"""Thin ctypes binding of the C-ABI (include/stlcalib.h).  No compute, no fallback."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _abi
from .pack import KeyFramePack, default_params

_dp = _abi._dp


def _check(lib, h, code):
    if code != 0:
        msg = lib.stl_last_error(h).decode() if h else ""
        raise _abi.StlError(code, msg)


class Context:
    """One GPU's evaluator: owns the device-resident pack, index and workspaces.

    Plays the role of BALoss's constructor state (iba_global.cpp:349-367)."""

    def __init__(self, params: _abi.Params | None = None, device: int = 0):
        self.lib = _abi.load_calib()
        self.params = params if params is not None else default_params()
        h = C.c_void_p()
        code = self.lib.stl_create(C.byref(self.params), device, C.byref(h))
        if code != 0:
            raise _abi.StlError(code, "stl_create failed (an sm_100 GPU is required; there is no CPU fallback)")
        self.h = h
        self.device = device
        self.pack = None
        self.selection = None  # keyframes selected by select_keyframes (None: all)
        self.n_problems = 0  # problems of the frozen set, set after each successful call that makes one (associate / step: 1, *_multi: P)

    def close(self):
        if getattr(self, "h", None):
            self.lib.stl_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- state -------------------------------------------------------------
    def upload(self, pack: KeyFramePack):
        cp = pack.as_c()
        _check(self.lib, self.h, self.lib.stl_upload_pack(self.h, C.byref(cp)))
        self.pack = pack
        self.selection = None  # an upload selects every keyframe again

    def select_keyframes(self, kf=None):
        """Restrict every call that walks keyframes to the local keyframes `kf` (strictly increasing; [] selects none) of the
        uploaded pack: results are those of a context holding ``pack.select(kf)``.  None selects all of them again.  Drops the
        frozen problem set: the linearise calls raise until the next association."""
        if kf is None:
            _check(self.lib, self.h, self.lib.stl_select_keyframes(self.h, None, 0))
            self.selection = None
        else:
            k = np.asarray(kf)
            if k.size == 0:
                k = k.astype(np.int64).reshape(0)
            if k.ndim != 1 or k.dtype.kind not in "iu":  # as KeyFramePack.select: no silent truncation of non-integers
                raise TypeError("select_keyframes: kf must be a 1-D list of integer keyframe indices")
            k = k.astype(np.int64)
            if k.size and (k.min() < -2**31 or k.max() >= 2**31):
                raise ValueError("keyframe index outside the int32 range")
            k = np.ascontiguousarray(k, dtype=np.int32)
            buf = k if k.size else np.zeros(1, np.int32)  # an empty selection is a non-null pointer with n = 0 (NULL selects all)
            _check(self.lib, self.h, self.lib.stl_select_keyframes(self.h, buf.ctypes.data_as(_abi._i32p), int(k.size)))
            self.selection = k.copy()
        self.n_blocks = None
        self.n_problems = 0

    def allow_oversize_keyframes(self, flag: bool):
        """Let the next :meth:`upload` accept keyframes whose K1 tables do not fit the one-kernel K1's shared memory (4K
        images, many keypoints); they run on the banded three-kernel K1 with the same results.  False (the default) refuses
        such a pack.  The resident pack is not touched."""
        if not (isinstance(flag, (bool, np.bool_)) or (isinstance(flag, (int, np.integer)) and flag in (0, 1))):
            raise TypeError("allow_oversize_keyframes: flag must be a bool (or 0 / 1)")
        _check(self.lib, self.h, self.lib.stl_allow_oversize_keyframes(self.h, 1 if flag else 0))

    def oversize_keyframes(self) -> np.ndarray:
        """Local keyframes of the resident pack that run on the oversize path, increasing (int32)."""
        n = C.c_int32(0)
        _check(self.lib, self.h, self.lib.stl_oversize_keyframes(self.h, None, 0, C.byref(n)))
        out = np.zeros(max(n.value, 1), dtype=np.int32)
        _check(self.lib, self.h, self.lib.stl_oversize_keyframes(self.h, out.ctypes.data_as(_abi._i32p), int(out.size), C.byref(n)))
        return out[: n.value].copy()

    def eval_frames(self, x) -> np.ndarray:
        """x [B,7] -> the per-keyframe record of BAError [B, n_kf, 13] (the 13 values of :meth:`debug_frame`, in its order) of
        every keyframe of the pack; rows of unselected keyframes are zero.  Each rank returns its own keyframes."""
        x = np.ascontiguousarray(np.atleast_2d(x), dtype=np.float64)
        B = x.shape[0]
        if self.pack is None:
            raise _abi.StlError(4, "no pack uploaded")
        out = np.empty((B, int(self.pack.n_kf), 13), dtype=np.float64)
        _check(self.lib, self.h, self.lib.stl_eval_frames(self.h, x.ctypes.data_as(_dp), B, out.ctypes.data_as(_dp)))
        return out

    # -- Nomad / iba_func path ---------------------------------------------
    def eval_sums(self, x) -> np.ndarray:
        """x [B,7] (host) -> partial sums [B,12] (host) of this context's keyframes."""
        x = np.ascontiguousarray(np.atleast_2d(x), dtype=np.float64)
        B = x.shape[0]
        out = np.empty((B, _abi.STL_EVAL_NSUMS), dtype=np.float64)
        _check(self.lib, self.h, self.lib.stl_eval_batch(self.h, x.ctypes.data_as(_dp), B,
                                                         out.ctypes.data_as(C.POINTER(_abi.EvalSums))))
        return out

    def eval_sums_device(self, x, d_out_ptr: int, stream_ptr: int = 0):
        """Enqueue on `stream_ptr`; result rows land in device memory at d_out_ptr ([B,12] fp64)."""
        x = np.ascontiguousarray(np.atleast_2d(x), dtype=np.float64)
        _check(self.lib, self.h, self.lib.stl_eval_batch_device(self.h, x.ctypes.data_as(_dp), x.shape[0],
                                                                C.c_void_p(d_out_ptr), C.c_void_p(stream_ptr)))

    def finalize(self, sums_row):
        """BAError's return tuple (f1, f2, C, valid_cnt_3d_2d, cnt_3d_2d), iba_global.cpp:330-343."""
        s = _abi.EvalSums(*[float(v) for v in sums_row])
        o = _abi.BAErrorOut()
        self.lib.stl_finalize(C.byref(self.params), C.byref(s), C.byref(o))
        return o.f1, o.f2, o.C, o.valid_cnt_3d_2d, o.cnt_3d_2d

    def bbo(self, ba):
        """BALoss::eval_x's BBO values (f, C1, C2, C3), iba_global.cpp:386-388."""
        o = _abi.BAErrorOut(ba[0], ba[1], ba[2], int(ba[3]), int(ba[4]))
        out = (C.c_double * 4)()
        self.lib.stl_bbo(C.byref(self.params), C.byref(o), out)
        return tuple(out)

    # -- LM path -------------------------------------------------------------
    def associate(self, x0, wait: bool = True):
        """BuildProblem at x0.  wait=False enqueues only (block counts through :meth:`block_counts` later)."""
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        if not wait:
            _check(self.lib, self.h, self.lib.stl_associate(self.h, x0.ctypes.data_as(_dp), None))
            self.n_blocks = None
            self.n_problems = 1
            return None
        nb = np.zeros(4, np.int64)
        _check(self.lib, self.h, self.lib.stl_associate(self.h, x0.ctypes.data_as(_dp), nb.ctypes.data_as(_abi._i64p)))
        self.n_blocks = nb.copy()
        self.n_problems = 1
        return nb

    def block_counts(self):
        nb = np.zeros(4, np.int64)
        _check(self.lib, self.h, self.lib.stl_block_counts(self.h, nb.ctypes.data_as(_abi._i64p)))
        self.n_blocks = nb.copy()
        return nb

    def step(self, x, reassociate: bool = True) -> np.ndarray:
        """BAError sums + (BuildProblem at x[0]) + linearisation of x [B,7] in one call -> [B,74] (host):
        columns 0..11 the evaluation sums, 12..73 the linearisation record."""
        x = np.ascontiguousarray(np.atleast_2d(x), dtype=np.float64)
        B = x.shape[0]
        out = np.empty((B, _abi.STL_STEP_NSUMS), dtype=np.float64)
        _check(self.lib, self.h, self.lib.stl_step_batch(self.h, x.ctypes.data_as(_dp), B, int(reassociate),
                                                         out.ctypes.data_as(C.POINTER(_abi.StepSums))))
        self.n_blocks = None
        if reassociate:
            self.n_problems = 1
        return out

    def step_device(self, x, d_out_ptr: int, stream_ptr: int = 0, reassociate: bool = True):
        x = np.ascontiguousarray(np.atleast_2d(x), dtype=np.float64)
        _check(self.lib, self.h, self.lib.stl_step_batch_device(self.h, x.ctypes.data_as(_dp), x.shape[0], int(reassociate),
                                                                C.c_void_p(d_out_ptr), C.c_void_p(stream_ptr)))
        self.n_blocks = None
        if reassociate:
            self.n_problems = 1

    # -- LM path, several starts (problem set) ---------------------------------------
    @staticmethod
    def _mask(rebuild, P):
        if rebuild is None:
            return None, None
        m = np.ascontiguousarray(np.asarray(rebuild).reshape(-1) != 0, dtype=np.uint8)
        if m.size != P:
            raise ValueError(f"rebuild has {m.size} entries for {P} starts")
        return m, m.ctypes.data_as(_abi._u8p)

    @staticmethod
    def _problems(problem, B):
        if problem is None:
            return None, None
        p = np.ascontiguousarray(np.asarray(problem).reshape(-1), dtype=np.int32)
        if p.size != B:
            raise ValueError(f"problem has {p.size} entries for {B} candidates")
        return p, p.ctypes.data_as(_abi._i32p)

    def associate_multi(self, X0, rebuild=None, wait: bool = True):
        """BuildProblem at X0[p] for every start p (X0 [P,7]) -> block counts [P,4] (None with wait=False).  rebuild (mask [P]):
        re-associate only the flagged problems of the current set of P; the others keep their blocks."""
        X0 = np.ascontiguousarray(np.atleast_2d(X0), dtype=np.float64)
        P = X0.shape[0]
        keep, m = self._mask(rebuild, P)
        nb = np.zeros((P, 4), np.int64)
        _check(self.lib, self.h, self.lib.stl_associate_multi(self.h, X0.ctypes.data_as(_dp), P, m,
                                                              nb.ctypes.data_as(_abi._i64p) if wait else None))
        self.n_blocks = None
        self.n_problems = P
        return nb if wait else None

    def block_counts_multi(self) -> np.ndarray:
        """Block counts [P,4] of the frozen set (waits for its association)."""
        nb = np.zeros((_abi.STL_MAX_PROBLEMS, 4), np.int64)
        _check(self.lib, self.h, self.lib.stl_block_counts_multi(self.h, nb.ctypes.data_as(_abi._i64p), _abi.STL_MAX_PROBLEMS))
        return nb[: self.n_problems].copy()

    def linearize_multi(self, X, problem=None) -> np.ndarray:
        """Candidate b (X [B,7]) on problem problem[b] (None: B == P, candidate b on problem b) -> [B,62] (host)."""
        X = np.ascontiguousarray(np.atleast_2d(X), dtype=np.float64)
        B = X.shape[0]
        keep, pp = self._problems(problem, B)
        out = np.empty((B, _abi.STL_LIN_NSUMS), dtype=np.float64)
        _check(self.lib, self.h, self.lib.stl_linearize_multi(self.h, X.ctypes.data_as(_dp), B, pp,
                                                              out.ctypes.data_as(C.POINTER(_abi.LinSums))))
        return out

    def linearize_frames(self, X, problem=None) -> np.ndarray:
        """Normal equations per keyframe: candidate b (X [B,7]) on problem problem[b] (None: every candidate on problem 0, which
        needs a frozen set of one) -> [B, n_kf, 62] (host), row f = the :meth:`linearize_multi` record of keyframe f's blocks
        alone.  The rows of a candidate sum to its record; rows of unselected keyframes are zero.  Each rank returns its own
        keyframes (no exchange)."""
        X = np.ascontiguousarray(np.atleast_2d(X), dtype=np.float64)
        if X.ndim != 2 or X.shape[1] != 7 or X.shape[0] == 0:
            raise ValueError(f"linearize_frames: X must be [B, 7] with B >= 1, got shape {X.shape}")
        B = X.shape[0]
        keep, pp = self._problems(problem, B)
        if self.pack is None:
            raise _abi.StlError(4, "no pack uploaded")
        out = np.empty((B, int(self.pack.n_kf), _abi.STL_LIN_NSUMS), dtype=np.float64)
        _check(self.lib, self.h, self.lib.stl_linearize_frames(self.h, X.ctypes.data_as(_dp), B, pp,
                                                               out.ctypes.data_as(C.POINTER(_abi.LinSums))))
        return out

    def linearize_multi_device(self, X, d_out_ptr: int, problem=None, stream_ptr: int = 0):
        X = np.ascontiguousarray(np.atleast_2d(X), dtype=np.float64)
        keep, pp = self._problems(problem, X.shape[0])
        _check(self.lib, self.h, self.lib.stl_linearize_multi_device(self.h, X.ctypes.data_as(_dp), X.shape[0], pp,
                                                                     C.c_void_p(d_out_ptr), C.c_void_p(stream_ptr)))

    def step_multi(self, X, rebuild=None) -> np.ndarray:
        """One LM iteration for each start (X [P,7]): evaluation sums, BuildProblem at X[p] of the flagged problems (None: all,
        a new set), linearisation of problem p at X[p] -> [P,74] (host)."""
        X = np.ascontiguousarray(np.atleast_2d(X), dtype=np.float64)
        P = X.shape[0]
        keep, m = self._mask(rebuild, P)
        out = np.empty((P, _abi.STL_STEP_NSUMS), dtype=np.float64)
        _check(self.lib, self.h, self.lib.stl_step_multi(self.h, X.ctypes.data_as(_dp), P, m, out.ctypes.data_as(C.POINTER(_abi.StepSums))))
        self.n_blocks = None
        self.n_problems = P
        return out

    def step_multi_device(self, X, d_out_ptr: int, rebuild=None, stream_ptr: int = 0):
        X = np.ascontiguousarray(np.atleast_2d(X), dtype=np.float64)
        keep, m = self._mask(rebuild, X.shape[0])
        _check(self.lib, self.h, self.lib.stl_step_multi_device(self.h, X.ctypes.data_as(_dp), X.shape[0], m,
                                                                C.c_void_p(d_out_ptr), C.c_void_p(stream_ptr)))
        self.n_blocks = None
        self.n_problems = X.shape[0]

    def gpr_hyper(self):
        """(sigma, l) of the GPR blocks of the last association, block order -> [nG, 2]."""
        nb = self.block_counts()
        out = np.zeros((max(int(nb[3]), 1), 2))
        _check(self.lib, self.h, self.lib.stl_gpr_hyper(self.h, out.ctypes.data_as(_dp), int(nb[3])))
        return out[: int(nb[3])]

    # -- the problems before the hot path (N4) --------------------------------------
    def he_linearize(self, edges: "HandEyeEdges", x, want_chi2: bool = False):
        """EdgeHE + EdgeRegulation (NLHECalib.hpp:27-116) at x [B,7] -> [B,62] (cost = sum rho(chi2), g, H) (, chi2 [B,n])."""
        x = np.ascontiguousarray(np.atleast_2d(x), dtype=np.float64)
        B = x.shape[0]
        out = np.zeros((B, _abi.STL_LIN_NSUMS))
        chi2 = np.zeros((B, max(edges.n, 1))) if want_chi2 else None
        c = edges.as_c()
        _check(self.lib, self.h, self.lib.stl_he_linearize(self.h, C.byref(c), x.ctypes.data_as(_dp), B, out.ctypes.data_as(C.POINTER(_abi.LinSums)),
                                                           chi2.ctypes.data_as(_dp) if want_chi2 else None))
        return (out, chi2[:, : edges.n]) if want_chi2 else out

    def calib_linearize(self, edges: "CalibBAEdges", x, want_chi2: bool = False):
        """calibEdge problem (Optimizer.cc:65-205,1399-1744) at x [B,7] -> [B,62] (, chi2 [B,n_edges])."""
        x = np.ascontiguousarray(np.atleast_2d(x), dtype=np.float64)
        B = x.shape[0]
        out = np.zeros((B, _abi.STL_LIN_NSUMS))
        chi2 = np.zeros((B, max(edges.n_edges, 1))) if want_chi2 else None
        c = edges.as_c()
        _check(self.lib, self.h, self.lib.stl_calib_linearize(self.h, C.byref(c), x.ctypes.data_as(_dp), B, out.ctypes.data_as(C.POINTER(_abi.LinSums)),
                                                              chi2.ctypes.data_as(_dp) if want_chi2 else None))
        return (out, chi2[:, : edges.n_edges]) if want_chi2 else out

    # -- multi-GPU -------------------------------------------------------------
    def comm_unique_id(self) -> bytes:
        """ncclGetUniqueId (call on one rank, hand the bytes to the others)."""
        buf = (C.c_uint8 * _abi.STL_COMM_ID_BYTES)()
        _check(self.lib, self.h, self.lib.stl_comm_unique_id(buf))
        return bytes(buf)

    def comm_init(self, uid: bytes, rank: int, n_ranks: int):
        """Attach an NCCL communicator: this context holds keyframe shard `rank` of `n_ranks`; every
        evaluation / linearisation / step then returns the all-reduced totals."""
        buf = (C.c_uint8 * _abi.STL_COMM_ID_BYTES).from_buffer_copy(uid)
        _check(self.lib, self.h, self.lib.stl_comm_init(self.h, buf, rank, n_ranks))

    def comm_stats(self):
        """dict(p2p: records exchanged inside the finishing kernel over peer memory?, p2p_exchanges, nccl_exchanges)."""
        out = np.zeros(3, np.int64)
        _check(self.lib, self.h, self.lib.stl_comm_stats(self.h, out.ctypes.data_as(_abi._i64p)))
        return dict(p2p=bool(out[0]), p2p_exchanges=int(out[1]), nccl_exchanges=int(out[2]))

    def comm_info(self):
        r, n = C.c_int32(0), C.c_int32(1)
        _check(self.lib, self.h, self.lib.stl_comm_info(self.h, C.byref(r), C.byref(n)))
        return r.value, n.value

    def linearize(self, x) -> np.ndarray:
        x = np.ascontiguousarray(np.atleast_2d(x), dtype=np.float64)
        B = x.shape[0]
        out = np.empty((B, _abi.STL_LIN_NSUMS), dtype=np.float64)
        _check(self.lib, self.h, self.lib.stl_linearize_batch(self.h, x.ctypes.data_as(_dp), B,
                                                              out.ctypes.data_as(C.POINTER(_abi.LinSums))))
        return out

    def linearize_device(self, x, d_out_ptr: int, stream_ptr: int = 0):
        x = np.ascontiguousarray(np.atleast_2d(x), dtype=np.float64)
        _check(self.lib, self.h, self.lib.stl_linearize_batch_device(self.h, x.ctypes.data_as(_dp), x.shape[0],
                                                                     C.c_void_p(d_out_ptr), C.c_void_p(stream_ptr)))

    def eval_blocks(self, x, rmax: int = 0):
        """Per-block residuals and Jacobians of the frozen problem at x (what each ceres::CostFunction /
        g2o edge of iba_local.cpp would return, before the robust kernel).  -> dict(type, kf, kp, n_res,
        residuals [nb, rmax], jacobians [nb, rmax, 7])."""
        x = np.ascontiguousarray(x, dtype=np.float64).reshape(7)
        ncov = int(self.pack.n_covis) if self.pack is not None else _abi.STL_MAX_COVIS
        rmax = int(rmax) if rmax else max(3, 2 * ncov)
        if getattr(self, "n_blocks", None) is None:
            self.block_counts()
        nb = int(self.n_blocks.sum())
        cap = max(nb, 1)
        out = dict(type=np.zeros(cap, np.int32), kf=np.zeros(cap, np.int32), kp=np.zeros(cap, np.int32), n_res=np.zeros(cap, np.int32),
                   residuals=np.zeros((cap, rmax)), jacobians=np.zeros((cap, rmax, 7)))
        n = C.c_int64(0)
        _check(self.lib, self.h, self.lib.stl_eval_blocks(
            self.h, x.ctypes.data_as(_dp), rmax, cap, out["type"].ctypes.data_as(_abi._i32p), out["kf"].ctypes.data_as(_abi._i32p),
            out["kp"].ctypes.data_as(_abi._i32p), out["n_res"].ctypes.data_as(_abi._i32p), out["residuals"].ctypes.data_as(_dp),
            out["jacobians"].ctypes.data_as(_dp), C.byref(n)))
        return {k: v[: n.value] for k, v in out.items()}

    # -- debug getters (parity tests) ------------------------------------------
    def debug_corrset(self, b: int, kf: int):
        cap = int(self.pack.kp_offset[kf + 1] - self.pack.kp_offset[kf]) if self.pack is not None else 65536
        kp = np.zeros(max(cap, 1), np.uint32)
        pt = np.zeros(max(cap, 1), np.uint32)
        n = C.c_int32(0)
        _check(self.lib, self.h, self.lib.stl_debug_corrset(self.h, b, kf, kp.ctypes.data_as(_abi._u32p),
                                                            pt.ctypes.data_as(_abi._u32p), cap, C.byref(n)))
        return kp[:n.value], pt[:n.value]

    def debug_align(self, b: int, kf: int):
        cap = int(self.pack.kp_offset[kf + 1] - self.pack.kp_offset[kf]) if self.pack is not None else 65536
        cap = max(cap, 1)
        kp = np.zeros(cap, np.uint32)
        nn = np.zeros(cap, np.uint32)
        m = np.zeros(cap, np.int32)
        pl = np.zeros(cap, np.int32)
        d = np.zeros(cap, np.float64)
        knn = np.zeros((cap, 32), np.uint32)
        n = C.c_int32(0)
        _check(self.lib, self.h, self.lib.stl_debug_align(
            self.h, b, kf, kp.ctypes.data_as(_abi._u32p), nn.ctypes.data_as(_abi._u32p), m.ctypes.data_as(_abi._i32p),
            pl.ctypes.data_as(_abi._i32p), d.ctypes.data_as(_dp), knn.ctypes.data_as(_abi._u32p), cap, C.byref(n)))
        k = n.value
        return dict(kp=kp[:k], nn=nn[:k], m=m[:k], is_plane=pl[:k], dist=d[:k], knn=knn[:k])

    def debug_frame(self, b: int, kf: int):
        out = np.zeros(13)
        _check(self.lib, self.h, self.lib.stl_debug_frame(self.h, b, kf, out.ctypes.data_as(_dp)))
        names = ("sum_3d2d", "valid_3d2d", "cnt_3d2d", "sum_he", "cnt_he", "kept", "n_corr", "n_queries",
                 "sum_3d3d", "valid_3d3d", "cnt_3d3d", "valid_pl", "valid_pt")
        return dict(zip(names, out))

    def debug_trig(self, x):
        """The device's acos (of x clamped to [-1, 1]) and cos, as the plane fit evaluates them."""
        x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1)
        a, c = np.zeros_like(x), np.zeros_like(x)
        _check(self.lib, self.h, self.lib.stl_debug_trig(self.h, x.ctypes.data_as(_dp), len(x), a.ctypes.data_as(_dp), c.ctypes.data_as(_dp)))
        return a, c

    def knn3d(self, kf: int, q, k: int, radius2: float = 0.0):
        q = np.ascontiguousarray(q, dtype=np.float64).reshape(-1, 3)
        nq = q.shape[0]
        idx = np.zeros((nq, k), np.uint32)
        d2 = np.zeros((nq, k), np.float64)
        cnt = np.zeros(nq, np.int32)
        _check(self.lib, self.h, self.lib.stl_knn3d(self.h, kf, q.ctypes.data_as(_dp), nq, k, radius2,
                                                    idx.ctypes.data_as(_abi._u32p), d2.ctypes.data_as(_dp),
                                                    cnt.ctypes.data_as(_abi._i32p)))
        return idx, d2, cnt

    # -- measurement -------------------------------------------------------------
    def set_stream(self, stream_ptr: int = 0):
        """All later calls without an explicit stream enqueue on this cudaStream_t (0 = the context's own)."""
        _check(self.lib, self.h, self.lib.stl_set_stream(self.h, C.c_void_p(stream_ptr)))

    def set_profiling(self, on: bool):
        _check(self.lib, self.h, self.lib.stl_set_profiling(self.h, int(on)))

    def stage_stats(self):
        ms = np.zeros(_abi.STL_NSTAGES)
        n = np.zeros(_abi.STL_NSTAGES, np.int64)
        _check(self.lib, self.h, self.lib.stl_stage_stats(self.h, ms.ctypes.data_as(_dp), n.ctypes.data_as(_abi._i64p)))
        return {name: (float(ms[i]), int(n[i])) for i, name in enumerate(_abi.STAGE_NAMES)}

    def work_counters(self):
        out = np.zeros(8)
        _check(self.lib, self.h, self.lib.stl_work_counters(self.h, out.ctypes.data_as(_dp)))
        return dict(points=out[0], q2d=out[1], q3d_nn=out[2], q3d_knn=out[3], k1_bytes=out[4], launches=out[5], k1_overflow_units=out[6],
                    assoc_reused=out[7])


class HandEyeEdges:
    """Host container of stl_he_edges_t: motion pairs (Ta camera, Tb LiDAR) as [n,12] row-major 3x4."""

    def __init__(self, Ta, Tb, info=None, huber_delta: float = 0.0, regulation: float = 0.0):
        self.Ta = np.ascontiguousarray(Ta, dtype=np.float64).reshape(-1, 12)
        self.Tb = np.ascontiguousarray(Tb, dtype=np.float64).reshape(-1, 12)
        self.n = len(self.Ta)
        self.info = None if info is None else np.ascontiguousarray(info, dtype=np.float64)
        self.huber_delta, self.regulation = float(huber_delta), float(regulation)

    def as_c(self):
        c = _abi.HeEdges(self.n, self.Ta.ctypes.data_as(_dp), self.Tb.ctypes.data_as(_dp),
                         self.info.ctypes.data_as(_dp) if self.info is not None else None, self.huber_delta, self.regulation)
        c._keep = self
        return c


class CalibBAEdges:
    """Host container of stl_calib_edges_t."""

    def __init__(self, edge_offset, Tlw_quat, intrinsics, Xw, obs, inv_sigma2, level=None, huber_delta: float = 5.991 ** 0.5):
        self.edge_offset = np.ascontiguousarray(edge_offset, dtype=np.int64)
        self.Tlw_quat = np.ascontiguousarray(Tlw_quat, dtype=np.float64).reshape(-1, 6)
        self.intrinsics = np.ascontiguousarray(intrinsics, dtype=np.float32).reshape(-1, 4)
        self.Xw = np.ascontiguousarray(Xw, dtype=np.float64).reshape(-1, 3)
        self.obs = np.ascontiguousarray(obs, dtype=np.float64).reshape(-1, 2)
        self.inv_sigma2 = np.ascontiguousarray(inv_sigma2, dtype=np.float32)
        self.level = None if level is None else np.ascontiguousarray(level, dtype=np.uint8)
        self.n_kf, self.n_edges = len(self.Tlw_quat), len(self.Xw)
        self.huber_delta = float(huber_delta)

    def as_c(self):
        c = _abi.CalibEdges(self.n_kf, self.n_edges, self.edge_offset.ctypes.data_as(_abi._i64p), self.Tlw_quat.ctypes.data_as(_dp),
                            self.intrinsics.ctypes.data_as(C.POINTER(C.c_float)), self.Xw.ctypes.data_as(_dp), self.obs.ctypes.data_as(_dp),
                            self.inv_sigma2.ctypes.data_as(C.POINTER(C.c_float)),
                            self.level.ctypes.data_as(C.POINTER(C.c_uint8)) if self.level is not None else None, self.huber_delta)
        c._keep = self
        return c


def gpr_nlml(x, y, sigma, l, sigma_noise: float = 1e-10, flavour: int = 0):
    """GPRHyperLoss::Evaluate (GPR.hpp:154-174) -> (cost, grad[2]); host only."""
    lib = _abi.load_calib()
    x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, 2)
    y = np.ascontiguousarray(y, dtype=np.float64)
    cost, g = C.c_double(0), np.zeros(2)
    code = lib.stl_gpr_nlml(x.ctypes.data_as(_dp), y.ctypes.data_as(_dp), len(y), sigma_noise, sigma, l, flavour, C.byref(cost), g.ctypes.data_as(_dp))
    if code != 0:
        raise _abi.StlError(code, "Cholesky factorisation of the kernel matrix failed")
    return cost.value, g


def gpr_fit(x, y, sigma0: float = 10.0, l0: float = 10.0, sigma_noise: float = 1e-10, max_iter: int = 15, flavour: int = 0):
    """GPR::fit (GPR.hpp:350-387) -> dict(sigma, l, cost0, cost, iterations, evaluations); host only."""
    lib = _abi.load_calib()
    x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, 2)
    y = np.ascontiguousarray(y, dtype=np.float64)
    out = np.zeros(6)
    code = lib.stl_gpr_fit(x.ctypes.data_as(_dp), y.ctypes.data_as(_dp), len(y), sigma_noise, sigma0, l0, max_iter, flavour, out.ctypes.data_as(_dp))
    if code != 0:
        raise _abi.StlError(code, "the objective could not be evaluated at the starting point")
    return dict(sigma=out[0], l=out[1], cost0=out[2], cost=out[3], iterations=int(out[4]), evaluations=int(out[5]))
