"""CPU ORACLE loader (test infrastructure, NOT product code).

ctypes wrapper of oracle/liboracle.so (self-contained port) and
oracle/_ref/liboracle_ref.so (same restatement, KNN through the reference's real
vendored nanoflann).  Only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs may import this module.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import importlib
import os
import subprocess
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
if _ROOT not in sys.path:
    sys.path.insert(0, _ROOT)
_pkg = importlib.import_module("spatial-temporal-lidar-camera-calibration_b200")
_abi = _pkg._abi

PORT_PATH = os.path.join(_HERE, "liboracle.so")
REF_PATH = os.path.join(_HERE, "_ref", "liboracle_ref.so")

_vp, _dp = C.c_void_p, C.POINTER(C.c_double)
_u32p, _i32p, _i64p = C.POINTER(C.c_uint32), C.POINTER(C.c_int32), C.POINTER(C.c_int64)

_SYMS = {
    "orc_backend": (C.c_char_p, []),
    "orc_max_threads": (C.c_int, []),
    "orc_create": (_vp, [C.POINTER(_abi.Pack), C.POINTER(_abi.Params), C.c_int, C.c_int, C.c_int]),
    "orc_destroy": (None, [_vp]),
    "orc_build_seconds": (C.c_double, [_vp]),
    "orc_ba_error": (None, [_vp, _dp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_abi.EvalSums), _i64p, _dp]),
    "orc_finalize": (None, [C.POINTER(_abi.Params), C.POINTER(_abi.EvalSums), C.POINTER(_abi.BAErrorOut)]),
    "orc_frame_debug": (C.c_int, [_vp, _dp, C.c_int, _i64p]),
    "orc_frame_sums": (None, [_vp, _dp, C.c_int, _dp]),
    "orc_frame_corr": (C.c_int, [_vp, _u32p, _u32p, C.c_int]),
    "orc_frame_align": (C.c_int, [_vp, _u32p, _u32p, _i32p, _i32p, _dp, _u32p, _dp, C.c_int]),
    "orc_knn3d": (None, [_vp, C.c_int, _dp, C.c_int, C.c_int, C.c_double, C.c_int, _u32p, _dp, _i32p, _i64p]),
    "orc_associate": (None, [_vp, _dp, C.c_int, _i64p, _i64p]),
    "orc_linearize": (None, [_vp, _dp, C.c_int, C.POINTER(_abi.LinSums)]),
    "orc_linearize_mt": (None, [_vp, _dp, C.c_int, C.c_int, C.POINTER(_abi.LinSums)]),
    "orc_num_blocks": (C.c_int64, [_vp]),
    "orc_block_key": (None, [_vp, C.c_int64, _i32p]),
    "orc_block_eval": (C.c_int, [_vp, C.c_int64, _dp, _dp, _dp]),
    "orc_block_eval_plain": (C.c_int, [_vp, C.c_int64, _dp, _dp]),
    "orc_gpr_hyper_loss": (C.c_int, [_dp, _dp, C.c_int, C.c_double, C.c_double, C.c_double, _dp, _dp]),
    "orc_set_gpr_hyper": (None, [_vp, _dp, C.c_int64]),
    "orc_gpr_train": (C.c_int, [_vp, C.c_int64, _dp, _dp, _dp]),
    "orc_he_linearize": (None, [C.POINTER(_abi.HeEdges), _dp, C.c_int, C.POINTER(_abi.LinSums), _dp]),
    "orc_calib_linearize": (None, [C.POINTER(_abi.CalibEdges), _dp, C.c_int, C.POINTER(_abi.LinSums), _dp]),
    "orc_he_edge": (None, [_dp, _dp, _dp, _dp, _dp]),
    "orc_calib_edge_plain": (None, [_dp, _dp, _dp, _dp, _dp, _dp]),
    "orc_rotvec": (None, [_dp, _dp]),
    "orc_covariance": (None, [_dp, _u32p, C.c_int, _dp]),
    "orc_smallest_eigvec": (None, [_dp, _dp]),
    "orc_sim3exp_dual": (None, [_dp, _dp]),
    "orc_se3exp": (None, [_dp, _dp, _dp]),
    "orc_sim3exp": (None, [_dp, _dp, _dp, _dp]),
    "orc_se3log": (None, [_dp, _dp, _dp]),
    "orc_plane_fit": (None, [_dp, C.c_int, _dp, _dp]),
}

_libs = {}


def build(verbose: bool = False) -> None:
    """Builds oracle/liboracle.so and, when /root/reference exists, oracle/_ref/."""
    r = subprocess.run(["make", "-C", _HERE], capture_output=True, text=True)
    if verbose or r.returncode:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode:
        raise RuntimeError("oracle build failed")


def load(kind: str = "port"):
    """kind: 'port' | 'ref' | 'best' (ref if present, else port)."""
    if kind == "best":
        kind = "ref" if os.path.exists(REF_PATH) else "port"
    if kind not in _libs:
        path = PORT_PATH if kind == "port" else REF_PATH
        if not os.path.exists(path):
            if kind == "port":
                build()
            else:
                raise FileNotFoundError(path)
        lib = C.CDLL(path)
        for name, (res, args) in _SYMS.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _libs[kind] = lib
    return _libs[kind]


REFMATH_PATH = os.path.join(_HERE, "_ref", "liboracle_refmath.so")


def load_refmath():
    """The reference's own arithmetic lines compiled verbatim (oracle/Makefile `refmath`); None if not built."""
    if not os.path.exists(REFMATH_PATH):
        return None
    if "refmath" not in _libs:
        lib = C.CDLL(REFMATH_PATH)
        lib.refm_covariance.argtypes = [_dp, C.c_int, _u32p, C.c_int, _dp]
        lib.refm_fast_eigen.argtypes = [_dp, _dp, _dp]
        lib.refm_sim3exp.argtypes = [_dp, _dp, _dp, _dp]
        lib.refm_sim3exp_dual.argtypes = [_dp, _dp]
        lib.refm_se3exp.argtypes = [_dp, _dp, _dp]
        for f in (lib.refm_covariance, lib.refm_fast_eigen, lib.refm_sim3exp, lib.refm_sim3exp_dual, lib.refm_se3exp):
            f.restype = None
        _libs["refmath"] = lib
    return _libs["refmath"]


def have_ref() -> bool:
    return os.path.exists(REF_PATH)


def digest(*arrays) -> int:
    """64-bit BLAKE2b of the arrays' dtypes, shapes and bytes (-0.0 counted as 0.0): what a stored fixture keeps
    of an output too large to store, equal exactly when the arrays are equal bit for bit."""
    h = hashlib.blake2b(digest_size=8)
    for a in arrays:
        a = np.ascontiguousarray(a)
        if a.dtype.kind == "f":
            a = a + a.dtype.type(0)
        h.update(f"{a.dtype.str}{a.shape}".encode())
        h.update(a.tobytes())
    return int.from_bytes(h.digest(), "little")


def _d(a):
    return a.ctypes.data_as(_dp)


class Oracle:
    """CPU restatement of BAError / BuildProblem over a KeyFramePack."""

    def __init__(self, pack, params=None, kind: str = "port", leaf2d: int = 10, leaf3d: int = 30, nthreads: int = 0):
        self.lib = load(kind)
        self.kind = self.lib.orc_backend().decode()
        self.pack = pack
        self.params = params if params is not None else _pkg.default_params()
        self._cpack = pack.as_c()
        self.h = self.lib.orc_create(C.byref(self._cpack), C.byref(self.params), leaf2d, leaf3d, nthreads)
        self.build_seconds = self.lib.orc_build_seconds(self.h)

    def close(self):
        if getattr(self, "h", None):
            self.lib.orc_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def max_threads(self) -> int:
        return self.lib.orc_max_threads()

    def ba_error_sums(self, x, mode: int = 1, strict: bool = False, nthreads: int = 0):
        """x: [B,7] -> (sums[B,12] ndarray, ties[3], counters[3])."""
        x = np.ascontiguousarray(np.atleast_2d(x), dtype=np.float64)
        B = x.shape[0]
        out = (_abi.EvalSums * B)()
        ties = np.zeros(3, dtype=np.int64)
        cnt = np.zeros(3, dtype=np.float64)
        self.lib.orc_ba_error(self.h, _d(x), B, mode, int(strict), nthreads, out, ties.ctypes.data_as(_i64p), _d(cnt))
        arr = np.frombuffer(out, dtype=np.float64).reshape(B, _abi.STL_EVAL_NSUMS).copy()
        return arr, ties, cnt

    def finalize(self, sums_row):
        s = _abi.EvalSums(*[float(v) for v in sums_row])
        o = _abi.BAErrorOut()
        self.lib.orc_finalize(C.byref(self.params), C.byref(s), C.byref(o))
        return o.f1, o.f2, o.C, o.valid_cnt_3d_2d, o.cnt_3d_2d

    def frame_debug(self, x, kf: int):
        """Returns dict(corr_kp, corr_pt, align_*, ties) for one keyframe."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        ties = np.zeros(3, dtype=np.int64)
        n = self.lib.orc_frame_debug(self.h, _d(x), kf, ties.ctypes.data_as(_i64p))
        kp = np.zeros(max(n, 1), np.uint32)
        pt = np.zeros(max(n, 1), np.uint32)
        self.lib.orc_frame_corr(self.h, kp.ctypes.data_as(_u32p), pt.ctypes.data_as(_u32p), n)
        cap = max(n, 1)
        akp = np.zeros(cap, np.uint32)
        ann = np.zeros(cap, np.uint32)
        am = np.zeros(cap, np.int32)
        apl = np.zeros(cap, np.int32)
        ad = np.zeros(cap, np.float64)
        aknn = np.zeros((cap, 32), np.uint32)
        anrm = np.zeros((cap, 3), np.float64)
        na = self.lib.orc_frame_align(self.h, akp.ctypes.data_as(_u32p), ann.ctypes.data_as(_u32p), am.ctypes.data_as(_i32p),
                                      apl.ctypes.data_as(_i32p), _d(ad), aknn.ctypes.data_as(_u32p), _d(anrm), cap)
        return dict(corr_kp=kp[:n], corr_pt=pt[:n], align_kp=akp[:na], align_nn=ann[:na], align_m=am[:na],
                    align_is_plane=apl[:na], align_dist=ad[:na], align_knn=aknn[:na], align_normal=anrm[:na], ties=ties)

    def frame_sums(self, x, kf: int):
        x = np.ascontiguousarray(x, dtype=np.float64)
        out = np.zeros(13)
        self.lib.orc_frame_sums(self.h, _d(x), kf, _d(out))
        names = ("sum_3d2d", "valid_3d2d", "cnt_3d2d", "sum_he", "cnt_he", "kept", "n_corr", "n_queries",
                 "sum_3d3d", "valid_3d3d", "cnt_3d3d", "valid_pl", "valid_pt")
        return dict(zip(names, out))

    def knn3d(self, kf: int, q, k: int, radius2: float = 0.0, strict: bool = False):
        q = np.ascontiguousarray(q, dtype=np.float64).reshape(-1, 3)
        nq = q.shape[0]
        idx = np.zeros((nq, k), np.uint32)
        d2 = np.zeros((nq, k), np.float64)
        cnt = np.zeros(nq, np.int32)
        ties = C.c_int64(0)
        self.lib.orc_knn3d(self.h, kf, _d(q), nq, k, radius2, int(strict), idx.ctypes.data_as(_u32p), _d(d2),
                           cnt.ctypes.data_as(_i32p), C.byref(ties))
        return idx, d2, cnt, ties.value

    def associate(self, x0, strict: bool = False):
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        nb = np.zeros(4, np.int64)
        ties = np.zeros(3, np.int64)
        self.lib.orc_associate(self.h, _d(x0), int(strict), nb.ctypes.data_as(_i64p), ties.ctypes.data_as(_i64p))
        return nb, ties

    def block_keys(self):
        n = self.lib.orc_num_blocks(self.h)
        keys = np.zeros((n, 3), np.int32)
        for i in range(n):
            self.lib.orc_block_key(self.h, i, keys[i].ctypes.data_as(_i32p))
        return keys

    def block_eval(self, i: int, x, plain: bool = False):
        x = np.ascontiguousarray(x, dtype=np.float64)
        e = np.zeros(2 * _abi.STL_MAX_COVIS)
        J = np.zeros((2 * _abi.STL_MAX_COVIS, 7))
        if plain:
            nr = self.lib.orc_block_eval_plain(self.h, i, _d(x), _d(e))
            return e[:nr], None
        nr = self.lib.orc_block_eval(self.h, i, _d(x), _d(e), _d(J))
        return e[:nr], J[:nr]

    def set_gpr_hyper(self, sigma_l):
        a = np.ascontiguousarray(sigma_l, dtype=np.float64).reshape(-1, 2)
        self.lib.orc_set_gpr_hyper(self.h, _d(a), a.shape[0])

    def gpr_train(self, g: int, x0):
        """Training pixels [n,2] and depths [n] of GPR block g at the association extrinsic x0."""
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        X, y = np.zeros((32, 2)), np.zeros(32)
        n = self.lib.orc_gpr_train(self.h, g, _d(x0), _d(X), _d(y))
        return X[:n].copy(), y[:n].copy()

    def linearize(self, x, nthreads: int = 1):
        """x: [B,7] -> [B,62] rows (cost, g[7], H[7,7], n_blocks_*, n_residuals).  nthreads = 1: one accumulator in
        block order (the goldens' order); otherwise the residual blocks of each x are evaluated by `nthreads`
        threads (0 = all), as Ceres does with options.num_threads (iba_local.cpp:439)."""
        x = np.ascontiguousarray(np.atleast_2d(x), dtype=np.float64)
        B = x.shape[0]
        out = (_abi.LinSums * B)()
        if nthreads == 1:
            self.lib.orc_linearize(self.h, _d(x), B, out)
        else:
            self.lib.orc_linearize_mt(self.h, _d(x), B, nthreads, out)
        return np.frombuffer(out, dtype=np.float64).reshape(B, _abi.STL_LIN_NSUMS).copy()


def sim3exp(x, kind="port"):
    lib = load(kind)
    x = np.ascontiguousarray(x, dtype=np.float64)
    R, t, s = np.zeros(9), np.zeros(3), C.c_double(0)
    lib.orc_sim3exp(_d(x), _d(R), _d(t), C.byref(s))
    return R.reshape(3, 3), t, s.value


def se3log(R, t, kind="port"):
    lib = load(kind)
    R = np.ascontiguousarray(R, dtype=np.float64).reshape(9)
    t = np.ascontiguousarray(t, dtype=np.float64)
    out = np.zeros(6)
    lib.orc_se3log(_d(R), _d(t), _d(out))
    return out


def plane_fit(pts, kind="port"):
    lib = load(kind)
    pts = np.ascontiguousarray(pts, dtype=np.float64).reshape(-1, 3)
    n = np.zeros(3)
    reg = C.c_double(0)
    lib.orc_plane_fit(_d(pts), pts.shape[0], _d(n), C.byref(reg))
    return n, reg.value


def gpr_hyper_loss(X, y, sigma, l, sigma_noise=1e-10, kind="port"):
    """GPRHyperLoss::Evaluate as coded (GPR.hpp:154-174) -> (cost, grad[2]) or None when the Cholesky fails."""
    lib = load(kind)
    X = np.ascontiguousarray(X, dtype=np.float64).reshape(-1, 2)
    y = np.ascontiguousarray(y, dtype=np.float64)
    cost, g = C.c_double(0), np.zeros(2)
    ok = lib.orc_gpr_hyper_loss(_d(X), _d(y), len(y), sigma_noise, sigma, l, C.byref(cost), _d(g))
    return (cost.value, g) if ok else None


def he_linearize(edges, x, kind="port"):
    """EdgeHE + EdgeRegulation problem (NLHECalib.hpp:27-116), g2o robust-kernel semantics -> ([B,62], chi2 [B,n])."""
    lib = load(kind)
    x = np.ascontiguousarray(np.atleast_2d(x), dtype=np.float64)
    B = x.shape[0]
    out = (_abi.LinSums * B)()
    chi2 = np.zeros((B, max(edges.n, 1)))
    c = edges.as_c()
    lib.orc_he_linearize(C.byref(c), _d(x), B, out, _d(chi2))
    return np.frombuffer(out, dtype=np.float64).reshape(B, _abi.STL_LIN_NSUMS).copy(), chi2[:, : edges.n]


def calib_linearize(edges, x, kind="port"):
    lib = load(kind)
    x = np.ascontiguousarray(np.atleast_2d(x), dtype=np.float64)
    B = x.shape[0]
    out = (_abi.LinSums * B)()
    chi2 = np.zeros((B, max(edges.n_edges, 1)))
    c = edges.as_c()
    lib.orc_calib_linearize(C.byref(c), _d(x), B, out, _d(chi2))
    return np.frombuffer(out, dtype=np.float64).reshape(B, _abi.STL_LIN_NSUMS).copy(), chi2[:, : edges.n_edges]


def he_edge(Ta, Tb, x, kind="port"):
    lib = load(kind)
    Ta, Tb, x = (np.ascontiguousarray(a, dtype=np.float64).reshape(-1) for a in (Ta, Tb, x))
    e, J = np.zeros(3), np.zeros((3, 7))
    lib.orc_he_edge(_d(Ta), _d(Tb), _d(x), _d(e), _d(J))
    return e, J


def calib_edge(x, Xw, Tlw_quat, intr, obs, kind="port"):
    lib = load(kind)
    a = [np.ascontiguousarray(v, dtype=np.float64).reshape(-1) for v in (x, Xw, Tlw_quat, intr, obs)]
    err = np.zeros(2)
    lib.orc_calib_edge_plain(*[_d(v) for v in a], _d(err))
    return err


def rotvec(R, kind="port"):
    lib = load(kind)
    R = np.ascontiguousarray(R, dtype=np.float64).reshape(9)
    rv = np.zeros(3)
    lib.orc_rotvec(_d(R), _d(rv))
    return rv
