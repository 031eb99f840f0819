"""Generates the stored vectors of tests/test_oracle_pin.py and tests/test_oracle_refmath.py
(tests/golden/pin/: pin_small.npz, pin_ties.npz, refmath.npz).

Every expected value comes from the original project's code when oracle/_ref is built (its vendored
nanoflann for the neighbour searches, its own source lines for the arithmetic), otherwise from the
in-repo restatement; the fixture records which in `backend`.  The inputs come from the seeded generators below
(the tests rebuild them and check them against the stored `input_digest`); outputs are stored as arrays where small
and as oracle.digest() of their exact bytes where large.

    python tests/golden/pin/make_pin_golden.py
"""
import ctypes as C
import importlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, ROOT)
PKG = "spatial-temporal-lidar-camera-calibration_b200"
synth = importlib.import_module(PKG + ".synth")
from oracle import oracle as O  # noqa: E402

KNN_K = (1, 5, 20, 30)
TIE_K = (1, 4, 30)
FRAME_KEYS = ("corr_kp", "corr_pt", "align_nn", "align_m", "align_is_plane", "align_knn", "align_dist", "align_normal")
_dp, _u32p = C.POINTER(C.c_double), C.POINTER(C.c_uint32)


def _d(a):
    return a.ctypes.data_as(_dp)


def knn_queries(P, k):
    """Near the surface, exactly on data points, and far / outside the bounding box."""
    rng = np.random.default_rng(k)
    return np.concatenate([P[rng.choice(len(P), 300)] + rng.normal(0, 0.05, (300, 3)),
                           P[rng.choice(len(P), 200)],
                           rng.uniform(-120, 120, (100, 3))])


def tie_pack():
    """Every point twice and many sharing a coordinate: exact distance ties."""
    pack, _, _ = synth.generate(n_kf=1, beams=8, az_steps=300, n_kp=50, seed=5)
    xyz = pack.scan_xyz.copy()
    n = len(xyz)
    xyz[n // 2:] = xyz[: n - n // 2]
    xyz[:, 2] = np.round(xyz[:, 2], 1)
    pack.scan_xyz = np.ascontiguousarray(xyz)
    return pack


def pack_digest(pack):
    return O.digest(*pack.to_npz_dict().values())


def pin_inputs():
    """Two keyframes of 32-beam scans, four candidates."""
    pack, x_gt, _ = synth.generate(n_kf=2, beams=32, az_steps=600, n_kp=500, seed=1000)
    return pack, synth.candidates(x_gt, 4, spread=0.5)


def make_pin(kind):
    pack, X = pin_inputs()
    orc = O.Oracle(pack, kind=kind)
    out = dict(X=X, input_digest=np.uint64(pack_digest(pack)), backend=np.array(orc.kind))
    P = pack.scan_xyz[: int(pack.scan_offset[1])].astype(np.float64)
    for k in KNN_K:
        q = knn_queries(P, k)
        out[f"knn{k}"] = np.uint64(O.digest(q, *orc.knn3d(0, q, k, strict=True)[:3]))
    sums, ties, cnt = orc.ba_error_sums(X, mode=0)
    assert ties.sum() == 0, "the fixture must be free of exact KNN ties"
    out.update(sums=sums, counters=cnt, sums_strict=orc.ba_error_sums(X, mode=0, strict=True)[0])
    for kf in range(pack.n_kf):
        d = orc.frame_debug(X[1], kf)
        out.update({f"kf{kf}_{key}": np.uint64(O.digest(d[key])) for key in FRAME_KEYS})
    nb, _ = orc.associate(X[0])
    out.update(lm_nblocks=nb, lm_keys=orc.block_keys(), lm_lin=orc.linearize(X[:2]))
    np.savez_compressed(os.path.join(HERE, "pin_small.npz"), **out)

    tp = tie_pack()
    orc = O.Oracle(tp, kind=kind)
    out = dict(input_digest=np.uint64(pack_digest(tp)), backend=np.array(orc.kind))
    q = tp.scan_xyz[::7].astype(np.float64)
    for k in TIE_K:
        out[f"tie{k}"] = np.uint64(O.digest(*orc.knn3d(0, q, k, strict=True)[:2]))
    np.savez_compressed(os.path.join(HERE, "pin_ties.npz"), **out)


def refmath_inputs():
    """Covariance / smallest-eigenvector trials (near a plane, general, nearly collinear, axis-aligned grid) and
    Sim3Exp / SE3Exp arguments (every fifth in the Taylor branch)."""
    rng = np.random.default_rng(0)
    pts, idx, off, kinds = [], [], [0], []
    for trial in range(400):
        m = int(rng.integers(3, 31))
        kind = trial % 4
        if kind == 0:
            nrm = rng.normal(size=3); nrm /= np.linalg.norm(nrm)
            P = rng.normal(0, 0.3, (m, 3)); P -= np.outer(P @ nrm, nrm) * 0.98
        elif kind == 1:
            P = rng.normal(0, 0.3, (m, 3))
        elif kind == 2:
            d = rng.normal(size=3); P = np.outer(rng.normal(0, 0.5, m), d) + rng.normal(0, 1e-3, (m, 3))
        else:
            P = np.zeros((m, 3)); P[:, trial % 3] = np.arange(m) * 0.1
        pts.append((P + rng.uniform(-30, 30, 3)).astype(np.float32).astype(np.float64))   # scan coordinates are float32 values
        idx.append(rng.permutation(m).astype(np.uint32))
        off.append(off[-1] + m)
        kinds.append(kind)
    rng = np.random.default_rng(1)
    xs = []
    for trial in range(300):
        x = np.concatenate([rng.normal(0, 1.0, 3), rng.normal(0, 0.5, 3), [rng.uniform(0.5, 30)]])
        if trial % 5 == 0:
            x[:3] *= 1e-5
        xs.append(x)
    return (np.concatenate(pts), np.concatenate(idx), np.array(off, np.int64), np.array(kinds, np.int32), np.array(xs))


def sim3_se3(lib, pre, x):
    """Sim3Exp(x) -> R, t, s; its dual with all 7 partials; SE3Exp(-x[0:6]) -> R, t.  `pre`: "refm_" or "orc_"."""
    x = np.ascontiguousarray(x)
    R, t, s, dual, Rm, tm = np.zeros(9), np.zeros(3), C.c_double(0), np.zeros(13 * 8), np.zeros(9), np.zeros(3)
    getattr(lib, pre + "sim3exp")(_d(x), _d(R), _d(t), C.byref(s))
    getattr(lib, pre + "sim3exp_dual")(_d(x), _d(dual))
    getattr(lib, pre + "se3exp")(_d(np.ascontiguousarray(-x[:6])), _d(Rm), _d(tm))
    return R, t, np.array([s.value]), dual, Rm, tm


def make_refmath():
    P, idx, off, kinds, xs = refmath_inputs()
    refm = O.load_refmath()
    port = O.load("port")
    n = len(off) - 1
    cov, ev = np.zeros((n, 6)), np.zeros((n, 3))
    for i in range(n):
        p, j, m = np.ascontiguousarray(P[off[i]:off[i + 1]]), np.ascontiguousarray(idx[off[i]:off[i + 1]]), int(off[i + 1] - off[i])
        if refm is not None:
            full = np.zeros(9)
            refm.refm_covariance(_d(p), m, j.ctypes.data_as(_u32p), m, _d(full))
            cov[i] = full.reshape(3, 3)[np.triu_indices(3)]
            refm.refm_fast_eigen(_d(full), _d(ev[i]), _d(np.zeros(3)))
        else:
            port.orc_covariance(_d(p), j.ctypes.data_as(_u32p), m, _d(cov[i]))
            port.orc_smallest_eigvec(_d(cov[i]), _d(ev[i]))
    lib = refm if refm is not None else port
    pre = "refm_" if refm is not None else "orc_"
    exp = np.zeros(len(xs), np.uint64)
    for i, x in enumerate(xs):
        exp[i] = O.digest(*sim3_se3(lib, pre, x))
    backend = "reference source lines (oracle/_ref/liboracle_refmath.so)" if refm is not None else port.orc_backend().decode()
    np.savez_compressed(os.path.join(HERE, "refmath.npz"), input_digest=np.uint64(O.digest(P, idx, off, kinds, xs)),
                        cov=cov, ev=ev, exp=exp, backend=np.array(backend))


if __name__ == "__main__":
    kind = "ref" if O.have_ref() else "port"
    make_pin(kind)
    make_refmath()
    for f in ("pin_small.npz", "pin_ties.npz", "refmath.npz"):
        print(f, os.path.getsize(os.path.join(HERE, f)), "bytes, backend", np.load(os.path.join(HERE, f))["backend"])
