"""KeyFramePack: the flattened, candidate-independent state the hot path reads.

Host-side container (numpy) of ``stl_pack_t`` (include/stlcalib.h).  It replaces
what the reference keeps in ``std::vector<VecVector3d> PointClouds``,
``std::vector<ORB_SLAM2::KeyFrame*> KeyFrames`` and ``vTwl``
(src/examples/iba_global.cpp:473-511).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, fields

import numpy as np

from . import _abi

_SPEC = {
    # name: (dtype, trailing shape builder)
    "scan_offset": np.int64, "scan_xyz": np.float32, "intrinsics": np.float32, "image_wh": np.int32,
    "kp_offset": np.int64, "kp_xy": np.float32, "kp_mappoint": np.float32, "Tcw": np.float32,
    "covis_relpose": np.float32, "covis_valid": np.uint8, "covis_uv": np.float32,
    "he_Tc": np.float32, "he_Tl": np.float64, "he_valid": np.uint8,
}


@dataclass
class KeyFramePack:
    n_kf: int
    n_covis: int
    scan_offset: np.ndarray    # [F+1] int64
    scan_xyz: np.ndarray       # [sumN,3] f32
    intrinsics: np.ndarray     # [F,4] f32
    image_wh: np.ndarray       # [F,2] i32
    kp_offset: np.ndarray      # [F+1] int64
    kp_xy: np.ndarray          # [sumK,2] f32
    kp_mappoint: np.ndarray    # [sumK,3] f32 (NaN = none)
    Tcw: np.ndarray            # [F,12] f32
    covis_relpose: np.ndarray  # [F,C,12] f32
    covis_valid: np.ndarray    # [F,C] u8
    covis_uv: np.ndarray       # [sumK,C,2] f32 (NaN = unmatched)
    he_Tc: np.ndarray          # [F,12] f32
    he_Tl: np.ndarray          # [F,12] f64
    he_valid: np.ndarray       # [F] u8

    def __post_init__(self):
        for name, dt in _SPEC.items():
            a = np.ascontiguousarray(getattr(self, name), dtype=dt)
            setattr(self, name, a)
        F, Cc = self.n_kf, self.n_covis
        nk = int(self.kp_offset[-1])
        npts = int(self.scan_offset[-1])
        self.scan_xyz = self.scan_xyz.reshape(npts, 3)
        self.intrinsics = self.intrinsics.reshape(F, 4)
        self.image_wh = self.image_wh.reshape(F, 2)
        self.kp_xy = self.kp_xy.reshape(nk, 2)
        self.kp_mappoint = self.kp_mappoint.reshape(nk, 3)
        self.Tcw = self.Tcw.reshape(F, 12)
        self.covis_relpose = self.covis_relpose.reshape(F, Cc, 12)
        self.covis_valid = self.covis_valid.reshape(F, Cc)
        self.covis_uv = self.covis_uv.reshape(nk, Cc, 2)
        self.he_Tc = self.he_Tc.reshape(F, 12)
        self.he_Tl = self.he_Tl.reshape(F, 12)
        self.he_valid = self.he_valid.reshape(F)

    # -- C view ---------------------------------------------------------
    def as_c(self) -> _abi.Pack:
        """ctypes view; the numpy arrays must outlive it (they are referenced, not copied)."""
        p = _abi.Pack()
        p.n_kf, p.n_covis = self.n_kf, self.n_covis
        for name, ctype in _abi.Pack._fields_[2:]:
            arr = getattr(self, name)
            setattr(p, name, arr.ctypes.data_as(ctype))
        p._keepalive = self
        return p

    @classmethod
    def from_c(cls, p: _abi.Pack, copy: bool = True) -> "KeyFramePack":
        F, Cc = p.n_kf, p.n_covis
        so = np.ctypeslib.as_array(p.scan_offset, (F + 1,))
        ko = np.ctypeslib.as_array(p.kp_offset, (F + 1,))
        npts, nk = int(so[-1]), int(ko[-1])
        shapes = {
            "scan_offset": (F + 1,), "scan_xyz": (max(npts, 1) * 3,), "intrinsics": (F * 4,),
            "image_wh": (F * 2,), "kp_offset": (F + 1,), "kp_xy": (max(nk, 1) * 2,),
            "kp_mappoint": (max(nk, 1) * 3,), "Tcw": (F * 12,), "covis_relpose": (max(F * Cc, 1) * 12,),
            "covis_valid": (max(F * Cc, 1),), "covis_uv": (max(nk * Cc, 1) * 2,), "he_Tc": (F * 12,),
            "he_Tl": (F * 12,), "he_valid": (F,),
        }
        sizes = {"scan_xyz": npts * 3, "kp_xy": nk * 2, "kp_mappoint": nk * 3,
                 "covis_relpose": F * Cc * 12, "covis_valid": F * Cc, "covis_uv": nk * Cc * 2}
        kw = {}
        for name, _ in _abi.Pack._fields_[2:]:
            ptr = getattr(p, name)
            if not ptr:  # stl_pack_t allows NULL for empty members (no keypoints, n_covis = 0)
                if sizes.get(name, 1) != 0:
                    raise ValueError(f"stl_pack_t.{name} is NULL")
                kw[name] = np.zeros(0, _SPEC[name])
                continue
            a = np.ctypeslib.as_array(ptr, shapes[name])
            a = a[: sizes.get(name, a.size)]
            kw[name] = a.copy() if copy else a
        return cls(n_kf=F, n_covis=Cc, **kw)

    # -- slicing / persistence --------------------------------------------
    def shard(self, begin: int, end: int) -> "KeyFramePack":
        """Keyframes [begin, end) as a self-contained pack (keyframe sharding, SURVEY §8e).

        Covisible data is baked per keyframe, so no halo is needed.  ``he_valid`` already
        encodes whether a *global* successor exists, so the last keyframe of a shard keeps
        its hand-eye term."""
        so, ko = self.scan_offset, self.kp_offset
        s0, s1, k0, k1 = int(so[begin]), int(so[end]), int(ko[begin]), int(ko[end])
        return KeyFramePack(
            n_kf=end - begin, n_covis=self.n_covis,
            scan_offset=so[begin:end + 1] - s0, scan_xyz=self.scan_xyz[s0:s1],
            intrinsics=self.intrinsics[begin:end], image_wh=self.image_wh[begin:end],
            kp_offset=ko[begin:end + 1] - k0, kp_xy=self.kp_xy[k0:k1], kp_mappoint=self.kp_mappoint[k0:k1],
            Tcw=self.Tcw[begin:end], covis_relpose=self.covis_relpose[begin:end],
            covis_valid=self.covis_valid[begin:end], covis_uv=self.covis_uv[k0:k1],
            he_Tc=self.he_Tc[begin:end], he_Tl=self.he_Tl[begin:end], he_valid=self.he_valid[begin:end])

    def select(self, kf) -> "KeyFramePack":
        """The keyframes ``kf`` (strictly increasing indices into this pack) as a self-contained pack: ``shard`` for any
        index list, ``shard(b, e) == select(range(b, e))``.

        Every keyframe keeps its own rows, its hand-eye pair (f, f+1) included as ``he_valid`` bakes it, whether or not f+1
        is selected.  It is what a context computes over this pack after ``Context.select_keyframes(kf)``."""
        k = np.asarray(kf)
        if k.size == 0:
            k = k.astype(np.int64).reshape(0)
        if k.ndim != 1 or k.dtype.kind not in "iu":
            raise TypeError("select: kf must be a 1-D list of integer keyframe indices")
        k = k.astype(np.int64)
        if k.size and (k[0] < 0 or k[-1] >= self.n_kf):
            raise ValueError(f"select: keyframe indices must lie in [0, {self.n_kf})")
        if np.any(np.diff(k) <= 0):
            raise ValueError("select: keyframe indices must be strictly increasing")

        def rows(off):  # row indices of the selected keyframes and their new offsets
            n = off[k + 1] - off[k]
            new_off = np.concatenate(([0], np.cumsum(n))).astype(np.int64)
            return np.repeat(off[k] - new_off[:-1], n) + np.arange(new_off[-1], dtype=np.int64), new_off

        pts, so = rows(self.scan_offset)
        kps, ko = rows(self.kp_offset)
        return KeyFramePack(
            n_kf=int(k.size), n_covis=self.n_covis,
            scan_offset=so, scan_xyz=self.scan_xyz[pts],
            intrinsics=self.intrinsics[k], image_wh=self.image_wh[k],
            kp_offset=ko, kp_xy=self.kp_xy[kps], kp_mappoint=self.kp_mappoint[kps],
            Tcw=self.Tcw[k], covis_relpose=self.covis_relpose[k],
            covis_valid=self.covis_valid[k], covis_uv=self.covis_uv[kps],
            he_Tc=self.he_Tc[k], he_Tl=self.he_Tl[k], he_valid=self.he_valid[k])

    def to_npz_dict(self) -> dict:
        d = {f.name: getattr(self, f.name) for f in fields(self) if f.name not in ("n_kf", "n_covis")}
        d["n_kf"] = np.int64(self.n_kf)
        d["n_covis"] = np.int64(self.n_covis)
        return d

    @classmethod
    def from_npz_dict(cls, d) -> "KeyFramePack":
        kw = {k: d[k] for k in _SPEC}
        return cls(n_kf=int(d["n_kf"]), n_covis=int(d["n_covis"]), **kw)

    @property
    def n_points(self) -> int:
        return int(self.scan_offset[-1])

    @property
    def n_keypoints(self) -> int:
        return int(self.kp_offset[-1])

    def nbytes(self) -> int:
        return sum(getattr(self, n).nbytes for n in _SPEC)


def default_params() -> _abi.Params:
    """KITTI-00 values (config/calib/00/iba_calib_global.yml:21-48).  Pure-Python so that the
    CPU-only tests and the oracle do not need the CUDA library; tests check it against
    ``stl_default_params``."""
    p = _abi.Params()
    p.max_pixel_dist = 1.5
    p.corr_3d_2d_threshold = 40.0
    p.corr_3d_3d_threshold = 10.0
    p.norm_radius = 0.6
    p.norm_reg_threshold = 0.02
    p.min_diff_dist = 0.2
    p.err_weight[0], p.err_weight[1] = 1.0, 1.0
    p.he_threshold = 0.094
    p.valid_rate = 0.95
    p.max_3d_dist = 1.0
    p.robust_kernel_delta = 2.98
    p.robust_kernel_3ddelta = 1.0
    p.num_min_corr = 30
    p.norm_max_pts = 30
    p.norm_min_pts = 5
    p.use_plane = 1
    p.use_gpr = 0
    p.gpr_sigma, p.gpr_l, p.gpr_sigma_noise = 10.0, 10.0, 1e-10
    p.plane_index = 1
    p.variant = 0
    p.gpr_optimize = 0
    p.gpr_grad_flavour = 0
    return p
