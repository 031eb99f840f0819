"""ctypes mirror of include/stlcalib.h and include/stlsynth.h.

Only declarations live here: struct layouts, the symbol table of the C-ABI and
the loaders.  There is no compute and no fallback in this module: if
``libstlcalib.so`` (the CUDA library) is missing, :func:`load_calib` raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))

STL_MAX_COVIS = 10
STL_EVAL_NSUMS = 12
STL_LIN_NSUMS = 62
STL_STEP_NSUMS = STL_EVAL_NSUMS + STL_LIN_NSUMS
STL_COMM_ID_BYTES = 128
STL_MAX_PROBLEMS = 256
STL_NSTAGES = 8
STAGE_NAMES = ("assoc2d", "knn3d", "reduce", "linearize", "build", "assoc_lm", "allreduce", "plane_index")

STATUS = {0: "STL_OK", 1: "STL_ERR_INVALID", 2: "STL_ERR_CUDA", 3: "STL_ERR_NO_DEVICE",
          4: "STL_ERR_STATE", 5: "STL_ERR_CAPACITY"}


class StlError(RuntimeError):
    def __init__(self, code: int, msg: str = ""):
        self.code = code
        super().__init__(f"{STATUS.get(code, code)}: {msg}")


class Params(C.Structure):
    """stl_params_t (IBAGlobalParams iba_global.cpp:26-52, IBALocalParams IBACalib2.hpp:104-137)."""
    _fields_ = [
        ("max_pixel_dist", C.c_double),
        ("corr_3d_2d_threshold", C.c_double),
        ("corr_3d_3d_threshold", C.c_double),
        ("norm_radius", C.c_double),
        ("norm_reg_threshold", C.c_double),
        ("min_diff_dist", C.c_double),
        ("err_weight", C.c_double * 2),
        ("he_threshold", C.c_double),
        ("valid_rate", C.c_double),
        ("max_3d_dist", C.c_double),
        ("robust_kernel_delta", C.c_double),
        ("robust_kernel_3ddelta", C.c_double),
        ("num_min_corr", C.c_int32),
        ("norm_max_pts", C.c_int32),
        ("norm_min_pts", C.c_int32),
        ("use_plane", C.c_int32),
        ("use_gpr", C.c_int32),
        ("gpr_sigma", C.c_double),
        ("gpr_l", C.c_double),
        ("gpr_sigma_noise", C.c_double),
        ("plane_index", C.c_int32),
        ("variant", C.c_int32),
        ("gpr_optimize", C.c_int32),
        ("gpr_grad_flavour", C.c_int32),
    ]


class Pack(C.Structure):
    """stl_pack_t."""
    _fields_ = [
        ("n_kf", C.c_int32),
        ("n_covis", C.c_int32),
        ("scan_offset", C.POINTER(C.c_int64)),
        ("scan_xyz", C.POINTER(C.c_float)),
        ("intrinsics", C.POINTER(C.c_float)),
        ("image_wh", C.POINTER(C.c_int32)),
        ("kp_offset", C.POINTER(C.c_int64)),
        ("kp_xy", C.POINTER(C.c_float)),
        ("kp_mappoint", C.POINTER(C.c_float)),
        ("Tcw", C.POINTER(C.c_float)),
        ("covis_relpose", C.POINTER(C.c_float)),
        ("covis_valid", C.POINTER(C.c_uint8)),
        ("covis_uv", C.POINTER(C.c_float)),
        ("he_Tc", C.POINTER(C.c_float)),
        ("he_Tl", C.POINTER(C.c_double)),
        ("he_valid", C.POINTER(C.c_uint8)),
    ]


class EvalSums(C.Structure):
    _fields_ = [(n, C.c_double) for n in (
        "sum_3d2d", "sum_3d3d", "sum_he", "cnt_he", "cnt_3d2d", "valid_3d2d", "cnt_3d3d",
        "valid_3d3d", "valid_pl", "valid_pt", "n_frames", "n_corr")]


class BAErrorOut(C.Structure):
    _fields_ = [("f1", C.c_double), ("f2", C.c_double), ("C", C.c_double),
                ("valid_cnt_3d_2d", C.c_int32), ("cnt_3d_2d", C.c_int32)]


class LinSums(C.Structure):
    _fields_ = [("cost", C.c_double), ("g", C.c_double * 7), ("H", C.c_double * 49),
                ("n_blocks_2d", C.c_double), ("n_blocks_pt", C.c_double),
                ("n_blocks_pl", C.c_double), ("n_residuals", C.c_double), ("n_blocks_gpr", C.c_double)]


class StepSums(C.Structure):
    _fields_ = [("eval", EvalSums), ("lin", LinSums)]


class HeEdges(C.Structure):
    """stl_he_edges_t (NLHECalib.hpp:27-116)."""
    _fields_ = [("n", C.c_int32), ("Ta", C.POINTER(C.c_double)), ("Tb", C.POINTER(C.c_double)), ("info", C.POINTER(C.c_double)),
                ("huber_delta", C.c_double), ("regulation", C.c_double)]


class CalibEdges(C.Structure):
    """stl_calib_edges_t (Optimizer.cc:65-205,1399-1744)."""
    _fields_ = [("n_kf", C.c_int32), ("n_edges", C.c_int64), ("edge_offset", C.POINTER(C.c_int64)), ("Tlw_quat", C.POINTER(C.c_double)),
                ("intrinsics", C.POINTER(C.c_float)), ("Xw", C.POINTER(C.c_double)), ("obs", C.POINTER(C.c_double)),
                ("inv_sigma2", C.POINTER(C.c_float)), ("level", C.POINTER(C.c_uint8)), ("huber_delta", C.c_double)]


class SynthCfg(C.Structure):
    _fields_ = [
        ("n_kf", C.c_int32), ("kf_begin", C.c_int32), ("n_kf_total", C.c_int32),
        ("beams", C.c_int32), ("az_steps", C.c_int32), ("n_kp", C.c_int32), ("n_covis", C.c_int32),
        ("width", C.c_int32), ("height", C.c_int32),
        ("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float),
        ("anchored_frac", C.c_double), ("mappoint_frac", C.c_double), ("match_frac", C.c_double),
        ("outlier_frac", C.c_double), ("scale_gt", C.c_double), ("kf_spacing", C.c_double),
        ("max_range", C.c_double), ("elev_top_deg", C.c_double), ("elev_bottom_deg", C.c_double),
        ("x_gt", C.c_double * 7), ("seed", C.c_uint64),
    ]


_vp = C.c_void_p
_dp = C.POINTER(C.c_double)
_u32p = C.POINTER(C.c_uint32)
_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)
_u8p = C.POINTER(C.c_uint8)

# Every symbol include/stlcalib.h declares: name -> (restype, argtypes)
CALIB_SYMBOLS = {
    "stl_default_params": (None, [C.POINTER(Params)]),
    "stl_create": (C.c_int, [C.POINTER(Params), C.c_int32, C.POINTER(_vp)]),
    "stl_destroy": (None, [_vp]),
    "stl_last_error": (C.c_char_p, [_vp]),
    "stl_abi_version": (C.c_int32, []),
    "stl_upload_pack": (C.c_int, [_vp, C.POINTER(Pack)]),
    "stl_eval_batch": (C.c_int, [_vp, _dp, C.c_int32, C.POINTER(EvalSums)]),
    "stl_eval_batch_device": (C.c_int, [_vp, _dp, C.c_int32, _vp, _vp]),
    "stl_finalize": (None, [C.POINTER(Params), C.POINTER(EvalSums), C.POINTER(BAErrorOut)]),
    "stl_bbo": (None, [C.POINTER(Params), C.POINTER(BAErrorOut), _dp]),
    "stl_associate": (C.c_int, [_vp, _dp, _i64p]),
    "stl_linearize_batch": (C.c_int, [_vp, _dp, C.c_int32, C.POINTER(LinSums)]),
    "stl_linearize_batch_device": (C.c_int, [_vp, _dp, C.c_int32, _vp, _vp]),
    "stl_eval_blocks": (C.c_int, [_vp, _dp, C.c_int32, C.c_int64, _i32p, _i32p, _i32p, _i32p, _dp, _dp, C.POINTER(C.c_int64)]),
    "stl_block_counts": (C.c_int, [_vp, _i64p]),
    "stl_gpr_nlml": (C.c_int, [_dp, _dp, C.c_int32, C.c_double, C.c_double, C.c_double, C.c_int32, _dp, _dp]),
    "stl_gpr_fit": (C.c_int, [_dp, _dp, C.c_int32, C.c_double, C.c_double, C.c_double, C.c_int32, C.c_int32, _dp]),
    "stl_gpr_hyper": (C.c_int, [_vp, _dp, C.c_int64]),
    "stl_step_batch": (C.c_int, [_vp, _dp, C.c_int32, C.c_int32, C.POINTER(StepSums)]),
    "stl_step_batch_device": (C.c_int, [_vp, _dp, C.c_int32, C.c_int32, _vp, _vp]),
    "stl_associate_multi": (C.c_int, [_vp, _dp, C.c_int32, _u8p, _i64p]),
    "stl_block_counts_multi": (C.c_int, [_vp, _i64p, C.c_int32]),
    "stl_linearize_multi": (C.c_int, [_vp, _dp, C.c_int32, _i32p, C.POINTER(LinSums)]),
    "stl_linearize_multi_device": (C.c_int, [_vp, _dp, C.c_int32, _i32p, _vp, _vp]),
    "stl_linearize_frames": (C.c_int, [_vp, _dp, C.c_int32, _i32p, C.POINTER(LinSums)]),
    "stl_step_multi": (C.c_int, [_vp, _dp, C.c_int32, _u8p, C.POINTER(StepSums)]),
    "stl_step_multi_device": (C.c_int, [_vp, _dp, C.c_int32, _u8p, _vp, _vp]),
    "stl_he_linearize": (C.c_int, [_vp, C.POINTER(HeEdges), _dp, C.c_int32, C.POINTER(LinSums), _dp]),
    "stl_calib_linearize": (C.c_int, [_vp, C.POINTER(CalibEdges), _dp, C.c_int32, C.POINTER(LinSums), _dp]),
    "stl_comm_unique_id": (C.c_int, [C.POINTER(C.c_uint8)]),
    "stl_comm_init": (C.c_int, [_vp, C.POINTER(C.c_uint8), C.c_int32, C.c_int32]),
    "stl_comm_info": (C.c_int, [_vp, _i32p, _i32p]),
    "stl_comm_stats": (C.c_int, [_vp, _i64p]),
    "stl_select_keyframes": (C.c_int, [_vp, _i32p, C.c_int32]),
    "stl_eval_frames": (C.c_int, [_vp, _dp, C.c_int32, _dp]),
    "stl_allow_oversize_keyframes": (C.c_int, [_vp, C.c_int32]),
    "stl_oversize_keyframes": (C.c_int, [_vp, _i32p, C.c_int32, _i32p]),
    "stl_debug_corrset": (C.c_int, [_vp, C.c_int32, C.c_int32, _u32p, _u32p, C.c_int32, _i32p]),
    "stl_debug_align": (C.c_int, [_vp, C.c_int32, C.c_int32, _u32p, _u32p, _i32p, _i32p, _dp, _u32p,
                                  C.c_int32, _i32p]),
    "stl_debug_frame": (C.c_int, [_vp, C.c_int32, C.c_int32, _dp]),
    "stl_debug_trig": (C.c_int, [_vp, _dp, C.c_int32, _dp, _dp]),
    "stl_knn3d": (C.c_int, [_vp, C.c_int32, _dp, C.c_int32, C.c_int32, C.c_double, _u32p, _dp, _i32p]),
    "stl_set_stream": (C.c_int, [_vp, _vp]),
    "stl_set_profiling": (C.c_int, [_vp, C.c_int32]),
    "stl_stage_stats": (C.c_int, [_vp, _dp, _i64p]),
    "stl_work_counters": (C.c_int, [_vp, _dp]),
}

SYNTH_SYMBOLS = {
    "stl_synth_default_cfg": (None, [C.POINTER(SynthCfg)]),
    "stl_synth_create": (_vp, [C.POINTER(SynthCfg)]),
    "stl_synth_pack": (C.POINTER(Pack), [_vp]),
    "stl_synth_x_gt": (_dp, [_vp]),
    "stl_synth_Twl": (_dp, [_vp]),
    "stl_synth_destroy": (None, [_vp]),
    "stl_synth_candidates": (None, [_dp, C.c_uint64, C.c_int32, C.c_double, _dp]),
}


def _bind(lib, table):
    for name, (res, args) in table.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    return lib


CALIB_LIB_PATH = os.path.join(_HERE, "libstlcalib.so")
SYNTH_LIB_PATH = os.path.join(_HERE, "libstlsynth.so")

_calib = None
_synth = None


def load_calib():
    """Loads the CUDA library.  Raises (never falls back) if it is not built."""
    global _calib
    if _calib is None:
        if not os.path.exists(CALIB_LIB_PATH):
            raise ImportError(
                f"{CALIB_LIB_PATH} is not built; run `python -c 'import __graft_entry__ as g; g.build()'`."
                " There is no CPU fallback for the cost-evaluation path.")
        _calib = _bind(C.CDLL(CALIB_LIB_PATH), CALIB_SYMBOLS)
    return _calib


def load_synth():
    global _synth
    if _synth is None:
        if not os.path.exists(SYNTH_LIB_PATH):
            raise ImportError(f"{SYNTH_LIB_PATH} is not built; run __graft_entry__.build()")
        _synth = _bind(C.CDLL(SYNTH_LIB_PATH), SYNTH_SYMBOLS)
    return _synth
