"""ctypes binding of libekfslam.so (include/ekfslam.h).

There is no CPU fallback: if the shared library is missing the import of any compute entry
point raises, and if no CUDA device is visible ``ekfslam_create`` returns ERR_NODEVICE which
surfaces as :class:`EkfSlamError`.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libekfslam.so")

# flag bits / feature types (include/ekfslam.h)
FEAT_NONE, FEAT_INVERSEDEPTH, FEAT_CARTESIAN = 0, 1, 2
F_HAS_H, F_HAS_Z, F_IC, F_LI, F_HI, F_CAND = 1, 2, 4, 8, 16, 32


class EkfSlamError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libekfslam error %d: %s" % (code, msg))
        self.code = code


class Camera(C.Structure):
    _fields_ = [("k1", C.c_double), ("k2", C.c_double), ("Cx", C.c_double), ("Cy", C.c_double),
                ("f", C.c_double), ("dx", C.c_double), ("dy", C.c_double),
                ("nRows", C.c_int32), ("nCols", C.c_int32)]


class Params(C.Structure):
    _fields_ = [("std_a", C.c_double), ("std_alpha", C.c_double), ("std_z", C.c_double),
                ("delta_t", C.c_double), ("chi2_gate", C.c_double), ("p_spurious_free", C.c_double),
                ("max_hyp", C.c_int32), ("fixed_hyp", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("n_ic", C.c_int32), ("ransac_iters", C.c_int32), ("ransac_scored", C.c_int32),
                ("max_support", C.c_int32), ("n_li", C.c_int32), ("n_hi", C.c_int32),
                ("status", C.c_int32), ("reserved", C.c_int32)]


STATS_FIELDS = [f[0] for f in Stats._fields_]


class Eval(C.Structure):
    _fields_ = [("pos_sq_err", C.c_double), ("rot_sq_err", C.c_double), ("nees_pos", C.c_double),
                ("nees_pose", C.c_double), ("map_sq_err", C.c_double), ("map_nees", C.c_double),
                ("n_map", C.c_int32), ("n_skip", C.c_int32), ("frames", C.c_int32), ("status", C.c_int32)]


EVAL_FIELDS = [f[0] for f in Eval._fields_]
# ekfslam_eval.status bits
EVAL_CAM_NOT_SPD, EVAL_NO_TRUTH, EVAL_NOT_EVALUABLE = 1, 2, 4
# per-filter status of ekfslam_update_camera
CAM_APPLIED, CAM_OFF, CAM_GATED, CAM_NOT_SPD = 0, 1, 2, 3


class WorldParams(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("b_offset", C.c_int32), ("flaky_mod", C.c_int32), ("noise_px", C.c_double),
                ("gross_px", C.c_double), ("p_outlier", C.c_double), ("p_flaky", C.c_double), ("band_px", C.c_double)]

_P = C.c_void_p
_I = C.c_int
_SIGS = {
    "ekfslam_last_error": (C.c_char_p, []),
    "ekfslam_version": (_I, []),
    "ekfslam_device_count": (_I, []),
    "ekfslam_default_camera": (None, [C.POINTER(Camera)]),
    "ekfslam_default_params": (None, [C.POINTER(Params)]),
    "ekfslam_create": (_I, [C.POINTER(_P), _I, _I, _I, _I]),
    "ekfslam_destroy": (_I, [_P]),
    "ekfslam_set_stream": (_I, [_P, _P]),
    "ekfslam_set_camera": (_I, [_P, C.POINTER(Camera)]),
    "ekfslam_set_params": (_I, [_P, C.POINTER(Params)]),
    "ekfslam_synchronize": (_I, [_P]),
    "ekfslam_dims": (_I, [_P, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I), C.POINTER(_I)]),
    "ekfslam_device_bytes": (C.c_int64, [_P]),
    "ekfslam_launch_count": (C.c_int64, [_P]),
    "ekfslam_upload_state": (_I, [_P, _I, _I, _I, _P, _P, _P]),
    "ekfslam_download_state": (_I, [_P, _I, _I, _I, _P, _P, _P]),
    "ekfslam_upload_feature_types": (_I, [_P, _I, _I, _P, _P]),
    "ekfslam_upload_matches": (_I, [_P, _I, _I, _P, _P]),
    "ekfslam_upload_candidates": (_I, [_P, _I, _I, _P, _P]),
    "ekfslam_upload_uniforms": (_I, [_P, _I, _I, _P, _I]),
    "ekfslam_download_features": (_I, [_P, _I, _I, _P, _P, _P, _P, _P, _P, _P]),
    "ekfslam_upload_features": (_I, [_P, _I, _I, _P, _P, _P, _P, _P]),
    "ekfslam_download_feature_types": (_I, [_P, _I, _I, _P, _P]),
    "ekfslam_download_stats": (_I, [_P, _I, _I, _P]),
    "ekfslam_begin_frame": (_I, [_P]),
    "ekfslam_predict": (_I, [_P]),
    "ekfslam_measure": (_I, [_P, _I]),
    "ekfslam_features": (_I, [_P, _I, _I]),
    "ekfslam_hp": (_I, [_P, _I, _I]),
    "ekfslam_innovation": (_I, [_P]),
    "ekfslam_gate": (_I, [_P]),
    "ekfslam_apply_matches": (_I, [_P]),
    "ekfslam_ransac": (_I, [_P]),
    "ekfslam_update_li": (_I, [_P]),
    "ekfslam_rescue": (_I, [_P]),
    "ekfslam_update_hi": (_I, [_P]),
    "ekfslam_update_masked": (_I, [_P, _I, _I]),
    "ekfslam_update_iterated": (_I, [_P, _I, _I, _I]),
    "ekfslam_step": (_I, [_P, _I, _I]),
    "ekfslam_step_graph": (_I, [_P, _I, _I]),
    "ekfslam_stage_frame": (_I, [_P, _P, _P, _P, _I]),
    "ekfslam_step_host": (_I, [_P, _I, _P, _P, _P, _I, _P, _P, _P]),
    "ekfslam_reset_filters": (_I, [_P, _I, _I, _P, _P]),
    "ekfslam_inversedepth_2_cartesian": (_I, [_P, C.c_double, _I, _P]),
    "ekfslam_delete_features": (_I, [_P, _I, _I, _P]),
    "ekfslam_add_features": (_I, [_P, _I, _I, _P, _P, C.c_double, C.c_double, C.c_double]),
    "ekfslam_map_management": (_I, [_P, _I]),
    "ekfslam_upload_detections": (_I, [_P, _I, _I, _I, _P, _P, _P]),
    "ekfslam_download_detections": (_I, [_P, _I, _I, _I, _P, _P, _P]),
    "ekfslam_upload_feature_meta": (_I, [_P, _I, _I, _P, _P]),
    "ekfslam_download_feature_tags": (_I, [_P, _I, _I, _P]),
    "ekfslam_download_candidates": (_I, [_P, _I, _I, _P, _P]),
    "ekfslam_world_upload": (_I, [_P, _I, _I, _P, _P, C.POINTER(WorldParams)]),
    "ekfslam_world_candidates": (_I, [_P, _I]),
    "ekfslam_world_detect": (_I, [_P, _I, _I]),
    "ekfslam_world_uniforms": (_I, [_P, _I, _I]),
    "ekfslam_download_uniforms": (_I, [_P, _I, _I, _P, _I]),
    "ekfslam_evaluate": (_I, [_P, _I]),
    "ekfslam_download_eval": (_I, [_P, _I, _I, _I, _P, _P, _P]),
    "ekfslam_reset_eval": (_I, [_P]),
    "ekfslam_map_cartesian": (_I, [_P, _I, _I, _P, _P]),
    "ekfslam_update_camera": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, C.c_double, _I]),
    "ekfslam_download_camera_update": (_I, [_P, _I, _I, _P, _P]),
    "ekfslam_device_ptr": (_P, [_P, C.c_char_p]),
    "ekfslam_enable_timing": (_I, [_P, _I]),
    "ekfslam_kernel_count": (_I, []),
    "ekfslam_kernel_time": (_I, [_P, _I, C.c_char_p, _I, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "ekfslam_bind_frame": (_I, [_P, _P, _P, _P, _I]),
    "ekfslam_unbind_frame": (_I, [_P]),
}

EXPORTS = sorted(_SIGS)
_lib = None


def load():
    """Loads libekfslam.so (built in-tree by __graft_entry__.build() / csrc/build.sh)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EkfSlamError(-5, "%s not found - build it with ekf-slam_b200/csrc/build.sh "
                               "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)  # AttributeError here = header / library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code):
    if code != 0:
        raise EkfSlamError(code, load().ekfslam_last_error().decode("utf-8", "replace"))
