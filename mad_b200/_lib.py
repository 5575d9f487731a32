"""ctypes binding of libmad_b200.so (the C ABI of include/mad_b200.h).

There is NO fallback: if the CUDA library is missing this module raises at import, and every
wrapper raises ``MadError`` when a call returns a non-zero status.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libmad_b200.so")


class MadError(RuntimeError):
    pass


if not os.path.exists(LIB_PATH):
    raise ImportError(
        "mad_b200: %s is missing -- build the CUDA library first (python -m mad_b200.build). "
        "There is no CPU fallback." % LIB_PATH)

lib = C.CDLL(LIB_PATH)

KEYPOINT_DTYPE = np.dtype([("vox", "<i4", 3), ("oct", "<i4"), ("off", "<f4", 3), ("val", "<f4"),
                           ("peak", "<i4", 3), ("accepted", "<i4")])
ORIENTED_DTYPE = np.dtype([("kp", "<i4"), ("main", "<i2"), ("sec", "<i2")])
assert KEYPOINT_DTYPE.itemsize == 48 and ORIENTED_DTYPE.itemsize == 8
MAX_ORI = 36
DSC_LEN = 1024
DSC_REFUSED = 1 << 30          # max_entry of a set that is not a descriptor set (negative entry / squared norm >= 2^31)
TOPK_INCOMPLETE = -2           # top-k index of an incomplete list (kernel hand-off time-out): discard the result
TOPK_MAX = 32
ZONE_FAST_BYTES = 2048


class MadZoneTable(C.Structure):
    _fields_ = [("n_zones", C.c_int32), ("n_belts", C.c_int32), ("bounds", C.c_void_p),
                ("belt_first", C.c_void_p), ("belt_phi", C.c_void_p), ("fast", C.c_void_p)]


class MadDscSet(C.Structure):
    _fields_ = [("dsc", C.c_void_p), ("half", C.c_void_p), ("norm2", C.c_void_p), ("u8", C.c_void_p),
                ("rnorm", C.c_void_p), ("rows", C.c_int32), ("rows_padded", C.c_int32), ("max_entry", C.c_int32),
                ("max_norm2", C.c_int32)]


_P = C.c_void_p
_I = C.c_int
_SZ = C.c_size_t

# name -> (restype, argtypes); must list every symbol include/mad_b200.h declares
SIGNATURES = {
    "mad_last_error_string": (C.c_char_p, []),
    "mad_version": (_I, []),
    "mad_device_info": (_I, [C.POINTER(_I), C.POINTER(_I), C.POINTER(_I)]),
    "mad_launch_count": (C.c_longlong, []),
    "mad_profile_enable": (_I, [_I]),
    "mad_profile_count": (_I, []),
    "mad_profile_get": (_I, [_I, C.POINTER(C.c_char_p), C.POINTER(C.c_float)]),
    "mad_profile_reset": (_I, []),
    "mad_publish_small": (_I, [_P, _P, _I, _P]),
    "mad_copy_to_host": (_I, [_P, _P, C.c_longlong, _I, _P]),
    "mad_zone_fast_build": (_I, [C.POINTER(MadZoneTable), _P, _P]),
    "mad_grid_max": (_I, [_P, C.c_longlong, _P, _P]),
    "mad_grid_max_decode": (C.c_float, [C.c_uint]),
    "mad_threshold_normalise": (_I, [_P, C.c_longlong, C.c_float, C.c_float, _I, _P]),
    "mad_grid_bbox": (_I, [_P, _I, _I, _I, _P, _P]),
    "mad_crop_pad3d": (_I, [_P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P]),
    "mad_pad3d": (_I, [_P, _I, _I, _I, _I, _P, _P]),
    "mad_upsample_workspace_bytes": (_SZ, [_I, _I, _I]),
    "mad_upsample_presmooth": (_I, [_P, _I, _I, _I, _P, _I, _P, _P, _SZ, _P]),
    "mad_log_gauss_workspace_bytes": (_SZ, [_I, _I, _I]),
    "mad_log_gauss": (_I, [_P, _I, _I, _I, _P, _P, _I, C.c_float, _P, _P, _P, _SZ, _I, _P]),
    "mad_gradient": (_I, [_P, _I, _I, _I, _P, _P]),
    "mad_gradient_tiles": (_SZ, [_I, _I, _I]),
    "mad_gradient_mark": (_I, [_P, _I, _P, _I, _I, _P, _P, _P]),
    "mad_gradient_masked": (_I, [_P, _I, _I, _I, _P, _P, _P]),
    "mad_detect": (_I, [_P, _I, _I, _I, _I, _I, C.c_float, _P, _I, _P, _P]),
    "mad_sort_keypoints_workspace_bytes": (_SZ, [_I]),
    "mad_sort_keypoints": (_I, [_P, _I, _P, _P, _P, _P, _SZ, _P]),
    "mad_orient": (_I, [_P, _P, _P, _P, _I, _I, C.POINTER(MadZoneTable), _P, _I, _I, _P, _P, _P]),
    "mad_compact_oriented_workspace_bytes": (_SZ, [_I]),
    "mad_compact_oriented": (_I, [_P, _P, _I, _P, _I, _P, _P, _SZ, _P]),
    "mad_describe": (_I, [_P, _P, _P, _P, _P, _I, _I, C.POINTER(MadZoneTable), _P, _P, _I, _P, _P]),
    "mad_dsc_prepare": (_I, [_P, _I, _I, _P, _P, _P, _P, _P, _P]),
    "mad_match_pairs": (_I, [C.POINTER(MadDscSet), C.POINTER(MadDscSet), C.c_double, _P, _P, C.c_uint64, _P, _P]),
    "mad_match_pairs_finish_workspace_bytes": (_SZ, [C.c_longlong]),
    "mad_match_pairs_finish": (_I, [_P, _P, C.c_longlong, _I, _I, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "mad_match_pairs_finish_dot": (_I, [_P, _P, C.c_longlong, _I, _I, _P, _P, _P, _P, _SZ, _P]),
    "mad_dsc_norms": (_I, [_P, _I, _P, _P]),
    "mad_dsc_to_half": (_I, [_P, _I, _I, _P, _P]),
    "mad_match_segments": (_I, [_I, _I, _I]),
    "mad_match_count": (_I, [C.POINTER(MadDscSet), C.POINTER(MadDscSet), C.c_double, _I, _P, _I, _P]),
    "mad_match_fill": (_I, [C.POINTER(MadDscSet), C.POINTER(MadDscSet), C.c_double, _I, _P, _P, _P, _P, _I, _P]),
    "mad_exclusive_scan_workspace_bytes": (_SZ, [_I]),
    "mad_exclusive_scan_i32_to_i64": (_I, [_P, _I, _P, _P, _P, _SZ, _P]),
    "mad_match_topk_workspace_bytes": (_SZ, [_I, _I, _I, _I]),
    "mad_match_topk": (_I, [C.POINTER(MadDscSet), C.POINTER(MadDscSet), _I, _I, _P, _P, _P, _SZ, _I, _P]),
    "mad_topk_merge": (_I, [_P, _P, _I, _I, _I, _P, _P, _P]),
    "mad_density_splat": (_I, [_P, _P, _I, _P, C.c_double, _I, _I, _I, _I, _P, _P]),
    "mad_normalise_f64": (_I, [_P, C.c_longlong, _P, _P]),
    "mad_conv_full_f64": (_I, [_P, C.c_longlong, _I, C.c_longlong, _P, _I, _P, _I, _P]),
    "mad_mark_used": (_I, [_P, C.c_longlong, _P, _P]),
    "mad_repeatability": (_I, [_P, _P, _P, C.c_longlong, _P, _P, _P, _P, _P, _P, _I, _P, _I, _P, _P, _P, _P, _P,
                               C.c_double, _P, _P]),
    "mad_repeat_counts": (_I, [_P, _P, C.c_longlong, C.c_longlong, _P, _P, _P, _P, _P, _P, _I, _P, _I, _P, _P, _P, _P, _P,
                               C.c_double, _P, _P]),
    "mad_repeat_rows": (_I, [_P, _P, _P, C.c_longlong, _P, _P, _P, _P, _P, _P, _I, _P, _I, _P, _P]),
    "mad_anchor_cloud_workspace_bytes": (_SZ, [_I]),
    "mad_anchor_cloud": (_I, [_P, _P, _I, C.c_double, _P, _P, _P, _P, _SZ, _P]),
    "mad_cloud_grid_workspace_bytes": (_SZ, [_I]),
    "mad_cloud_grid": (_I, [_P, _I, _P, _P, C.c_double, _P, _P, _P, _P, _SZ, _P]),
    "mad_box_scores_workspace_bytes": (_SZ, [_I, _I, _I]),
    "mad_box_scores": (_I, [_P, _I, _I, _I, _P, _I, _I, _I, _P, C.c_float, _P, _P, _SZ, _P]),
    "mad_grid_count_gt": (_I, [_P, C.c_longlong, C.c_float, _P, _P]),
    "mad_mask_with": (_I, [_P, _I, _I, _I, _P, _I, _I, _I, _P, _P, _P, _P]),
    "mad_refine_rigid": (_I, [_P, _I, _I, _I, _P, _P, _P, C.c_double, _P, _P, _P, _I, _I, _I, C.c_double, C.c_double,
                              _P, _P, _P]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _f = getattr(lib, _name)          # AttributeError here = the library does not export the ABI
    _f.restype = _res
    _f.argtypes = _args


def last_error():
    s = lib.mad_last_error_string()
    return s.decode() if s else ""


def check(rc, what):
    if rc != 0:
        raise MadError("%s failed with status %d: %s" % (what, rc, last_error()))


def call(name, *args):
    check(getattr(lib, name)(*args), name)
