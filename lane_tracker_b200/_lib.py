"""ctypes binding of liblane_tracker_b200.so (include/lane_tracker_b200.h).

There is no fallback: if the CUDA library is missing or cannot be loaded this
module raises, and every class of the package fails with it.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "liblane_tracker_b200.so")

LT_MAX_AVERAGE = 8
LT_MAX_PROFILES = 16
LT_MAX_CAMERAS = 64
LT_MAX_LEVELS = 128
LT_ABI_VERSION = 4
LT_NSTAGES = 16
# lt_import_states status codes
LT_RECORD_OK, LT_RECORD_BAD_HEADER, LT_RECORD_BAD_STATE = 0, 1, 2

i32, f64 = C.c_int32, C.c_double


class lt_config(C.Structure):
    _fields_ = [("img_w", i32), ("img_h", i32), ("bv_w", i32), ("bv_h", i32),
                ("cam_matrix", f64 * 9), ("dist_coeffs", f64 * 5), ("M", f64 * 9), ("Minv", f64 * 9),
                ("mppv", f64), ("mpph", f64),
                ("n_fail", i32), ("n_reset", i32), ("n_average", i32), ("print_frame_count", i32),
                ("max_streams", i32), ("device", i32)]


class lt_camera(C.Structure):
    _fields_ = [("cam_matrix", f64 * 9), ("dist_coeffs", f64 * 5), ("M", f64 * 9), ("Minv", f64 * 9),
                ("mppv", f64), ("mpph", f64)]


class lt_params(C.Structure):
    _fields_ = [("ksize_r", i32), ("C_r", i32), ("ksize_b", i32), ("C_b", i32), ("filter_type", i32),
                ("mask_noise", i32), ("noise_thresh", i32), ("ksize_noise", i32), ("C_noise", i32),
                ("window_width", i32), ("window_height", i32), ("search_range", i32), ("mu", f64),
                ("no_success_limit", i32), ("start_slice", f64), ("ignore_sides", i32),
                ("ignore_bottom", i32), ("bandwidth", i32), ("partial", f64), ("n_tries", i32)]


class lt_result(C.Structure):
    _fields_ = [("counter", i32), ("attempts", i32), ("search_mode", i32), ("detected_pixels", i32),
                ("valid_lane_lines", i32), ("last_detection", i32), ("drew_lane", i32),
                ("n_left", i32), ("n_right", i32), ("n_left_avg", i32), ("n_right_avg", i32),
                ("success", i32), ("fit_rank_deficient", i32),
                ("first_detected", i32), ("first_valid", i32), ("first_n_left", i32), ("first_n_right", i32),
                ("reserved0", i32),
                ("left_curve_radius", C.c_int64), ("right_curve_radius", C.c_int64), ("average_curve_radius", C.c_int64),
                ("left_fit", f64 * 3), ("right_fit", f64 * 3), ("left_avg", f64 * 3), ("right_avg", f64 * 3),
                ("eccentricity", f64), ("validity_d", f64 * 3),
                ("first_left_fit", f64 * 3), ("first_right_fit", f64 * 3)]


class lt_state(C.Structure):
    _fields_ = [("last_detection", i32), ("counter", i32), ("success", i32), ("ring_len", i32),
                ("ring_empty", i32 * LT_MAX_AVERAGE),
                ("ring_left", (f64 * 3) * LT_MAX_AVERAGE), ("ring_right", (f64 * 3) * LT_MAX_AVERAGE),
                ("has_last", i32), ("last_left", f64 * 3), ("last_right", f64 * 3),
                ("has_avg", i32), ("left_avg", f64 * 3), ("right_avg", f64 * 3),
                ("n_left_avg", i32), ("n_right_avg", i32), ("radii_len", i32),
                ("radii", C.c_int64 * LT_MAX_AVERAGE), ("average_curve_radius", C.c_int64), ("eccentricity", f64)]


class lt_validity(C.Structure):
    _fields_ = [("min_dist_y1", f64), ("max_dist_y1", f64), ("min_dist_y2", f64), ("max_dist_y2", f64),
                ("min_dist_y3", f64), ("max_dist_y3", f64), ("tangent_thresh", f64)]


# every symbol include/lane_tracker_b200.h declares: (restype, argtypes)
P = C.c_void_p
class lt_vis(C.Structure):
    _fields_ = [("mode", C.c_int32), ("n_left", C.c_int32), ("n_right", C.c_int32), ("n_rects", C.c_int32),
                ("bandwidth", C.c_int32), ("reserved0", C.c_int32), ("partial", C.c_double),
                ("band_left", C.c_double * 3), ("band_right", C.c_double * 3),
                ("left_fit", C.c_double * 3), ("right_fit", C.c_double * 3)]


SIGNATURES = {
    "lt_create": (C.c_int, [C.POINTER(lt_config), C.POINTER(P)]),
    "lt_destroy": (C.c_int, [P]),
    "lt_reset": (C.c_int, [P, C.POINTER(i32), i32]),
    "lt_set_validity": (C.c_int, [P, C.POINTER(lt_validity)]),
    "lt_get_validity": (C.c_int, [P, C.POINTER(lt_validity)]),
    "lt_last_error": (C.c_char_p, []),
    "lt_abi_version": (C.c_int, []),
    "lt_default_params": (None, [C.POINTER(lt_params)]),
    "lt_launch_count": (C.c_int64, []),
    "lt_process": (C.c_int, [P, P, P, i32, C.POINTER(lt_params), P, P]),
    "lt_process_front": (C.c_int, [P, P, i32, C.POINTER(lt_params), i32, P]),
    "lt_process_back": (C.c_int, [P, P, P, i32, C.POINTER(lt_params), i32, P, P]),
    "lt_process_streams": (C.c_int, [P, P, P, C.POINTER(i32), i32, C.POINTER(lt_params), P, P]),
    "lt_process_back_streams": (C.c_int, [P, P, P, C.POINTER(i32), i32, C.POINTER(lt_params), i32, P, P]),
    "lt_process_sequence": (C.c_int, [P, P, P, C.POINTER(i32), i32, C.POINTER(lt_params), P, P]),
    "lt_process_back_sequence": (C.c_int, [P, P, P, C.POINTER(i32), i32, C.POINTER(lt_params), i32, P, P]),
    "lt_set_profile": (C.c_int, [P, i32, C.POINTER(lt_params), C.POINTER(lt_validity)]),
    "lt_process_profiles": (C.c_int, [P, P, P, C.POINTER(i32), C.POINTER(i32), i32, P, P]),
    "lt_process_front_profiles": (C.c_int, [P, P, C.POINTER(i32), i32, i32, P]),
    "lt_process_back_profiles": (C.c_int, [P, P, P, C.POINTER(i32), C.POINTER(i32), i32, i32, P, P]),
    "lt_set_camera": (C.c_int, [P, i32, C.POINTER(lt_camera)]),
    "lt_process_cameras": (C.c_int, [P, P, P, C.POINTER(i32), C.POINTER(i32), i32, C.POINTER(lt_params), C.POINTER(i32),
                                     P, P]),
    "lt_process_front_cameras": (C.c_int, [P, P, C.POINTER(i32), i32, C.POINTER(lt_params), C.POINTER(i32), i32, P]),
    "lt_process_back_cameras": (C.c_int, [P, P, P, C.POINTER(i32), C.POINTER(i32), i32, C.POINTER(lt_params),
                                          C.POINTER(i32), i32, P, P]),
    "lt_set_capture": (C.c_int, [P, i32]),
    "lt_set_pixel_capacity": (C.c_int, [P, i32]),
    "lt_read_capture": (C.c_int, [P, i32, i32, i32, P, i32, C.POINTER(i32), P, C.POINTER(i32)]),
    "lt_set_text_sprites": (C.c_int, [P, P, i32, P, i32, P, P, P, i32, P, i32]),
    "lt_set_remap_mode": (C.c_int, [P, i32]),
    "lt_set_frame_format": (C.c_int, [P, i32]),
    "lt_memcpy_rows": (C.c_int, [P, P, P, i32, i32, i32, i32, P]),
    "lt_profile_begin": (C.c_int, [P, i32]),
    "lt_profile_read": (C.c_int, [P, C.POINTER(f64), C.POINTER(i32)]),
    "lt_profile_select": (C.c_int, [P, C.c_uint32]),
    "lt_stage_name": (C.c_char_p, [i32]),
    "lt_remap": (C.c_int, [P, P, P, i32, P]),
    "lt_filter_lane_points": (C.c_int, [P, P, P, i32] + [i32] * 9 + [P]),
    "lt_sliding_window_search": (C.c_int, [P, P, i32, i32, i32, i32, f64, i32, f64, i32, i32, f64,
                                           P, i32, P, P, P, P, P]),
    "lt_band_search": (C.c_int, [P, P, i32, P, i32, i32, f64, P, i32, P, P, P]),
    "lt_fit_poly": (C.c_int, [P, P, i32, P, i32, P, P]),
    "lt_check_validity": (C.c_int, [P, P, i32, P, P, P]),
    "lt_get_poly_points": (C.c_int, [P, P, i32, f64, P, P, P]),
    "lt_draw_lane": (C.c_int, [P, P, P, i32, P, P, P]),
    "lt_lane_metrics": (C.c_int, [P, P, P, P, i32, P, P, P]),
    "lt_bilateral_adaptive_threshold": (C.c_int, [P, i32, i32, C.c_int64, P, C.c_int64, i32, i32, i32, i32, i32, P]),
    "lt_draw_text": (C.c_int, [P, P, i32, P, P, P, P, P]),
    "lt_warp_frame": (C.c_int, [P, P, i32, P, P]),
    "lt_nv12_to_rgb": (C.c_int, [P, P, i32, i32, i32, P]),
    "lt_visualize_search": (C.c_int, [P, C.POINTER(lt_vis), P, P, P, P, P, P]),
    "lt_resize_linear": (C.c_int, [P, i32, i32, i32, C.c_int64, P, i32, i32, C.c_int64, P]),
    "lt_get_state": (C.c_int, [P, i32, C.POINTER(lt_state), P, P]),
    "lt_set_state": (C.c_int, [P, i32, C.POINTER(lt_state), P, P]),
    "lt_debug_read": (C.c_int64, [P, i32, i32, P, C.c_int64]),
    "lt_reset_async": (C.c_int, [P, C.POINTER(i32), i32, P]),
    "lt_state_record_bytes": (C.c_int64, [P]),
    "lt_export_states": (C.c_int, [P, C.POINTER(i32), i32, P, P]),
    "lt_import_states": (C.c_int, [P, C.POINTER(i32), i32, P, P, P]),
}

_lib = None


class LaneTrackerError(RuntimeError):
    pass


def load():
    """Load the CUDA library; raise loudly when it is absent (no CPU path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LaneTrackerError(
            "lane_tracker_b200: %s is missing. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError if the library does not export the symbol
        fn.restype = res
        fn.argtypes = args
    if lib.lt_abi_version() != LT_ABI_VERSION:
        raise LaneTrackerError("ABI version mismatch: library %d, binding %d" % (lib.lt_abi_version(), LT_ABI_VERSION))
    _lib = lib
    return lib


def check(rc):
    if rc < 0:
        msg = load().lt_last_error()
        raise LaneTrackerError("lane_tracker_b200 error %d: %s" % (rc, msg.decode() if msg else "?"))
    return rc
