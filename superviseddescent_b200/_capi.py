"""ctypes binding of the C ABI in include/sd_b200.h (libsd_b200.so).

There is no CPU fallback: if the shared object is missing, or no CUDA device is usable, every entry
point raises.  torch is used by callers only for device buffers / streams / torch.distributed.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libsd_b200.so")


class SdError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"sd_b200 error {code}: {msg}")
        self.code = code


class HogParam(C.Structure):
    """rcr::HoGParam (reference include/rcr/adaptive_vlhog.hpp:41-60)."""
    _fields_ = [("variant", C.c_int32), ("num_cells", C.c_int32), ("cell_size", C.c_int32),
                ("num_bins", C.c_int32), ("relative_patch_size", C.c_float)]


class RegulariserC(C.Structure):
    _fields_ = [("type", C.c_int32), ("param", C.c_float), ("regularise_last_row", C.c_int32)]


class NormalisationC(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n_right", C.c_int32), ("n_left", C.c_int32),
                ("right_idx", C.c_int32 * 4), ("left_idx", C.c_int32 * 4)]


class ImageBatchC(C.Structure):
    _fields_ = [("d_data", C.c_void_p), ("width", C.c_int32), ("height", C.c_int32), ("row_stride", C.c_int32),
                ("image_stride", C.c_int64), ("count", C.c_int32), ("d_roi", C.c_void_p), ("d_roi_miss", C.c_void_p),
                ("d_frames", C.c_void_p)]


class FrameC(C.Structure):
    """sd_frame: one frame of a batch with differently sized frames."""
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("row_stride", C.c_int32), ("reserved", C.c_int32), ("offset", C.c_int64)]


class HostFrameC(C.Structure):
    """sd_host_frame: one frame in host memory for sd_detect_faces_host / sd_detect_faces_host_init; channels 0 or 1 = 8UC1,
    3 = 8UC3 B,G,R."""
    _fields_ = [("h_data", C.c_void_p), ("width", C.c_int32), ("height", C.c_int32), ("row_stride", C.c_int32), ("channels", C.c_int32)]


# every symbol declared in include/sd_b200.h (tests/test_abi.py checks the list against the header)
EXPORTS = [
    "sd_ctx_create", "sd_ctx_destroy", "sd_last_error", "sd_sync", "sd_version", "sd_launch_count", "sd_roi_fallback_count",
    "sd_malloc", "sd_free", "sd_host_alloc", "sd_host_free", "sd_memcpy_h2d", "sd_memcpy_d2h", "sd_memset",
    "sd_memcpy2d_h2d", "sd_memcpy2d_d2h", "sd_memcpy2d_d2d",
    "sd_hog_feature_length", "sd_hog_batch", "sd_hog_debug", "sd_bgr2gray",
    "sd_learn", "sd_centre_features", "sd_learn_centred", "sd_learn_rank_revealing", "sd_gram", "sd_solve_gram", "sd_predict", "sd_test_residual", "sd_solver_timings", "sd_set_gram_mode", "sd_set_solver", "sd_solver_iterations",
    "sd_comm_get_unique_id", "sd_comm_create", "sd_comm_adopt", "sd_comm_destroy", "sd_comm_rank", "sd_comm_size",
    "sd_comm_sum_int64", "sd_comm_allgather", "sd_allreduce_gram", "sd_reduce_scatter_gram", "sd_solve_gram_dist", "sd_learn_dist",
    "sd_cascade_targets", "sd_cascade_update", "sd_subtract_templates",
    "sd_model_load", "sd_model_save", "sd_model_create", "sd_model_destroy", "sd_model_num_levels",
    "sd_model_num_landmarks", "sd_model_hog_param", "sd_model_regulariser", "sd_model_normalisation",
    "sd_model_get_mean", "sd_model_get_weights", "sd_model_landmark_id", "sd_align_mean",
    "sd_perturb_box", "sd_normalised_landmark_errors",
    "sd_detect_batch_device", "sd_detect_batch_host",
    "sd_model_align_boxes", "sd_detect_faces_device", "sd_detect_faces_host", "sd_detect_faces_host_init",
]

_lib = None


def lib():
    """Loads libsd_b200.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SdError(2, f"{LIB_PATH} is missing: run `python -m superviseddescent_b200.build` "
                             f"(the CUDA extension is mandatory, there is no CPU path)")
        l = C.CDLL(LIB_PATH)
        l.sd_last_error.restype = C.c_char_p
        l.sd_version.restype = C.c_char_p
        l.sd_launch_count.restype = C.c_int64
        l.sd_roi_fallback_count.restype = C.c_int64
        l.sd_roi_fallback_count.argtypes = [C.c_void_p]
        l.sd_model_landmark_id.restype = C.c_char_p
        l.sd_last_error.argtypes = [C.c_void_p]
        l.sd_launch_count.argtypes = [C.c_void_p]
        l.sd_ctx_destroy.argtypes = [C.c_void_p]
        l.sd_model_destroy.argtypes = [C.c_void_p]
        l.sd_model_landmark_id.argtypes = [C.c_void_p, C.c_int]
        l.sd_comm_destroy.argtypes = [C.c_void_p]
        l.sd_solver_iterations.argtypes = [C.c_void_p]
        l.sd_comm_rank.argtypes = [C.c_void_p]
        l.sd_comm_size.argtypes = [C.c_void_p]
        _lib = l
    return _lib


def ptr(t) -> C.c_void_p:
    """Device pointer of a torch tensor (or None / int passthrough)."""
    if t is None:
        return C.c_void_p(0)
    if isinstance(t, int):
        return C.c_void_p(t)
    return C.c_void_p(t.data_ptr())
