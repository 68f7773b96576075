"""ctypes binding of libekpose_b200.so (include/ekpose_b200.h).

The library is the product: there is no Python or CPU implementation behind it.  If the
shared object has not been built (``python -c 'import __graft_entry__ as g; g.build()'`` or
``make -C torch_ekpose_b200/csrc``) importing this module raises immediately.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# EKPOSE_B200_SO selects another build of the same library (kernel sweeps in tools/)
SO_PATH = os.environ.get("EKPOSE_B200_SO") or os.path.join(HERE, "libekpose_b200.so")

NUM_PART, NUM_LIMB, HEAT_CH, PAF_CH, UP, SUBSET_COLS = 18, 19, 19, 38, 8, 20
LAYOUT_NCHW, LAYOUT_NHWC = 0, 1
DTYPE_F32, DTYPE_BF16, DTYPE_F16 = 0, 1, 2
FRONTEND_DENSE, FRONTEND_REFERENCE, FRONTEND_REFERENCE_COARSE, FRONTEND_REFERENCE_GAUSS = 0, 1, 2, 3
OK, ERR_ARG, ERR_CUDA, ERR_CAPACITY, ERR_STATE = 0, -1, -2, -3, -4
OVF_PEAKS, OVF_PART, OVF_CANDIDATES, OVF_HUMANS, OVF_BADPEAK = 1, 2, 4, 8, 16
MAX_PART, MAX_CAND = 256, 2048                                              # EKP_MAX_PART / EKP_MAX_CAND (defaults)
LIMIT_PEAKS, LIMIT_HUMANS, LIMIT_PART, LIMIT_CAND = 16384, 1024, 1024, 8192  # EKP_LIMIT_*
DRAW_MAX_SIDE = 16384                                                       # EKP_DRAW_MAX_SIDE


class EkpError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libekpose_b200 error {code}: {message}")
        self.code = code


class EkpCapacityError(EkpError):
    pass


class Peak(C.Structure):  # ekp_peak
    _fields_ = [("x", C.c_int), ("y", C.c_int), ("score", C.c_float), ("id", C.c_int)]


class DeviceResults(C.Structure):  # ekp_device_results: device pointers, None = that table is not written
    _fields_ = [("num_humans", C.c_void_p), ("overflow", C.c_void_p), ("n_peaks", C.c_void_p), ("subset", C.c_void_p),
                ("parts", C.c_void_p), ("scores", C.c_void_p)]


# every symbol include/ekpose_b200.h declares: (restype, argtypes)
_vp, _i, _f = C.c_void_p, C.c_int, C.c_float
SIGNATURES = {
    "ekp_create": (_i, [C.POINTER(_vp), _i, _i, _i, _i, _i, _i]),
    "ekp_create_ex": (_i, [C.POINTER(_vp), _i, _i, _i, _i, _i, _i, _i, _i]),
    "ekp_destroy": (None, [_vp]),
    "ekp_last_error": (C.c_char_p, []),
    "ekp_version": (C.c_char_p, []),
    "ekp_postprocess": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _f, _i, _vp, _vp, _vp]),
    "ekp_postprocess_host": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _f, _i, _i, _vp]),
    "ekp_postprocess_typed": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _i, _vp, _vp, _vp]),
    "ekp_postprocess_host_typed": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _i, _i, _vp]),
    "ekp_process_paf_dev": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _i, _i, _i, _vp]),
    "ekp_results": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "ekp_results_humans": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "ekp_results_device": (_i, [_vp, _i, C.POINTER(DeviceResults), _vp]),
    "ekp_scipy_gauss3_weights": (_i, [_vp]),
    "ekp_debug_std_sort": (_i, [_vp, _vp, _vp, _i, _vp]),
    "ekp_results_parts": (_i, [_vp, _vp]),
    "ekp_dense_smooth_debug": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "ekp_preprocess_dims": (_i, [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "ekp_preprocess": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "ekp_set_timing": (_i, [_vp, _i]),
    "ekp_stage_times": (_i, [_vp, _vp, _vp]),
    "ekp_last_batch": (_i, [_vp]),
    "ekp_max_batch": (_i, [_vp]),
    "ekp_max_peaks": (_i, [_vp]),
    "ekp_max_humans": (_i, [_vp]),
    "ekp_max_part": (_i, [_vp]),
    "ekp_max_cand": (_i, [_vp]),
    "ekp_kernel_launches": (C.c_longlong, [_vp]),
    "ekp_graph_launches": (C.c_longlong, [_vp]),
    "ekp_host_alloc": (_i, [C.POINTER(_vp), C.c_size_t, _i]),
    "ekp_host_free": (_i, [_vp]),
    "ekp_draw_humans": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "ekp_debug_raster_host": (_i, [_i, _i, _i, _i, _i, _i, _i, _vp]),
    "ekp_debug_draw_host": (_i, [_vp, _vp, _i, _i, _i, _vp, _i, _i, _i]),
    # the reference operator surface, lib/pafprocess/pafprocess.h:53-59
    "process_paf": (_i, [_i, _i, _i, _vp, _i, _i, _i, _vp, _i, _i, _i, _vp]),
    "get_num_humans": (_i, []),
    "get_part_cid": (_i, [_i, _i]),
    "get_score": (_f, [_i]),
    "get_part_x": (_i, [_i]),
    "get_part_y": (_i, [_i]),
    "get_part_score": (_f, [_i]),
}


def load() -> C.CDLL:
    if not os.path.exists(SO_PATH):
        raise ImportError(
            f"{SO_PATH} is missing: build the CUDA library first (make -C torch_ekpose_b200/csrc, or "
            "__graft_entry__.build()).  torch_ekpose_b200 has no CPU fallback.")
    lib = C.CDLL(SO_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here == header and library disagree
        fn.restype = res
        fn.argtypes = args
    return lib


lib = load()


def last_error() -> str:
    return (lib.ekp_last_error() or b"").decode()


def check(rc: int) -> None:
    if rc == OK:
        return
    msg = last_error()
    if rc == ERR_CAPACITY:
        raise EkpCapacityError(rc, msg)
    raise EkpError(rc, msg)
