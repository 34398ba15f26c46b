"""ctypes binding of libdist_b200.so (include/dist_b200.h).

The product path has no fallback: if the shared library is missing or a symbol is absent this module raises at
import of the renderer, and every call that fails inside the library raises ``DistError`` with its message.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libdist_b200.so")

ABI_VERSION = 3
MAX_LAYERS = 16
MAX_WIDTH = 512
MAX_BUFFER = 8
ENGINE_SIMT, ENGINE_TC = 0, 1
MARCH_TRIVIAL, MARCH_RECURSIVE, MARCH_PYRAMID = 0, 1, 2

c_f32p = C.POINTER(C.c_float)


class DistError(RuntimeError):
    pass


class Net(C.Structure):
    _fields_ = [("n_layers", C.c_int32), ("latent_size", C.c_int32), ("latent_in", C.c_int32),
                ("use_tanh", C.c_int32), ("K", C.c_int32 * MAX_LAYERS), ("N", C.c_int32 * MAX_LAYERS),
                ("Wt", C.c_void_p * MAX_LAYERS), ("W", C.c_void_p * MAX_LAYERS), ("bias", C.c_void_p * MAX_LAYERS),
                ("Wz0", C.c_void_p), ("b0", C.c_void_p), ("Wzl", C.c_void_p), ("bl", C.c_void_p),
                ("tc_blob", C.c_void_p), ("tc_scale", C.c_void_p), ("tc_blob_bytes", C.c_int64),
                ("tc_bias", C.c_void_p * MAX_LAYERS), ("n_codes", C.c_int32), ("row_code", C.c_void_p)]


class Camera(C.Structure):
    _fields_ = [("Kinv", C.c_float * 9), ("M", C.c_float * 9), ("Mn", C.c_float * 9), ("R", C.c_void_p),
                ("cam_pos", C.c_void_p),
                ("width", C.c_int32), ("height", C.c_int32), ("row0", C.c_int32), ("row_step", C.c_int32),
                ("n_rows", C.c_int32), ("radius", C.c_float), ("n_views", C.c_int32), ("row_group", C.c_int32)]


class March(C.Structure):
    _fields_ = [("march_step", C.c_int32), ("buffer_size", C.c_int32), ("marching_type", C.c_int32),
                ("first_query_check", C.c_int32), ("ratio", C.c_float), ("threshold", C.c_float),
                ("clamp_dist", C.c_float), ("replay_grad_rounding", C.c_int32), ("coarse_steps", C.c_int32 * 2),
                ("screen", C.c_int32), ("screen_margin", C.c_float), ("screen_tpred", C.c_float),
                ("screen_ext_margin", C.c_float),
                ("cam_grad_levels", C.c_int32)]


WS_FIELDS = ["ray", "entry", "exit_", "dist", "z", "flags", "nreal", "top_sdf", "top_pt", "top_zafter", "top_zgen",
             "list_a", "list_b", "pts", "sdf", "counts", "sdf_origin", "entry0", "top_lvl", "pyr_f", "pyr_i", "pyr_b",
             "seg_approx", "sprev", "rq_idx", "rq_pts", "rq_sdf", "rq_cnt", "mask_buf", "mask_base", "top_slot", "bm_row", "bm_slot",
             "bm_sdf", "bm_coef", "bm_dpts", "bm_cnt", "tile_counters", "mask_cap", "view_stat"]


class Workspace(C.Structure):
    _fields_ = [(n, C.c_int64 if n == "mask_cap" else C.c_void_p) for n in WS_FIELDS]


# name -> (restype, argtypes); mirrors include/dist_b200.h one to one
PROTOTYPES = {
    "dist_abi_version": (C.c_int, []),
    "dist_last_error": (C.c_char_p, []),
    "dist_launch_count": (C.c_longlong, []),
    "dist_profile_begin": (C.c_int, []),
    "dist_profile_end": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_longlong)]),
    "dist_device_supports_tc": (C.c_int, [C.c_int]),
    "dist_fold_latent": (C.c_int, [C.POINTER(Net), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dist_decoder_forward": (C.c_int, [C.POINTER(Net), C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_float,
                                       C.c_void_p, C.c_void_p]),
    "dist_decoder_forward_tiers": (C.c_int, [C.POINTER(Net), C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_float,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dist_decoder_forward_masks": (C.c_int, [C.POINTER(Net), C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                             C.c_void_p]),
    "dist_decoder_backward_masked": (C.c_int, [C.POINTER(Net), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_float,
                                               C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dist_decoder_input_grad": (C.c_int, [C.POINTER(Net), C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_float,
                                          C.c_void_p, C.c_void_p, C.c_void_p]),
    "dist_decoder_backward": (C.c_int, [C.POINTER(Net), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                        C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dist_render_depth_fwd": (C.c_int, [C.POINTER(Net), C.c_int, C.POINTER(Camera), C.POINTER(March),
                                        C.POINTER(Workspace), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p]),
    "dist_render_normal_fwd": (C.c_int, [C.POINTER(Net), C.c_int, C.POINTER(Camera), C.c_void_p, C.c_void_p,
                                         C.c_float, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p]),
    "dist_render_depth_bwd": (C.c_int, [C.POINTER(Net), C.c_int, C.POINTER(Camera), C.POINTER(March),
                                        C.POINTER(Workspace)] + [C.c_void_p] * 15),
    "dist_warp_loss_fwd": (C.c_int, [C.POINTER(Camera), C.POINTER(C.c_float)] + [C.c_void_p] * 7 + [C.c_float] +
                           [C.c_void_p] * 6),
    "dist_warp_loss_bwd": (C.c_int, [C.POINTER(Camera), C.POINTER(C.c_float)] + [C.c_void_p] * 13),
    "dist_scan_scratch_elems": (C.c_int64, [C.c_int64]),
    "dist_mc_count": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float] + [C.c_void_p] * 5),
    "dist_mc_emit": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.POINTER(C.c_float), C.POINTER(C.c_float)] +
                     [C.c_void_p] * 5),
    "dist_tri_area_scan": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64] + [C.c_void_p] * 4),
    "dist_surface_sample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64] +
                            [C.c_void_p] * 3),
    "dist_nearest_sqdist": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64] + [C.c_void_p] * 4),
}

_lib = None


def lib():
    """Loads libdist_b200.so (once) and binds every prototype.  Raises if the library or a symbol is missing."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise DistError("libdist_b200.so not built: run `python __graft_entry__.py build` "
                            "(there is no CPU or PyTorch fallback for the rendering path)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)  # AttributeError if the symbol is missing
            fn.restype, fn.argtypes = res, args
        if L.dist_abi_version() != ABI_VERSION:
            raise DistError("libdist_b200.so ABI version mismatch")
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise DistError("libdist_b200: error %d: %s" % (rc, lib().dist_last_error().decode()))


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())
