"""ctypes binding of libswm_orb.so (the C ABI declared in include/swm_orb.h).

There is deliberately no fallback: if the shared library is missing, or no sm_100 device is
present, the calls raise.  Nothing in this package imports the CPU oracle.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# SWM_LIB_PATH: developer switch for A/B runs of kernel variants built under build/variants/ (tools/ab_variants.sh)
LIB_PATH = os.environ.get("SWM_LIB_PATH") or os.path.join(HERE, "libswm_orb.so")

SWM_OK = 0
ERRORS = {-1: "SWM_E_INVALID", -2: "SWM_E_CUDA", -3: "SWM_E_NODEVICE", -4: "SWM_E_CAPACITY", -5: "SWM_E_STATE"}

STAGE_PYRAMID, STAGE_NMS, STAGE_OCTREE, STAGE_DESCRIBE = 1, 2, 4, 8

KP_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"),
                     ("octave", "<i4"), ("class_id", "<i4")])
assert KP_DTYPE.itemsize == 28


class SwmError(RuntimeError):
    pass


class OrbCfg(C.Structure):
    _fields_ = [("nfeatures", C.c_int32), ("scale_factor", C.c_float), ("nlevels", C.c_int32),
                ("ini_th_fast", C.c_int32), ("min_th_fast", C.c_int32), ("max_batch", C.c_int32),
                ("max_fast_per_level", C.c_int32)]


class FrameView(C.Structure):
    _fields_ = [("n", C.c_int32), ("x", C.c_void_p), ("y", C.c_void_p), ("octave", C.c_void_p),
                ("angle", C.c_void_p), ("desc", C.c_void_p), ("min_x", C.c_float), ("min_y", C.c_float),
                ("max_x", C.c_float), ("max_y", C.c_float)]


class WindowQuery(C.Structure):
    _fields_ = [("m", C.c_int32), ("desc", C.c_void_p), ("u", C.c_void_p), ("v", C.c_void_p),
                ("radius", C.c_void_p), ("min_level", C.c_void_p), ("max_level", C.c_void_p),
                ("valid", C.c_void_p), ("angle", C.c_void_p), ("blocks", C.c_void_p)]


class Camera(C.Structure):
    _fields_ = [("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float),
                ("k1", C.c_float), ("k2", C.c_float), ("p1", C.c_float), ("p2", C.c_float), ("k3", C.c_float)]


class TriangulationQuery(C.Structure):
    _fields_ = [("F12", C.c_void_p), ("ex", C.c_float), ("ey", C.c_float), ("scale_factors2", C.c_void_p),
                ("level_sigma2", C.c_void_p), ("nlevels", C.c_int32)]


class BestQuery(C.Structure):
    _fields_ = [("m", C.c_int32), ("desc", C.c_void_p), ("u", C.c_void_p), ("v", C.c_void_p), ("radius", C.c_void_p),
                ("min_level", C.c_void_p), ("max_level", C.c_void_p), ("valid", C.c_void_p),
                ("inv_level_sigma2", C.c_void_p), ("nlevels", C.c_int32), ("chi2", C.c_float)]


class BowOut(C.Structure):
    _fields_ = [("word_ids", C.c_void_p), ("word_values", C.c_void_p), ("n_words", C.c_void_p),
                ("node_ids", C.c_void_p), ("node_offsets", C.c_void_p), ("feats", C.c_void_p), ("n_nodes", C.c_void_p)]


class FeatVec(C.Structure):
    _fields_ = [("n_nodes", C.c_int32), ("node_ids", C.c_void_p), ("offsets", C.c_void_p), ("feats", C.c_void_p)]


class WindowJob(C.Structure):
    _fields_ = [("tgt", C.c_void_p), ("tgt_resident", C.c_void_p), ("q", C.c_void_p), ("tgt_blocked", C.c_void_p),
                ("th_dist", C.c_int32), ("ratio_mode", C.c_int32), ("nnratio", C.c_float), ("check_ori", C.c_int32),
                ("assignment", C.c_void_p), ("nmatches", C.c_int32)]


class InitJob(C.Structure):
    _fields_ = [("f1", C.c_void_p), ("f2", C.c_void_p), ("r1", C.c_void_p), ("r2", C.c_void_p),
                ("prev_xy", C.c_void_p), ("matches12", C.c_void_p), ("window", C.c_int32), ("nnratio", C.c_float),
                ("check_ori", C.c_int32), ("nmatches", C.c_int32)]


class BowJob(C.Structure):
    _fields_ = [("f1", C.c_void_p), ("f2", C.c_void_p), ("r1", C.c_void_p), ("r2", C.c_void_p),
                ("fv1", C.c_void_p), ("fv2", C.c_void_p), ("valid1", C.c_void_p), ("valid2", C.c_void_p),
                ("mode", C.c_int32), ("nnratio", C.c_float), ("check_ori", C.c_int32), ("matches", C.c_void_p),
                ("nmatches", C.c_int32)]


# every symbol include/swm_orb.h declares: (name, restype, argtypes)
_vp, _i, _f, _sz, _i64 = C.c_void_p, C.c_int, C.c_float, C.c_size_t, C.c_int64
SYMBOLS = [
    ("swm_version", C.c_char_p, []),
    ("swm_orb_create", _i, [_vp, _i, _vp]),
    ("swm_orb_destroy", None, [_vp]),
    ("swm_last_error", C.c_char_p, [_vp]),
    ("swm_orb_extract", _i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i, _vp]),
    ("swm_orb_extract_batch", _i, [_vp, _vp, _i, _i, _i, _i, _sz, _vp, _vp, _i, _vp]),
    ("swm_orb_extract_batch_async", _i, [_vp, _vp, _i, _i, _i, _i, _sz, _vp, _vp, _i, _vp]),
    ("swm_orb_sync", _i, [_vp]),
    ("swm_orb_extract_batch_device", _i, [_vp, _vp, _i, _i, _i, _i, _sz, _vp, _vp, _i, _vp, _vp]),
    ("swm_orb_level_ptr", _i, [_vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    ("swm_orb_scale_tables", _i, [_vp, _vp, _vp, _vp, _vp]),
    ("swm_orb_level_quotas", _i, [_vp, _vp]),
    ("swm_orb_max_keypoints", _i, [_vp]),
    ("swm_orb_last_launches", _i, [_vp]),
    ("swm_orb_run_stage", _i, [_vp, _i, _i, _vp]),
    ("swm_orb_stereo_match", _i, [_vp, _vp, C.c_float, C.c_float, _vp, _vp, _i]),
    ("swm_orb_set_debug", _i, [_vp, _i]),
    ("swm_orb_debug_plane", _i, [_vp, _i, _i, _i, _vp, _i]),
    ("swm_orb_debug_points", _i, [_vp, _i, _i, _i, _vp, _i]),
    ("swm_hamming_matrix_device", _i, [_vp, _i, _vp, _i, _vp, _vp]),
    ("swm_hamming_matrix", _i, [_vp, _i, _vp, _i, _vp, _i]),
    ("swm_hamming_pairs", _i, [_vp, _vp, _i, _vp, _i]),
    ("swm_distinctive_descriptors", _i, [_vp, _vp, _i, _vp, _vp, _i]),
    ("swm_matcher_create", _i, [_i, _vp]),
    ("swm_matcher_destroy", None, [_vp]),
    ("swm_matcher_last_error", C.c_char_p, [_vp]),
    ("swm_grid_build", _i, [_vp, _vp, _vp, _vp]),
    ("swm_match_init", _i, [_vp, _vp, _vp, _vp, _vp, _i, _f, _i, _vp]),
    ("swm_match_window", _i, [_vp, _vp, _vp, _vp, _i, _i, _f, _i, _vp, _vp]),
    ("swm_match_bow", _i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _f, _i, _vp, _vp]),
    ("swm_window_best", _i, [_vp, _vp, _vp, _vp, _vp]),
    ("swm_window_best_resident", _i, [_vp, _vp, _vp, _vp, _vp]),
    ("swm_match_triangulation", _i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp]),
    ("swm_match_triangulation_resident", _i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp]),
    ("swm_camera_bounds", _i, [_i, _vp, _i, _i, _vp]),
    ("swm_frame_create", _i, [_i, _vp]),
    ("swm_frame_destroy", None, [_vp]),
    ("swm_frame_last_error", C.c_char_p, [_vp]),
    ("swm_frame_size", C.c_int32, [_vp]),
    ("swm_frame_from_extractor", _i, [_vp, _vp, _i, _vp, _vp]),
    ("swm_frame_upload", _i, [_vp, _vp]),
    ("swm_frame_download", _i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    ("swm_frame_slab_bytes", _sz, [C.c_int32]),
    ("swm_frame_export", _i, [_vp, _vp, _sz, _vp]),
    ("swm_frame_import", _i, [_vp, _vp, _sz]),
    ("swm_match_init_resident", _i, [_vp, _vp, _vp, _vp, _vp, _i, _f, _i, _vp]),
    ("swm_match_window_resident", _i, [_vp, _vp, _vp, _vp, _i, _i, _f, _i, _vp, _vp]),
    ("swm_match_bow_resident", _i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _f, _i, _vp, _vp]),
    ("swm_match_window_batch", _i, [_vp, _vp, _i]),
    ("swm_match_init_batch", _i, [_vp, _vp, _i]),
    ("swm_match_bow_batch", _i, [_vp, _vp, _i]),
    ("swm_frames_from_extractor", _i, [_vp, _i, _vp, _vp, _vp, _vp]),
    ("swm_matcher_last_device_ms", C.c_float, [_vp]),
    ("swm_vocab_create", _i, [_i, _vp, _sz, _vp]),
    ("swm_vocab_destroy", None, [_vp]),
    ("swm_vocab_last_error", C.c_char_p, [_vp]),
    ("swm_vocab_info", _i, [_vp, _vp, _vp, _vp, _vp]),
    ("swm_bow_transform", _i, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    ("swm_bow_transform_frame", _i, [_vp, _vp, _i, _vp]),
    ("swm_bow_score", _i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    ("swm_kfdb_create", _i, [_vp, _vp]),
    ("swm_kfdb_destroy", None, [_vp]),
    ("swm_kfdb_last_error", C.c_char_p, [_vp]),
    ("swm_kfdb_size", _i64, [_vp]),
    ("swm_kfdb_add", _i, [_vp, _i, _vp, _vp, _vp, _vp]),
    ("swm_kfdb_erase", _i, [_vp, _i, _vp]),
    ("swm_kfdb_clear", _i, [_vp]),
    ("swm_kfdb_query", _i, [_vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int32]),
    ("swm_kfdb_finish", _i, [_vp, _vp, _vp, _vp, _vp, C.c_int32]),
    ("swm_kfdb_last_device_ms", C.c_float, [_vp]),
    ("swm_db_create", _i, [_i, _vp, _i64, C.c_int32, _i64, _vp]),
    ("swm_db_create_device", _i, [_i, _vp, _i64, C.c_int32, _i64, _vp]),
    ("swm_db_destroy", None, [_vp]),
    ("swm_db_query_device", _i, [_vp, _vp, _i, _i, _vp, _vp, _i, _vp]),
    ("swm_db_merge_gathered", _i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i, _vp]),
    ("swm_db_query_sharded", _i, [_vp, _vp, _i, _vp, _i, _i, _vp, _vp, _i, _vp]),
    ("swm_db_peer_window", _i, [_vp, _i, _i, _vp, _vp]),
    ("swm_db_peer_open", _i, [_vp, _i, _vp, _vp]),
    ("swm_db_query_peers", _i, [_vp, _vp, _i, _i, _vp, _vp, _i, _vp]),
    ("swm_db_size", _i64, [_vp]),
    ("swm_i8_peak", _i, [_i, _i, _i, _vp]),
]

_lib = None


def load():
    """Loads libswm_orb.so; raises if it has not been built (no fallback of any kind)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SwmError(f"{LIB_PATH} is missing: build it with `python -m swarmmap_b200.build` "
                           "(there is no CPU or PyTorch fallback for the ORB front-end)")
        lib = C.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(lib, name)  # AttributeError if the ABI is incomplete
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def check(rc, handle=None, what=""):
    if rc != SWM_OK:
        lib = load()
        msg = lib.swm_last_error(handle)
        raise SwmError(f"{what}: {ERRORS.get(rc, rc)}: {msg.decode() if msg else ''}")
