"""ctypes binding of lib/libplmatch.so (the C ABI of include/plmatch.h).

There is no fallback: if the CUDA library has not been built, importing the symbols raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libplmatch.so")

PLM_OK = 0
PLM_E_INVALID, PLM_E_SIZE, PLM_E_TRAIN, PLM_E_GRID = -1, -2, -3, -4
PLM_E_RATIO, PLM_E_CUDA, PLM_E_NOMEM, PLM_E_UNSUPPORTED = -5, -6, -7, -8
KEY_ABSENT = np.uint64(0xFFFFFFFFFFFFFFFF)

u8p = C.POINTER(C.c_uint8)
i32p = C.POINTER(C.c_int32)
u64p = C.POINTER(C.c_uint64)
f32p = C.POINTER(C.c_float)
f64p = C.POINTER(C.c_double)
intp = C.POINTER(C.c_int)
vp = C.c_void_p


class PairJob(C.Structure):
    _fields_ = [("off1", C.c_int64), ("off2", C.c_int64), ("off_m", C.c_int64), ("n1", C.c_int32), ("n2", C.c_int32)]


class GridJob(C.Structure):
    _fields_ = [("off_coords", C.c_int64), ("off1", C.c_int64), ("off2", C.c_int64), ("off_cell_start", C.c_int64),
                ("off_cell_items", C.c_int64), ("off_dirs2", C.c_int64), ("off_m", C.c_int64), ("n1", C.c_int32),
                ("n2", C.c_int32), ("is_lines", C.c_int32), ("pad_", C.c_int32), ("win", C.c_int32 * 4)]


class DevGridArgs(C.Structure):
    _fields_ = [("coords", vp), ("d1", vp), ("cell_start", vp), ("cell_items", vp), ("d2", vp), ("dirs2", vp),
                ("m12_inout", vp), ("count", vp), ("i1_base", C.c_int64), ("ratio", C.c_double),
                ("line_sim_th", C.c_double), ("n1", C.c_int32), ("n2", C.c_int32), ("grid_rows", C.c_int32),
                ("grid_cols", C.c_int32), ("is_lines", C.c_int32), ("best_lr", C.c_int32), ("win", C.c_int32 * 4)]


class MapView(C.Structure):
    _fields_ = [("T", C.c_double * 12), ("fx", C.c_double), ("fy", C.c_double), ("cx", C.c_double), ("cy", C.c_double),
                ("inv_width", C.c_double), ("inv_height", C.c_double), ("width", C.c_int32), ("height", C.c_int32)]


class PeerGroup(C.Structure):
    _fields_ = [("xchg", C.POINTER(vp)), ("gather", C.POINTER(vp)), ("rank", C.c_int32), ("world", C.c_int32),
                ("q_cap", C.c_int32), ("pad_", C.c_int32), ("n_rows_cap", C.c_int64), ("xchg_epoch", C.c_uint32),
                ("gather_epoch", C.c_uint32)]


class FrameRec(C.Structure):
    _fields_ = [("desc_pl", C.c_int64), ("desc_pr", C.c_int64), ("desc_ll", C.c_int64), ("desc_lr", C.c_int64),
                ("kp_l", C.c_int64), ("kp_r", C.c_int64), ("ln_l", C.c_int64), ("ln_r", C.c_int64),
                ("n_pl", C.c_int32), ("n_pr", C.c_int32), ("n_ll", C.c_int32), ("n_lr", C.c_int32)]


class FrameConfig(C.Structure):
    _fields_ = [("inv_width", C.c_double), ("inv_height", C.c_double), ("grid_rows", C.c_int32),
                ("grid_cols", C.c_int32), ("matching_s_ws", C.c_int32), ("best_lr", C.c_int32),
                ("min_ratio_12p", C.c_double), ("min_ratio_12l", C.c_double), ("line_sim_th", C.c_double),
                ("max_dist_epip", C.c_double), ("min_disp", C.c_double), ("line_horiz_th", C.c_double),
                ("stereo_overlap_th", C.c_double), ("ls_min_disp_ratio", C.c_double), ("cam_b", C.c_double),
                ("cam_fx", C.c_double), ("cam_cx", C.c_double), ("cam_cy", C.c_double)]


class FramesOut(C.Structure):
    _fields_ = [(n, vp) for n in ("stereo_m12_p", "stereo_m12_l", "kept_p", "kept_l", "pt_disp", "pt_P", "ls_disp",
                                  "ls_sP", "ls_eP", "ls_le", "f2f_m12_p", "f2f_m12_l", "counts")]


FRAME_REC_DTYPE = np.dtype([("desc_pl", "<i8"), ("desc_pr", "<i8"), ("desc_ll", "<i8"), ("desc_lr", "<i8"),
                            ("kp_l", "<i8"), ("kp_r", "<i8"), ("ln_l", "<i8"), ("ln_r", "<i8"), ("n_pl", "<i4"),
                            ("n_pr", "<i4"), ("n_ll", "<i4"), ("n_lr", "<i4")])
assert FRAME_REC_DTYPE.itemsize == C.sizeof(FrameRec)

PAIR_JOB_DTYPE = np.dtype([("off1", "<i8"), ("off2", "<i8"), ("off_m", "<i8"), ("n1", "<i4"), ("n2", "<i4")])
GRID_JOB_DTYPE = np.dtype([("off_coords", "<i8"), ("off1", "<i8"), ("off2", "<i8"), ("off_cell_start", "<i8"),
                           ("off_cell_items", "<i8"), ("off_dirs2", "<i8"), ("off_m", "<i8"), ("n1", "<i4"),
                           ("n2", "<i4"), ("is_lines", "<i4"), ("pad_", "<i4"), ("win", "<i4", (4,))])
assert PAIR_JOB_DTYPE.itemsize == C.sizeof(PairJob) and GRID_JOB_DTYPE.itemsize == C.sizeof(GridJob)

_DESC = [u8p, C.c_int, C.c_size_t]

# name -> (restype, argtypes); every symbol include/plmatch.h declares
SIGNATURES = {
    "plm_version": (C.c_int, []),
    "plm_status_string": (C.c_char_p, [C.c_int]),
    "plm_last_error": (C.c_char_p, []),
    "plm_device_count": (C.c_int, [intp]),
    "plm_ctx_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
    "plm_ctx_destroy": (C.c_int, [vp]),
    "plm_ctx_stream": (vp, [vp]),
    "plm_ctx_set_stream": (C.c_int, [vp, vp, C.c_int]),
    "plm_ctx_synchronize": (C.c_int, [vp]),
    "plm_ctx_set_profiling": (C.c_int, [vp, C.c_int]),
    "plm_ctx_read_profile": (C.c_int, [vp, f64p, intp]),
    "plm_ctx_launch_count": (C.c_uint64, [vp]),
    "plm_hamming256": (C.c_int, [vp, u8p, C.c_size_t, u8p, C.c_size_t, C.c_int, i32p]),
    "plm_knn2": (C.c_int, [vp] + _DESC + _DESC + [C.c_uint64, u64p]),
    "plm_match_nnr": (C.c_int, [vp] + _DESC + _DESC + [C.c_float, i32p, intp]),
    "plm_match": (C.c_int, [vp] + _DESC + _DESC + [C.c_float, C.c_int, i32p, intp]),
    "plm_frame_begin": (C.c_int, [vp]),
    "plm_frame_active": (C.c_int, [vp]),
    "plm_frame_end": (C.c_int, [vp]),
    "plm_match_grid_points": (C.c_int, [vp, i32p] + _DESC + [i32p, i32p, C.c_int, C.c_int] + _DESC +
                              [i32p, C.c_double, C.c_int, i32p, intp]),
    "plm_match_grid_lines": (C.c_int, [vp, i32p] + _DESC + [i32p, i32p, C.c_int, C.c_int] + _DESC +
                             [f64p, C.c_double, i32p, C.c_double, C.c_int, i32p, intp]),
    "plm_stereo_filter_points": (C.c_int, [vp, f32p, C.c_int, f32p, C.c_int, i32p, C.c_double, C.c_double, u8p, f64p,
                                           intp]),
    "plm_stereo_filter_lines": (C.c_int, [vp, f32p, C.c_int, f32p, C.c_int, i32p, C.c_double, C.c_double, C.c_double,
                                          C.c_double, u8p, f64p, intp]),
    "plm_line_pair_filter": (C.c_int, [vp, f32p, C.c_int, f32p, C.c_int, i32p, C.c_double, C.c_double, u8p, f64p, f64p, intp]),
    "plm_batch_create": (C.c_int, [vp, C.POINTER(vp)]),
    "plm_batch_destroy": (C.c_int, [vp]),
    "plm_batch_set_match": (C.c_int, [vp, vp, C.c_int64, vp, C.c_int, C.c_float, C.c_int, vp, C.c_int64]),
    "plm_batch_set_match_dev": (C.c_int, [vp, vp, C.c_int64, vp, C.c_int, C.c_float, C.c_int, vp, C.c_int64]),
    "plm_batch_set_match_grid": (C.c_int, [vp, vp, C.c_int64, vp, C.c_int64, vp, C.c_int64, vp, C.c_int64, vp,
                                           C.c_int64, C.c_int, C.c_int, vp, C.c_int, C.c_double, C.c_double, C.c_int,
                                           vp, C.c_int64]),
    "plm_batch_run": (C.c_int, [vp]),
    "plm_batch_fetch": (C.c_int, [vp, vp, vp]),
    "plm_batch_h2d_bytes": (C.c_int64, [vp]),
    "plm_batch_d2h_bytes": (C.c_int64, [vp]),
    "plm_frames_create": (C.c_int, [vp, C.POINTER(vp)]),
    "plm_frames_destroy": (C.c_int, [vp]),
    "plm_frames_upload": (C.c_int, [vp, vp, C.c_int64, vp, C.c_int64, vp, C.c_int64, vp, C.c_int,
                                    C.POINTER(FrameConfig)]),
    "plm_frames_process": (C.c_int, [vp, vp, C.c_int64, vp, C.c_int64, vp, C.c_int64, vp, C.c_int,
                                     C.POINTER(FrameConfig), C.POINTER(FramesOut), C.c_int]),
    "plm_frames_run": (C.c_int, [vp]),
    "plm_frames_fetch": (C.c_int, [vp, C.POINTER(FramesOut)]),
    "plm_frames_h2d_bytes": (C.c_int64, [vp]),
    "plm_frames_d2h_bytes": (C.c_int64, [vp]),
    "plm_dev_knn2": (C.c_int, [vp, vp, C.c_int, vp, C.c_int64, C.c_uint64, vp]),
    "plm_dev_top2_merge": (C.c_int, [vp, vp, C.c_int, C.c_int, vp]),
    "plm_dev_nnr_accept": (C.c_int, [vp, vp, C.c_int, C.c_float, vp, vp]),
    "plm_dev_cross_check": (C.c_int, [vp, vp, C.c_int, C.c_int64, vp, C.c_int64, vp]),
    "plm_dev_grid_colmin": (C.c_int, [vp, C.POINTER(DevGridArgs), vp]),
    "plm_dev_grid_match": (C.c_int, [vp, C.POINTER(DevGridArgs), vp, vp]),
    "plm_dev_m21_from_keys": (C.c_int, [vp, vp, C.c_int, vp]),
    "plm_dev_match_grid": (C.c_int, [vp, C.POINTER(DevGridArgs), C.c_int]),
    "plm_peer_buffer_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "plm_peer_alloc": (C.c_int, [vp, C.c_int, C.c_int, C.POINTER(vp), u8p]),
    "plm_peer_open": (C.c_int, [vp, u8p, C.POINTER(vp)]),
    "plm_peer_close": (C.c_int, [vp, vp]),
    "plm_peer_free": (C.c_int, [vp, vp]),
    "plm_dev_top2_exchange": (C.c_int, [vp, C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_uint32, vp, C.c_int, vp,
                                        C.c_float, vp, vp, vp]),
    "plm_peer_emulate_begin": (C.c_int, [C.c_int]),
    "plm_peer_emulate_run": (C.c_int, [vp]),
    "plm_peer_gather_bytes": (C.c_size_t, [C.c_int, C.c_int64]),
    "plm_peer_alloc_bytes": (C.c_int, [vp, C.c_size_t, C.POINTER(vp), u8p]),
    "plm_dev_peer_allgather_i32": (C.c_int, [vp, C.POINTER(vp), C.c_int, C.c_int, C.c_int64, C.c_uint32, vp, C.c_int64,
                                             C.c_int64, C.c_int64, vp, vp, vp, vp]),
    "plm_dev_sharded_match_grid": (C.c_int, [vp, C.POINTER(DevGridArgs), C.POINTER(PeerGroup), C.c_int64, vp, vp, vp]),
    "plm_dev_sharded_match": (C.c_int, [vp, vp, C.c_int, C.c_int64, vp, C.c_int, C.c_float, C.c_int, vp, C.POINTER(PeerGroup),
                                        C.c_int64, vp, vp, vp]),
    "plm_dev_peer_reduce": (C.c_int, [vp, C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_int, vp, C.c_int, vp, vp]),
    "plm_map_select": (C.c_int, [vp, C.c_int, f64p, u8p, C.c_int, C.POINTER(MapView), i32p, i32p, f64p, intp]),
    "plm_map_gate": (C.c_int, [vp, C.c_int, f64p, i32p, C.c_int, f64p, C.c_int, C.c_double, u8p, intp]),
    "plm_dev_map_select": (C.c_int, [vp, C.c_int, vp, vp, C.c_int, C.POINTER(MapView), vp, vp, vp, vp]),
    "plm_dev_gather_rows": (C.c_int, [vp, vp, vp, vp, C.c_int, vp]),
    "plm_dev_map_gate": (C.c_int, [vp, C.c_int, vp, vp, vp, C.c_int, vp, C.c_int, C.c_double, vp, vp]),
    "plm_shard_create": (C.c_int, [intp, C.c_int, C.c_int, C.c_int64, C.POINTER(vp)]),
    "plm_shard_destroy": (C.c_int, [vp]),
    "plm_shard_n_devices": (C.c_int, [vp]),
    "plm_shard_n_rows": (C.c_int64, [vp]),
    "plm_shard_range": (C.c_int, [vp, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "plm_shard_launch_count": (C.c_uint64, [vp]),
    "plm_shard_synchronize": (C.c_int, [vp]),
    "plm_shard_upload": (C.c_int, [vp, u8p, C.c_int64, C.c_size_t, i32p, C.c_int]),
    "plm_shard_match_nnr": (C.c_int, [vp, u8p, C.c_int, C.c_size_t, C.c_float, u64p, i32p, intp]),
    "plm_shard_match_grid": (C.c_int, [vp, i32p, i32p, C.c_int, C.c_int] + _DESC + [f64p, C.c_double, i32p, C.c_double, C.c_int,
                                       i32p, intp]),
    "plm_shard_match": (C.c_int, [vp] + _DESC + [C.c_float, C.c_int, i32p, intp]),
    "plm_db_create": (C.c_int, [vp, C.c_int64, C.POINTER(vp)]),
    "plm_db_destroy": (C.c_int, [vp]),
    "plm_db_upload": (C.c_int, [vp, vp, C.c_int64, C.c_size_t, C.c_int64]),
    "plm_db_size": (C.c_int64, [vp]),
    "plm_db_device_ptr": (vp, [vp]),
    "plm_db_knn2": (C.c_int, [vp, u8p, C.c_int, C.c_size_t, C.c_uint64, u64p]),
    "plm_voc_create": (C.c_int, [vp, C.c_int, i32p, i32p, u8p, f64p, i32p, C.c_int, C.c_int, C.POINTER(vp)]),
    "plm_voc_destroy": (C.c_int, [vp]),
    "plm_voc_words": (C.c_int, [vp]),
    "plm_bow_transform": (C.c_int, [vp, u8p, C.c_int64, C.c_size_t, i32p, C.c_int, vp, f64p, i32p]),
    "plm_dev_bow_transform": (C.c_int, [vp, vp, C.c_int64, vp, C.c_int, C.c_int, vp, vp, vp]),
    "plm_bow_score": (C.c_int, [vp, vp, f64p, vp, i32p, C.c_int, vp, f64p, vp, i32p, C.c_int, f64p]),
    "plm_dev_bow_score": (C.c_int, [vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int64, vp, vp, vp, vp, C.c_int, vp]),
    "plm_loopdb_create": (C.c_int, [vp, vp, C.c_int, C.c_int, C.POINTER(vp)]),
    "plm_loopdb_destroy": (C.c_int, [vp]),
    "plm_loopdb_insert": (C.c_int, [vp, C.c_int] + _DESC + _DESC + [f64p, f64p]),
    "plm_loopdb_cull": (C.c_int, [vp, C.c_int]),
    "plm_loopdb_bow": (C.c_int, [vp, C.c_int, C.c_int, vp, f64p, i32p]),
    "plm_loopdb_match": (C.c_int, [vp, C.c_int, i32p, C.c_int, C.c_float, C.c_float, C.c_int, i32p, i32p, i32p, i32p]),
    "plm_loopdb_size": (C.c_int64, [vp]),
    "plm_loopdb_h2d_bytes": (C.c_int64, [vp]),
    "plm_loopdb_d2h_bytes": (C.c_int64, [vp]),
    "plm_med_desc": (C.c_int, [vp, u8p, C.c_int64, C.c_size_t, f64p, i32p, C.c_int, i32p, u8p, f64p]),
    "plm_dev_med_desc": (C.c_int, [vp, vp, C.c_int64, vp, vp, C.c_int, vp, vp, vp, vp]),
    "plm_set_option": (C.c_int, [C.c_char_p, C.c_int]),
    "plm_measure_int_peaks": (C.c_int, [vp, f64p, f64p]),
    "plm_measure_mma_i8_peak": (C.c_int, [vp, f64p]),
    "plm_measure_mma_i8_rate": (C.c_int, [vp, C.c_int, C.c_int, f64p]),
}

_lib = None


def load():
    """The loaded library; raises when lib/libplmatch.so is missing (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m pl_inertial_slam_b200.build` "
                "(nvcc, sm_100a).  There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


class PlmError(RuntimeError):
    def __init__(self, status: int, where: str):
        lib = load()
        detail = lib.plm_last_error().decode(errors="replace")
        super().__init__(f"{where}: {lib.plm_status_string(status).decode()} ({status}) {detail}")
        self.status = status


def check(status: int, where: str) -> None:
    if status != PLM_OK:
        raise PlmError(status, where)


def desc_args(a: np.ndarray):
    """(pointer, rows, step) of an n x 32 uint8 descriptor matrix (rows may be strided)."""
    if a.dtype != np.uint8 or a.ndim != 2 or a.shape[1] != 32:
        raise ValueError(f"descriptors must be n x 32 uint8, got {a.dtype} {a.shape}")
    if a.shape[0] and a.strides[1] != 1:
        a = np.ascontiguousarray(a)
    step = a.strides[0] if a.shape[0] > 1 else 32
    if a.shape[0] > 1 and step < 32:
        a = np.ascontiguousarray(a)
        step = 32
    return a, a.ctypes.data_as(u8p), int(a.shape[0]), C.c_size_t(step)
