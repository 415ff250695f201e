"""ctypes binding of libssdgeom.so (include/ssdgeom.h).  There is no fallback: if the library
is missing or CUDA is unavailable, calls raise."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SSDGEOM_LIB selects another build of the same library (A/B measurements of kernel variants); never a fallback
LIB_PATH = os.environ.get("SSDGEOM_LIB") or os.path.join(_HERE, "_lib", "libssdgeom.so")

OK = 0
ERR_ARG, ERR_TOO_MANY_GT, ERR_THRESH, ERR_SHAPE, ERR_NO_POSITIVE = -1, -2, -3, -4, -5
ERR_TOPK_RANGE, ERR_WORKSPACE, ERR_ALIGN, ERR_LIMIT, ERR_POS_NEG_OVERLAP = -6, -7, -8, -9, -10
ERR_NO_NCCL, ERR_LABEL_RANGE, ERR_STALE_INDEX = -11, -12, -13
ERR_NCCL_BASE = 10000
F32, F64, I32, I64 = 0, 1, 2, 3
COMM_ID_BYTES = 128
LOSS_RESULT_LEN = 16
# words of the loss result block (include/ssdgeom.h, out_result)
LOSS_TOTAL, LOSS_POS, LOSS_NEG, LOSS_LOC = 0, 1, 2, 3     # total, "cls loss pos", "cls loss neg", "loc loss"
LOSS_NUM_POS, LOSS_NUM_NEG, LOSS_KTH, LOSS_STATUS = 4, 5, 6, 7
LOSS_SUM_POS_CE, LOSS_SUM_NEG_CE, LOSS_SUM_L1 = 8, 9, 10
LOSS_OWN_POS, LOSS_ERRORS = 11, 12     # this shard's own positives; its data-dependent error count
LOSS_ADDITIVE = slice(LOSS_NUM_POS, LOSS_OWN_POS)   # [4, 11): summed over the shards with per-shard mining
PROF_MATCH, PROF_CE, PROF_FILTER, PROF_NMS = 0, 1, 2, 3
PROF_BUCKET, PROF_SEARCH, PROF_LOSS_TAIL, PROF_GRAD = 4, 5, 6, 7

_vp, _i32, _i64, _f32, _f64, _sz = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double, C.c_size_t
_pi32, _pf64 = C.POINTER(C.c_int32), C.POINTER(C.c_double)

# name -> (restype, argtypes); every symbol include/ssdgeom.h declares
PROTOTYPES = {
    "ssdg_status_string": (C.c_char_p, [C.c_int]),
    "ssdg_version": (C.c_int, []),
    "ssdg_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "ssdg_set_device": (C.c_int, [C.c_int]),
    "ssdg_get_device": (C.c_int, [C.POINTER(C.c_int)]),
    "ssdg_device_alloc": (C.c_int, [C.POINTER(_vp), _sz]),
    "ssdg_device_free": (C.c_int, [_vp]),
    "ssdg_host_alloc": (C.c_int, [C.POINTER(_vp), _sz]),
    "ssdg_host_free": (C.c_int, [_vp]),
    "ssdg_memcpy_h2d": (C.c_int, [_vp, _vp, _sz, _vp]),
    "ssdg_memcpy_d2h": (C.c_int, [_vp, _vp, _sz, _vp]),
    "ssdg_memset": (C.c_int, [_vp, C.c_int, _sz, _vp]),
    "ssdg_stream_create": (C.c_int, [C.POINTER(_vp)]),
    "ssdg_stream_create_priority": (C.c_int, [C.POINTER(_vp), C.c_int]),
    "ssdg_stream_destroy": (C.c_int, [_vp]),
    "ssdg_stream_sync": (C.c_int, [_vp]),
    "ssdg_event_create": (C.c_int, [C.POINTER(_vp)]),
    "ssdg_event_destroy": (C.c_int, [_vp]),
    "ssdg_event_record": (C.c_int, [_vp, _vp]),
    "ssdg_stream_wait_event": (C.c_int, [_vp, _vp]),
    "ssdg_event_elapsed_ms": (C.c_int, [_vp, _vp, C.POINTER(_f32)]),
    "ssdg_profile_enable": (C.c_int, [C.c_int]),
    "ssdg_profile_last_ms": (C.c_int, [C.c_int, C.POINTER(_f32)]),
    "ssdg_profile_span_ms": (C.c_int, [_i32, _vp, C.POINTER(_f32), C.POINTER(_f32)]),
    "ssdg_prior_count": (_i64, [_pi32, _pi32, _pi32, _i32]),
    "ssdg_prior_boxes": (C.c_int, [_pi32, _pi32, _pf64, _pi32, _pf64, _i32, _f64, _vp, _i64, _vp]),
    "ssdg_match_workspace_bytes": (_sz, [_i32, _i32, _i32]),
    "ssdg_prior_index_bytes": (_sz, [_i32]),
    "ssdg_prior_index_build": (C.c_int, [_vp, _i32, _i32, _vp, _sz, _vp]),
    "ssdg_prior_index_destroy": (C.c_int, [_vp]),
    "ssdg_match_encode": (C.c_int, [_vp, _i32, _vp, _vp, _vp, _i32, _vp, _i32, _i32, _i32, _f64,
                                    _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ssdg_match_status": (C.c_int, [_vp, _pi32, _vp]),
    "ssdg_encode": (C.c_int, [_vp, _i32, _vp, _i32, _i64, _i32, _vp, _i32, _vp]),
    "ssdg_decode": (C.c_int, [_vp, _vp, _i32, _i64, _i32, _f64, _vp, _vp]),
    "ssdg_iou_pairs": (C.c_int, [_vp, _i32, _vp, _i32, _i64, _i32, _vp, _vp]),
    "ssdg_loss_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "ssdg_multibox_loss": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp,
                                     _vp, _sz, _vp]),
    "ssdg_multibox_loss_stage": (C.c_int, [_i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp,
                                           _vp, _vp, _vp, _sz, _vp]),
    "ssdg_loss_exchange": (C.c_int, [_vp, _i32, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "ssdg_gt_prepare": (C.c_int, [_vp, _i32, _vp, _vp, _i64, _i64, _vp, _vp]),
    "ssdg_image_normalize": (C.c_int, [_vp, _vp, _i64, _vp]),
    "ssdg_priors_clip": (C.c_int, [_vp, _i32, _i64, _vp]),
    "ssdg_loc_scale": (C.c_int, [_vp, _vp, _i64, _f32, _f32, _vp]),
    "ssdg_detect_workspace_bytes": (_sz, [_i64, _i32, _i32, _i32]),
    "ssdg_detect": (C.c_int, [_vp, _vp, _vp, _i32, _i64, _i32, _i32, _f32, _i32, _f32, _vp, _vp, _vp, _vp, _vp,
                              _f32, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ssdg_detect_stage": (C.c_int, [_i32, _vp, _vp, _vp, _i32, _i64, _i32, _i32, _f32, _i32, _f32, _vp, _vp, _vp, _vp,
                                    _vp, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ssdg_multibox_loss_fused": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp,
                                           _vp, _vp, _vp, _sz, _vp]),
    "ssdg_nms": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _f32, _i32, _f32, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ssdg_detect_keep_top_k": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp,
                                         _vp]),
    "ssdg_eval_state_bytes": (_sz, [_i32, _i64, _i32, _i32]),
    "ssdg_eval_reset": (C.c_int, [_vp, _sz, _vp]),
    "ssdg_eval_accumulate": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _i32, _pf64, _i32,
                                       _i32, _i64, _i64, _vp, _sz, _vp]),
    "ssdg_eval_exchange": (C.c_int, [_vp, _i32, _i64, _i32, _i32, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "ssdg_eval_status": (C.c_int, [_vp, _pi32, _vp]),
    "ssdg_eval_finalize_workspace_bytes": (_sz, [_i32, _i64, _i32]),
    "ssdg_eval_finalize": (C.c_int, [_vp, _sz, _i32, _i64, _i32, _i32, _pf64, _i32, _vp, _vp, _vp, _vp, _vp, _sz,
                                     _vp]),
    "ssdg_comm_available": (C.c_int, [C.POINTER(C.c_int)]),
    "ssdg_comm_unique_id": (C.c_int, [_vp]),
    "ssdg_comm_init_rank": (C.c_int, [C.POINTER(_vp), _vp, _i32, _i32]),
    "ssdg_comm_world": (C.c_int, [_vp, _pi32, _pi32]),
    "ssdg_comm_allreduce_sum": (C.c_int, [_vp, _vp, _i64, _i32, _vp]),
    "ssdg_comm_allreduce_sum_multi": (C.c_int, [_vp, _i32, C.POINTER(_vp), C.POINTER(_i64), _pi32, _vp]),
    "ssdg_comm_destroy": (C.c_int, [_vp]),
}

_lib = None


class SsdgeomError(RuntimeError):
    pass


def lib():
    """Load (once) and return the library with prototypes attached."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise SsdgeomError(
                "libssdgeom.so is not built (%s). Run `python ssd-object-detection_b200/build_native.py` "
                "or __graft_entry__.build(); there is no CPU fallback." % LIB_PATH)
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def status_string(status: int) -> str:
    return lib().ssdg_status_string(int(status)).decode()


def check(status: int, what: str = ""):
    """Map a status code to the exception type the reference would raise: the reference's
    asserts (utils/bbox.py:50-51, models/ssd_model.py:347-351,375) are AssertionError;
    everything else is ValueError (argument) or SsdgeomError (CUDA)."""
    status = int(status)
    if status == OK:
        return
    msg = "%s%s" % (what + ": " if what else "", status_string(status))
    if status in (ERR_TOO_MANY_GT, ERR_THRESH, ERR_SHAPE, ERR_POS_NEG_OVERLAP):
        raise AssertionError(msg)
    if status == ERR_NO_NCCL:
        raise SsdgeomError(msg)
    if status < 0:
        raise ValueError(msg)
    if status >= ERR_NCCL_BASE:
        raise SsdgeomError("NCCL error %d: %s" % (status - ERR_NCCL_BASE, msg))
    raise SsdgeomError("CUDA error %d: %s" % (status, msg))


def device_count() -> int:
    n = C.c_int(0)
    lib().ssdg_device_count(C.byref(n))
    return n.value
