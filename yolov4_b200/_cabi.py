"""ctypes binding of libyolohead.so (include/yolo_head.h).  No torch types cross this boundary: tensors are
passed as data_ptr() integers, the stream as torch.cuda.current_stream().cuda_stream.

There is no CPU or PyTorch fallback: if the library is missing (and cannot be built) or a call fails, this raises.
"""
import ctypes
import os

from . import build as _build

_f = ctypes.c_float
_i = ctypes.c_int
_l = ctypes.c_long
_p = ctypes.c_void_p
_sz = ctypes.c_size_t

_lib = None


class YoloHeadError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("YL_LIB")                  # YL_LIB: load a tuning build instead of the default library
    if path is None:
        # (re)build from source when the library is missing or older than csrc/ / include/ and a toolchain is present (a
        # stale .so must never be loaded silently); without a toolchain an existing library is used, a missing one raises.
        # There is no fall back to eager PyTorch.
        path = _build.LIB
        if _build.is_stale():
            try:
                path = _build.build_lib()
            except Exception:
                if not os.path.exists(path):
                    raise
    L = ctypes.CDLL(path)
    L.yl_source_hash.restype = ctypes.c_char_p
    L.yl_source_hash.argtypes = []
    if "YL_LIB" not in os.environ and L.yl_source_hash().decode() != _build.source_hash():
        raise YoloHeadError("libyolohead.so was built from other sources than csrc/ and include/ hold now, and it could "
                            "not be rebuilt (no nvcc?)")
    L.yl_abi_version.restype = _i
    L.yl_abi_version.argtypes = []
    L.yl_error_string.restype = ctypes.c_char_p
    L.yl_error_string.argtypes = [_i]
    L.yl_selftest_rcp.restype = _i
    L.yl_selftest_rcp.argtypes = [_p, _p]
    L.yl_decode_dense.restype = _i
    L.yl_decode_dense.argtypes = [_p, _i, _i, _i, _p, _f, _p, _l, _l, _p]
    L.yl_decode_dense_ex.restype = _i
    L.yl_decode_dense_ex.argtypes = [_p, _i, _i, _i, _p, _f, _f, _p, _l, _l, _p]
    L.yl_decode_train.restype = _i
    L.yl_decode_train.argtypes = [_p, _i, _i, _i, _p, _p, _p, _p]
    L.yl_decode_train_backward.restype = _i
    L.yl_decode_train_backward.argtypes = [_p, _p, _i, _i, _i, _p, _p]
    L.yl_decode_train_backward_raw.restype = _i
    L.yl_decode_train_backward_raw.argtypes = [_p, _p, _i, _i, _i, _p, _p]
    L.yl_post_workspace_bytes.restype = _sz
    L.yl_post_workspace_bytes.argtypes = [_i, _l, _i, _i]
    L.yl_post_reset.restype = _i
    L.yl_post_reset.argtypes = [_p, _sz, _i, _l, _i, _i, _p]
    L.yl_filter_raw.restype = _i
    L.yl_filter_raw.argtypes = [_p, _p, _i, _i, _i, _p, _p, _f, _p, _sz, _l, _i, _i, _i, _p]
    L.yl_filter_raw_stage.restype = _i
    L.yl_filter_raw_stage.argtypes = [_p, _p, _i, _i, _i, _p, _p, _f, _p, _sz, _l, _i, _i, _i, _i, _p]
    L.yl_filter_raw_typed.restype = _i
    L.yl_filter_raw_typed.argtypes = [_p, _i, _p, _i, _i, _i, _p, _p, _f, _p, _sz, _l, _i, _i, _i, _i, _p]
    L.yl_filter_raw_ex.restype = _i
    L.yl_filter_raw_ex.argtypes = [_p, _i, _p, _i, _i, _i, _p, _p, _f, _p, _p, _sz, _l, _i, _i, _i, _i, _p]
    L.yl_filter_dense.restype = _i
    L.yl_filter_dense.argtypes = [_p, _i, _l, _i, _i, _f, _p, _sz, _i, _i, _i, _p]
    L.yl_nms.restype = _i
    L.yl_nms.argtypes = [_p, _sz, _i, _l, _i, _i, _f, _p, _l, _p, _i, _i, _p]
    L.yl_nms_topk.restype = _i
    L.yl_nms_topk.argtypes = [_p, _sz, _i, _l, _i, _i, _f, _i, _p, _l, _p, _p, _i, _i, _p]
    L.yl_nms_ex.restype = _i
    L.yl_nms_ex.argtypes = [_p, _sz, _i, _l, _i, _i, _f, _i, _i, _p, _l, _p, _p, _i, _i, _p]
    L.yl_nms_ex2.restype = _i
    L.yl_nms_ex2.argtypes = [_p, _sz, _i, _l, _i, _i, _f, _i, _i, _i, _p, _l, _p, _p, _i, _i, _p]
    L.yl_post_workspace_bytes_ex.restype = _sz
    L.yl_post_workspace_bytes_ex.argtypes = [_i, _l, _i, _i, _i]
    L.yl_build_target.restype = _i
    L.yl_build_target.argtypes = [_p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _f, _p, _p, _p, _p, _p, _p]
    L.yl_build_target3.restype = _i
    L.yl_build_target3.argtypes = [_p, _p, _p, _i, _p, _i, _i, _i, _p, _p, _p, _f, _p, _p, _p, _p, _p, _p]
    L.yl_coco_rows.restype = _i
    L.yl_coco_rows.argtypes = [_p, _p, _l, _p, _p, _p, _i, _i, _p, _p]
    L.yl_coco_rows_padded.restype = _i
    L.yl_coco_rows_padded.argtypes = [_p, _p, _i, _l, _p, _p, _p, _i, _i, _p, _p]
    L.yl_loss_forward.restype = _i
    L.yl_loss_forward.argtypes = [_p, _p, _i, _i, _i, _i, _i, _p, _p, _f, _p, _p, _p, _p, _p, _p, _p]
    L.yl_loss_forward_chained.restype = _i
    L.yl_loss_forward_chained.argtypes = L.yl_loss_forward.argtypes
    L.yl_loss_backward.restype = _i
    L.yl_loss_backward.argtypes = [_p, _p, _p, _p, _i, _i, _i, _i, _p, _p]
    L.yl_loss_forward_typed.restype = _i
    L.yl_loss_forward_typed.argtypes = [_p, _i, _p, _i, _i, _i, _i, _i, _p, _p, _f, _p, _p, _p, _p, _p, _p, _p]
    L.yl_loss_forward_chained_typed.restype = _i
    L.yl_loss_forward_chained_typed.argtypes = L.yl_loss_forward_typed.argtypes
    L.yl_loss_forward_ex.restype = _i
    L.yl_loss_forward_ex.argtypes = [_p, _i, _p, _i, _i, _i, _i, _i, _p, _p, _f, _i, _f, _i, _p, _p, _p, _p, _p, _p, _p]
    L.yl_loss_forward_ex2.restype = _i
    L.yl_loss_forward_ex2.argtypes = [_p, _i, _p, _i, _i, _i, _i, _i, _p, _p, _f, _i, _f, _f, _i, _p, _p, _p, _p, _p, _p, _p]
    L.yl_loss_backward_typed.restype = _i
    L.yl_loss_backward_typed.argtypes = [_p, _p, _p, _p, _i, _i, _i, _i, _p, _i, _p]
    L.yl_context_create.restype = _i
    L.yl_context_create.argtypes = [ctypes.POINTER(_p), _i, _i, _p, _i, _i, _p, _p, _i, _l]
    L.yl_context_create_typed.restype = _i
    L.yl_context_create_typed.argtypes = [ctypes.POINTER(_p), _i, _i, _p, _i, _i, _i, _p, _p, _i, _l]
    L.yl_context_destroy.restype = _i
    L.yl_context_destroy.argtypes = [_p]
    L.yl_detect_host.restype = _i
    L.yl_detect_host.argtypes = [_p, _p, _f, _f, _p, _p]
    L.yl_detect_host_topk.restype = _i
    L.yl_detect_host_topk.argtypes = [_p, _p, _f, _f, _i, _p, _p]
    L.yl_detect_host_ex.restype = _i
    L.yl_detect_host_ex.argtypes = [_p, _p, _f, _f, _i, _i, _p, _p]
    L.yl_detect_host_ex2.restype = _i
    L.yl_detect_host_ex2.argtypes = [_p, _p, _f, _f, _i, _i, _i, _p, _p]
    L.yl_detect_host_ex3.restype = _i
    L.yl_detect_host_ex3.argtypes = [_p, _p, _f, _f, _i, _i, _i, _p, _p, _p]
    L.yl_xchg_create.restype = _i
    L.yl_xchg_create.argtypes = [ctypes.POINTER(_p), _i, _i, _i, _i, _l, _i]
    L.yl_xchg_window_bytes.restype = _sz
    L.yl_xchg_window_bytes.argtypes = [_i, _i, _l, _i]
    L.yl_xchg_create_external.restype = _i
    L.yl_xchg_create_external.argtypes = [ctypes.POINTER(_p), _i, _i, _i, _i, _l, _i, _p, _p]
    L.yl_xchg_destroy.restype = _i
    L.yl_xchg_destroy.argtypes = [_p]
    L.yl_xchg_handle_bytes.restype = _sz
    L.yl_xchg_handle_bytes.argtypes = []
    L.yl_xchg_local_handle.restype = _i
    L.yl_xchg_local_handle.argtypes = [_p, _p]
    L.yl_xchg_connect.restype = _i
    L.yl_xchg_connect.argtypes = [_p, _p]
    L.yl_xchg_push.restype = _i
    L.yl_xchg_push.argtypes = [_p, _p, _p, _i, _p]
    L.yl_xchg_wait.restype = _i
    L.yl_xchg_wait.argtypes = [_p, _i, _p]
    L.yl_xchg_release.restype = _i
    L.yl_xchg_release.argtypes = [_p, _i, _p]
    for name in ("yl_xchg_rows", "yl_xchg_counts"):
        getattr(L, name).restype = _p
        getattr(L, name).argtypes = [_p, _i]
    L.yl_xchg_status.restype = _p
    L.yl_xchg_status.argtypes = [_p]
    if L.yl_abi_version() != 1:
        raise YoloHeadError("libyolohead.so ABI version mismatch")
    _lib = L
    return L


EXPORTS = [
    "yl_abi_version", "yl_source_hash", "yl_error_string", "yl_selftest_rcp", "yl_decode_dense", "yl_decode_dense_ex", "yl_decode_train", "yl_decode_train_backward", "yl_decode_train_backward_raw",
    "yl_post_workspace_bytes", "yl_post_reset", "yl_filter_raw", "yl_filter_raw_stage", "yl_filter_raw_typed", "yl_filter_raw_ex", "yl_filter_dense", "yl_nms", "yl_nms_topk", "yl_nms_ex", "yl_nms_ex2", "yl_post_workspace_bytes_ex", "yl_build_target", "yl_build_target3", "yl_coco_rows", "yl_coco_rows_padded",
    "yl_loss_forward", "yl_loss_forward_chained", "yl_loss_backward", "yl_loss_forward_typed", "yl_loss_forward_chained_typed", "yl_loss_backward_typed", "yl_loss_forward_ex", "yl_loss_forward_ex2",
    "yl_context_create", "yl_context_create_typed", "yl_context_destroy", "yl_detect_host", "yl_detect_host_topk", "yl_detect_host_ex", "yl_detect_host_ex2", "yl_detect_host_ex3",
    "yl_xchg_create", "yl_xchg_create_external", "yl_xchg_window_bytes", "yl_xchg_destroy", "yl_xchg_handle_bytes", "yl_xchg_local_handle", "yl_xchg_connect", "yl_xchg_push",
    "yl_xchg_wait", "yl_xchg_release", "yl_xchg_rows", "yl_xchg_counts", "yl_xchg_status",
]


def check(rc):
    if rc != 0:
        raise YoloHeadError("libyolohead: %s (code %d)" % (lib().yl_error_string(rc).decode(), rc))


def floats(vals):
    return (ctypes.c_float * len(vals))(*[float(v) for v in vals])


def ints(vals):
    return (ctypes.c_int * len(vals))(*[int(v) for v in vals])


def longs(vals):
    return (ctypes.c_long * len(vals))(*[int(v) for v in vals])


def ptrs(vals):
    return (ctypes.c_void_p * len(vals))(*[int(v) for v in vals])
