"""ctypes binding of libyolo_b200.so (the C ABI declared in include/yolo_b200.h).

The shared library is built in-tree by ``__graft_entry__.build()`` /
``make -C tf2_yolo_b200/csrc``.  There is no fallback: if the library is
missing, importing this module raises, and every op raises on a non-zero status.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libyolo_b200.so")

YB_MAX_BOXES = 16
YB_MAX_SCALES = 4
YB_LOSS_TERMS = 8
YB_LOSS_METRICS = 10
YB_ENCODE_MAX_BOXES = 1024
YB_FUSED_MAX_ROWS = 2048
YB_KMEANS_HIST = 64
YB_MAX_PEERS = 16
YB_DIST_IOU, YB_DIST_EUCLID = 0, 1


class YoloB200Error(RuntimeError):
    pass


class LossParams(C.Structure):
    _fields_ = [
        ("version", C.c_int32),
        ("grid_h", C.c_int32), ("grid_w", C.c_int32),
        ("bbox_num", C.c_int32), ("class_num", C.c_int32),
        ("has_anchors", C.c_int32),
        ("anchors", C.c_float * (2 * YB_MAX_BOXES)),
        ("binary_weight", C.c_float),
        ("loss_weight", C.c_float * 4),
        ("wh_reg_weight", C.c_float),
        ("ignore_thresh", C.c_float),
        ("truth_thresh", C.c_float),
        ("label_smooth", C.c_float),
        ("focal_gamma", C.c_float),
        ("use_focal", C.c_int32),
        ("use_scale", C.c_int32),
        ("from_logits", C.c_int32),
        ("inv_batch", C.c_double),
    ]


class LossScale(C.Structure):
    _fields_ = [
        ("y_true", C.c_void_p),
        ("y_pred", C.c_void_p),
        ("dpred", C.c_void_p),
        ("n_cells", C.c_int64),
        ("p", LossParams),
    ]


class DecodeParams(C.Structure):
    _fields_ = [
        ("version", C.c_int32),
        ("class_num", C.c_int32),
        ("n_scales", C.c_int32),
        ("is_f64", C.c_int32),
        ("grid_h", C.c_int32 * YB_MAX_SCALES),
        ("grid_w", C.c_int32 * YB_MAX_SCALES),
        ("bbox_num", C.c_int32 * YB_MAX_SCALES),
        ("threshold", C.c_double),
    ]


_vp, _i64, _i32, _sz, _dbl = C.c_void_p, C.c_int64, C.c_int, C.c_size_t, C.c_double

# name -> (restype, argtypes); must list every symbol of include/yolo_b200.h
SIGNATURES = {
    "yb_abi_version": (C.c_int, []),
    "yb_status_string": (C.c_char_p, [C.c_int]),
    "yb_last_error_site": (C.c_char_p, []),
    "yb_mapped_host_pointer": (C.c_int, [_vp, C.POINTER(_vp)]),
    "yb_loss_workspace_bytes": (_sz, [_i32]),
    "yb_loss_fwd_bwd": (C.c_int, [C.POINTER(LossScale), _i32, _vp, _vp, _vp, _sz, _vp]),
    "yb_loss_fwd_bwd_metrics": (C.c_int, [C.POINTER(LossScale), _i32, _vp, _vp, _vp, _dbl, _vp, _sz, _vp]),
    "yb_loss_v1_fwd_bwd": (C.c_int, [_vp, _vp, _i64, _vp, _vp, C.POINTER(LossParams), _vp, _sz, _vp]),
    "yb_loss_v2_fwd_bwd": (C.c_int, [_vp, _vp, _i64, _vp, _vp, C.POINTER(LossParams), _vp, _sz, _vp]),
    "yb_loss_v3_fwd_bwd": (C.c_int, [_vp, _vp, _i64, _vp, _vp, C.POINTER(LossParams), _vp, _sz, _vp]),
    "yb_loss_v4_fwd_bwd": (C.c_int, [_vp, _vp, _i64, _vp, _vp, C.POINTER(LossParams), _vp, _sz, _vp]),
    "yb_activate_head": (C.c_int, [C.POINTER(LossParams), _vp, _vp, _i64, _vp]),
    "yb_grid_iou": (C.c_int, [_vp, _i32, _vp, _i32, _i64, _i32, _i32, _i32, _vp, _vp, _vp]),
    "yb_decode_workspace_bytes": (_sz, [C.POINTER(DecodeParams), _i64]),
    "yb_decode": (C.c_int, [C.POINTER(_vp), _i64, C.POINTER(DecodeParams), _vp, _i64, _vp, _vp, _sz, _vp]),
    "yb_loss_decode_fused": (C.c_int, [C.POINTER(LossScale), _i32, _vp, _vp, _dbl, _vp, _i64, _vp, _vp, _sz,
                                       _vp, _sz, _vp]),
    "yb_decode_finish": (C.c_int, [C.POINTER(_vp), _i64, C.POINTER(DecodeParams), _vp, _i64, _vp, _vp, _sz, _vp]),
    "yb_decode_nms_workspace_bytes": (_sz, [C.POINTER(DecodeParams), _i64, _i32]),
    "yb_decode_nms": (C.c_int, [C.POINTER(_vp), _i64, C.POINTER(DecodeParams), _dbl, _i32, _i32, _vp, _i64, _vp, _vp,
                                _vp, _sz, _vp]),
    "yb_decode_nms_finish": (C.c_int, [C.POINTER(_vp), _i64, C.POINTER(DecodeParams), _dbl, _i32, _i32, _vp, _i64, _vp,
                                       _vp, _vp, _sz, _vp]),
    "yb_loss_decode_nms_fused": (C.c_int, [C.POINTER(LossScale), _i32, _vp, _vp, _dbl, _dbl, _i32, _i32, _vp, _i64,
                                           _vp, _vp, _vp, _sz, _vp, _sz, _vp]),
    "yb_loss_decode_nms_fused_clean": (C.c_int, [C.POINTER(LossScale), _i32, _vp, _vp, _dbl, _dbl, _i32, _i32, _vp,
                                                 _i64, _vp, _vp, _vp, _sz, _vp, _sz, _vp]),
    "yb_nms_workspace_bytes": (_sz, [_i64, _i64, _i32]),
    "yb_nms": (C.c_int, [_vp, _vp, _i64, _i64, _i32, _dbl, _i32, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "yb_soft_nms": (C.c_int, [_vp, _vp, _i64, _i64, _i32, _dbl, _dbl, _dbl, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "yb_pairwise_iou": (C.c_int, [_vp, _i64, _i32, _vp, _i64, _i32, _i32, _vp, _vp]),
    "yb_elementwise_iou": (C.c_int, [_vp, _i32, _vp, _i32, _i64, _i32, _vp, _vp]),
    "yb_kmeans_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "yb_kmeans_assign": (C.c_int, [_vp, _i64, _i32, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _sz, _vp]),
    "yb_kmeans_dist": (C.c_int, [_vp, _i64, _vp, _i64, _i32, _i32, _i32, _vp, _vp]),
    "yb_kmeans_state_bytes": (_sz, [_i32, _i32]),
    "yb_kmeans_lloyd_init": (C.c_int, [_vp, _i32, _i32, _vp, _sz, _vp]),
    "yb_kmeans_lloyd_step": (C.c_int, [_vp, _i64, _i32, _vp, _i32, _i32, _dbl, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
    "yb_kmeans_lloyd_update": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _dbl, _i64, _vp, _vp]),
    "yb_peer_mailbox_bytes": (_sz, [_i32]),
    "yb_peer_alloc": (C.c_int, [_sz, C.POINTER(_vp), _vp]),
    "yb_peer_open": (C.c_int, [_vp, C.POINTER(_vp)]),
    "yb_peer_close": (C.c_int, [_vp]),
    "yb_peer_free": (C.c_int, [_vp]),
    "yb_kmeans_lloyd_step_peers": (C.c_int, [_vp, _i64, _i32, _vp, _i32, _i32, _dbl, _i64, _vp, _vp, _vp, _sz,
                                             C.POINTER(_vp), _i32, _i32, _vp]),
    "yb_minmax_f64": (C.c_int, [_vp, _i64, _vp, _vp, _sz, _vp]),
    "yb_encode_labels": (C.c_int, [_vp, _vp, _i64, _i32, _dbl, _dbl, _i32, _i32, _i32, _i32, C.POINTER(_vp), _i32,
                                   _vp, _vp]),
    "yb_down2x_labels": (C.c_int, [_vp, _i32, _i64, _i32, _i32, _i32, _vp, _vp]),
    "yb_column_sums_workspace_bytes": (_sz, [_i32]),
    "yb_column_sums": (C.c_int, [_vp, _i32, _i64, _i32, _vp, _vp, _sz, _vp]),
    "yb_map_match": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _i64, _i64, _vp, _vp, _vp, _vp]),
    "yb_map_accumulate_workspace_bytes": (_sz, [_i64, _i32]),
    "yb_map_accumulate": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _dbl, _i64, _vp, _vp, _vp, _vp, _vp,
                                    _vp, _vp, _vp, _sz, _vp]),
    "yb_map_append": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "yb_pr_points": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i64, _i32, _vp, _vp, _vp]),
    "yb_pr_curve_workspace_bytes": (_sz, [_i64, _i64]),
    "yb_pr_curve": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
}


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C tf2_yolo_b200/csrc`.  tf2_yolo_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def status_string(code):
    return lib.yb_status_string(int(code)).decode()


def check(code, what=""):
    if code != 0:
        site = lib.yb_last_error_site().decode() if code > 0 else ""
        raise YoloB200Error(f"{what or 'yolo_b200 call'} failed: status {code} ({status_string(code)})"
                            + (f" at {site}" if site else ""))
