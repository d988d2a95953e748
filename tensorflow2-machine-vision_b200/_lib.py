"""ctypes binding of libb200det.so (declared in include/b200det.h)."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200det.so")
_lib = None

c_f = ctypes.c_float
c_i = ctypes.c_int
c_p = ctypes.c_void_p
c_sz = ctypes.c_size_t

# name -> (restype, argtypes); every symbol include/b200det.h declares
SIGNATURES = {
    "b200_last_error": (ctypes.c_char_p, []),
    "b200_version": (c_i, []),
    "b200_device_ok": (c_i, []),
    "b200_set_l2_fetch_granularity": (c_i, [c_i]),
    "b200_get_l2_fetch_granularity": (c_i, []),
    "b200_detmath_eval": (c_i, [c_i, c_p, c_p, c_p, c_sz, c_p]),
    "b200_pairwise_iou": (c_i, [c_p, c_i, c_p, c_i, c_i, c_p, c_p]),
    "b200_elementwise_iou": (c_i, [c_p, c_p, c_sz, c_i, c_p, c_p]),
    "b200_ciou_v_grad": (c_i, [c_p, c_p, c_p, c_p, c_p, c_sz, c_p, c_p, c_p, c_p]),
    "b200_nms": (c_i, [c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_f, c_i, c_f, c_i, c_p, c_p, c_p]),
    "b200_yolo_decode_nms_workspace_bytes": (c_sz, [c_p, c_i, c_i, c_i]),
    "b200_yolo_decode_nms": (c_i, [c_p, c_p, c_i, c_i, c_i, c_p, c_p, c_f, c_f, c_f, c_i, c_i,
                                   c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_sz, c_p]),
    "b200_yolo_decode_dense": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p]),
    "b200_yolo_loss_workspace_bytes": (c_sz, [c_p, c_i, c_i]),
    "b200_yolo_loss": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_p, c_p, c_f, c_i, c_i, c_f, c_p, c_p, c_p, c_p, c_sz, c_p]),
    "b200_unletterbox_boxes": (c_i, [c_p, c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    "b200_letterbox_image": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p]),
    "b200_letterbox_batch": (c_i, [c_i, c_p, c_p, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    "b200_unletterbox_boxes_batch": (c_i, [c_p, c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p]),
    "b200_yolo_loss_stages": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_p, c_p, c_f, c_i, c_i, c_f, c_p, c_p, c_p, c_sz, c_i, c_p]),
    "b200_yolo_loss_grad": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_p, c_p, c_f, c_i, c_i, c_f, c_p, c_p, c_p, c_p, c_sz, c_p]),
    "b200_yolo_loss_from_boxes_workspace_bytes": (c_sz, [c_p, c_i, c_i, c_i]),
    "b200_yolo_loss_from_boxes": (c_i, [c_p, c_p, c_p, c_i, c_p, c_p, c_p, c_i, c_i, c_i, c_p, c_p, c_f, c_i, c_i, c_f, c_p, c_p,
                                        c_p, c_p, c_sz, c_p]),
    "b200_yolo_loss_from_boxes_grad": (c_i, [c_p, c_p, c_p, c_i, c_p, c_p, c_p, c_i, c_i, c_i, c_p, c_p, c_f, c_i, c_i, c_f, c_p,
                                             c_p, c_p, c_p, c_sz, c_p]),
    "b200_yolo_assign_targets": (c_i, [c_p, c_p, c_p, c_i, c_i, c_p, c_i, c_p, c_i, c_p, c_p, c_i, c_p]),
    "b200_fill_zero": (c_i, [c_p, c_sz, c_p]),
    "b200_yolo_reset_targets": (c_i, [c_p, c_p, c_i, c_i, c_p, c_i, c_p, c_i, c_p, c_p, c_p]),
    "b200_effdet_table_floats": (c_sz, [c_i, c_p, c_i]),
    "b200_effdet_anchors": (c_i, [c_i, c_p, c_i, c_p, c_i, c_p, c_p]),
    "b200_effdet_decode": (c_i, [c_i, c_p, c_i, c_p, c_i, c_p, c_p, c_p]),
    "b200_effdet_postprocess_workspace_bytes": (c_sz, [c_i, c_p, c_i, c_i, c_i]),
    "b200_effdet_postprocess": (c_i, [c_i, c_p, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_i, c_f, c_f, c_i,
                                      c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_sz, c_p]),
    "b200_effdet_assign_targets": (c_i, [c_i, c_p, c_i, c_p, c_i, c_i, c_p, c_p, c_p, c_f, c_p, c_p, c_p, c_p]),
    "b200_focal_elementwise": (c_i, [c_p, c_p, c_sz, c_f, c_f, c_f, c_f, c_p, c_p]),
    "b200_focal_box_workspace_bytes": (c_sz, [c_i, c_p, c_i]),
    "b200_effdet_assign_targets_indexed": (c_i, [c_i, c_p, c_i, c_p, c_i, c_i, c_p, c_p, c_p, c_f, c_p, c_p, c_p, c_p]),
    "b200_focal_box_partial_sums_indexed": (c_i, [c_i, c_p, c_i, c_p, c_p, c_p, c_p, c_p, c_f, c_f, c_f, c_f, c_p, c_p, c_sz, c_p]),
    "b200_focal_box_partial_sums": (c_i, [c_i, c_p, c_i, c_p, c_p, c_p, c_p, c_p, c_f, c_f, c_f, c_f, c_p, c_p, c_sz, c_p]),
    "b200_focal_box_grad": (c_i, [c_i, c_p, c_i, c_p, c_p, c_p, c_p, c_f, c_f, c_f, c_f, c_p, c_p, c_p, c_p, c_p]),
    "b200_focal_box_grad_indexed": (c_i, [c_i, c_p, c_i, c_p, c_p, c_p, c_p, c_f, c_f, c_f, c_f, c_p, c_p, c_p, c_p, c_p]),
    "b200_focal_box_finalize": (c_i, [c_i, c_p, c_p, c_p, c_p, c_p, c_p]),
    "b200_effdet_loss_from_boxes_workspace_bytes": (c_sz, [c_i, c_p, c_i, c_i]),
    "b200_effdet_loss_from_boxes_match": (c_i, [c_i, c_p, c_i, c_p, c_i, c_p, c_p, c_i, c_f, c_p, c_p, c_sz, c_p]),
    "b200_effdet_loss_from_boxes_grad": (c_i, [c_i, c_p, c_i, c_p, c_i, c_i, c_p, c_p, c_i, c_p, c_p, c_f, c_f, c_f, c_f, c_p, c_p,
                                               c_p, c_p, c_p, c_sz, c_p]),
    "b200_row_positions_workspace_bytes": (c_sz, [ctypes.c_longlong]),
    "b200_row_positions": (c_i, [c_p, ctypes.c_longlong, c_p, c_p, c_p, c_sz, c_p]),
    "b200_gather_rows": (c_i, [c_p, c_i, c_p, c_p, ctypes.c_longlong, c_p, c_p]),
    "b200_yolo_ground_truth_rows": (c_i, [c_p, ctypes.c_longlong, c_i, c_p, c_p, c_p]),
    "b200_peer_mailbox_bytes": (c_sz, []),
    "b200_peer_mailbox_create": (c_i, [c_p, c_p]),
    "b200_peer_mailbox_open": (c_i, [c_p, c_p]),
    "b200_peer_mailbox_close": (c_i, [c_p]),
    "b200_peer_mailbox_destroy": (c_i, [c_p]),
    "b200_peer_mailbox_status": (c_i, [c_p, c_p, c_p]),
    "b200_allreduce_loss_peer": (c_i, [c_p, c_i, c_i, c_i, c_p, c_p]),
    "b200_allreduce_sums_peer": (c_i, [c_p, c_i, c_i, c_i, c_p, c_p]),
    "b200_peer_exchange_selftest": (c_i, [c_i, c_i, c_i, c_p, c_sz, c_p, c_p]),
    "b200_yolo_loss_dp": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_p, c_p, c_f, c_i, c_i, c_f, c_p, c_p, c_p, c_sz, c_i, c_i, c_p, c_p]),
    "b200_yolo_loss_dp_publish": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_p, c_p, c_f, c_i, c_i, c_f, c_p, c_p, c_p, c_sz, c_i, c_i, c_p, c_p]),
    "b200_yolo_loss_collect_peer": (c_i, [c_p, c_p, c_i, c_i, c_p, c_p]),
    "b200_yolo_loss_from_boxes_dp": (c_i, [c_p, c_p, c_p, c_i, c_p, c_p, c_p, c_i, c_i, c_i, c_p, c_p, c_f, c_i, c_i, c_f, c_p, c_p,
                                           c_p, c_sz, c_i, c_i, c_p, c_p]),
    "b200_focal_box_finalize_dp": (c_i, [c_i, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_p, c_p]),
    "b200_nccl_unique_id": (c_i, [c_p]),
    "b200_nccl_comm_init": (c_i, [c_p, c_i, c_i, c_p]),
    "b200_nccl_comm_destroy": (c_i, [c_p]),
    "b200_allreduce_loss": (c_i, [c_p, c_p, c_i, c_p]),
    "b200_allreduce_sums": (c_i, [c_p, c_p, c_i, c_p]),
    "b200_yolo_loss_combine": (c_i, [c_p, c_p, c_p]),
    "b200_effdet_eval_workspace_bytes": (c_sz, [c_i, c_p, c_i, c_i, c_i]),
    "b200_effdet_eval_step": (c_i, [c_i, c_p, c_i, c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_f, c_f, c_f, c_f, c_p, c_p, c_i, c_f, c_f,
                                    c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_sz, c_p]),
    "b200_effdet_decode_postprocess": (c_i, [c_i, c_p, c_i, c_p, c_i, c_i, c_p, c_p, c_p, c_i, c_f, c_f, c_i, c_p, c_p, c_p, c_p, c_p,
                                             c_p, c_p, c_sz, c_p]),
    "b200_map_per_image": (c_i, [c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, ctypes.c_double, c_p, c_p]),
}

METRIC_YOLO = {"iou": 0, "diou": 1, "ciou": 2}
METRIC_EFF = {"iou": 3, "giou": 4, "diou": 5, "ciou": 6}
NMS_AGNOSTIC, NMS_BY_CLASS = 0, 1


def load():
    """Load the library once.  Raises RuntimeError (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libb200det.so not found at %s - build it with `python tensorflow2-machine-vision_b200/build.py` "
                "(or __graft_entry__.build()); this package has no CPU fallback" % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(status, what):
    if status != 0:
        msg = load().b200_last_error().decode("utf-8", "replace")
        if status == -1:
            raise ValueError("%s: %s" % (what, msg))
        raise RuntimeError("%s failed (%d): %s" % (what, status, msg))
