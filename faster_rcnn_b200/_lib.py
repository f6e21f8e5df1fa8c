"""ctypes binding of libfrcnn_b200.so (C ABI declared in include/frcnn_b200.h).

The shared library is built in-tree by `faster_rcnn_b200._build.build()` (called by
`__graft_entry__.build()`); there is no CPU fallback: when the library is missing,
or no sm_100 device is present, the first call raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfrcnn_b200.so")

OK, ERR_INVALID, ERR_CUDA, ERR_UNSUPPORTED, ERR_NOMEM = 0, -1, -2, -3, -4
ROI_RESIZE, ROI_MAX = 0, 1
ROI_I16, ROI_I32, ROI_F32 = 0, 1, 2
MAX_ANCHORS, MAX_GT = 64, 256
NMS_MAX_SORTED, NMS_MAX_UNSORTED, NMS_F64_MAX = 22528, 16384, 4096

_p, _i, _d, _z, _ll = C.c_void_p, C.c_int, C.c_double, C.c_size_t, C.c_longlong

# name -> (restype, argtypes); argument order is the header's
SIGNATURES = {
    "frcnn_abi_version": (_i, []),
    "frcnn_create": (_i, [C.POINTER(_p), _i]),
    "frcnn_destroy": (None, [_p]),
    "frcnn_last_error": (C.c_char_p, [_p]),
    "frcnn_reserve": (_i, [_p, _z]),
    "frcnn_launch_count": (_ll, [_p]),
    "frcnn_decode_topk": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p]),
    "frcnn_nms_i16": (_i, [_p, _p, _p, _p, _p, _i, _i, _d, _i, _p, _p, _p, _p]),
    "frcnn_nms_f64": (_i, [_p, _p, _p, _p, _p, _i, _i, _d, _i, _i, _p, _p]),
    "frcnn_proposals": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _d, _i, _i, _p, _p, _p]),
    "frcnn_label_anchors": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _i, _i, _p, _p, _p, _p]),
    "frcnn_decode_topk_ragged": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p]),
    "frcnn_proposals_ragged": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _d, _i, _i, _p, _p, _p, _p]),
    "frcnn_label_anchors_ragged": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _i, _i, _p, _p, _p, _p, _p]),
    "frcnn_clip_rois": (_i, [_p, _p, _p, _i, _i, _i, _p, _p]),
    "frcnn_pack_rpn_targets": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _p]),
    "frcnn_label_rois": (_i, [_p, _p, _p, _p, _i, _p, _p, _p, _i, _i, _i, _p, _p, _p, _p, _p]),
    "frcnn_roi_fwd": (_i, [_p, _p, _i, _p, _i, _i, _i, _p, _i, _i, _i, _i, _p, _p]),
    "frcnn_roi_bwd": (_i, [_p, _p, _i, _p, _p, _i, _p, _i, _i, _i, _i, _i, _i, _p]),
    "frcnn_roi_compact_supported": (_i, [_i, _i, _i, _i]),
    "frcnn_roi_max_fwd_compact": (_i, [_p, _p, _p, _i, _i, _i, _p, _i, _i, _i, _i, _p, _p]),
    "frcnn_roi_max_bwd_compact": (_i, [_p, _p, _p, _p, _i, _p, _i, _i, _i, _i, _i, _i, _p]),
    "frcnn_det_postprocess": (_i, [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _d, _d, _i, _i, _p, _p, _p, _p]),
    "frcnn_cross_ious": (_i, [_p, _p, _p, _i, _i, _p, _i, _p]),
    "frcnn_box_transform": (_i, [_p, _p, _p, _p, _i, _i, _i, _i]),
    "frcnn_anchor_grid": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _p]),
    "frcnn_valid_boxes": (_i, [_p, _p, _p, _i, _p, _p]),
    "frcnn_pad_rois": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _p, _p]),
    "frcnn_gather_det_samples": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _p, _p]),
    "frcnn_rpn_losses": (_i, [_p, _p, _p, _p, _p, _p, _p, _i, _i, _p, _p, _p]),
    "frcnn_rpn_losses_ragged": (_i, [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _p, _p, _p]),
    "frcnn_det_losses": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _p, _p, _p]),
    "frcnn_voc_match": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _d, _p, _p]),
    "frcnn_voc_pr_ap": (_i, [_p, _p, _p, _p, _i, _d, _p, _i, _p, _p, _p]),
    "frcnn_image_resize_cubic": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p, _p]),
    "frcnn_image_resize_cubic_ragged": (_i, [_p, _p, _p, _p, _ll, _p, _p, _i, _i, _i, _i, _p, _p, _p]),
    "frcnn_jpeg_inspect": (_i, [_p, _ll, _p]),
    "frcnn_jpeg_decode": (_i, [_p, _p, _p, _p, _p, _p, _i, _p, _p, _ll, _p]),
    "frcnn_gt_transform": (_i, [_p, _p, _p, _p, _i, _i, _p, _p, _p]),
    "frcnn_sample_rpn": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _p, _i]),
    "frcnn_sample_rpn_ragged": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _p, _i, _i, _p, _i]),
    "frcnn_sample_det": (_i, [_p, _p, _p, _p, _i, _i, _p, _i, _p, _p]),
}

_lib = None


class FrcnnError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("frcnn_b200 error %d: %s" % (code, message))
        self.code = code


def load():
    """dlopen the library once and attach the signatures.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(
            "%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). "
            "faster_rcnn_b200 has no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype, fn.argtypes = res, args
    if lib.frcnn_abi_version() != 1:
        raise RuntimeError("libfrcnn_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(handle, rc):
    if rc != OK:
        msg = load().frcnn_last_error(handle)
        raise FrcnnError(rc, msg.decode("utf-8", "replace") if msg else "")
