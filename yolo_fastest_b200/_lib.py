"""ctypes binding of libyf_b200.so (include/yf.h).  No CPU fallback: a missing library raises."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("YF_B200_LIB", os.path.join(_HERE, "libyf_b200.so"))   # override: tuning builds only

YF_MAX_ANCHORS = 8
MODE_DETECT = 0
MODE_VALIDATE = 1
VARIANT_FULL = 0
VARIANT_LITE = 1
STATUS_JPEG_CORRUPT = 4


class YfError(RuntimeError):
    pass


class YfDet(C.Structure):
    _fields_ = [("x1", C.c_double), ("y1", C.c_double), ("x2", C.c_double), ("y2", C.c_double),
                ("conf", C.c_double), ("cls_score", C.c_double), ("cls", C.c_int32), ("src", C.c_int32)]


DET_DTYPE = np.dtype([("x1", "<f8"), ("y1", "<f8"), ("x2", "<f8"), ("y2", "<f8"), ("conf", "<f8"),
                      ("cls_score", "<f8"), ("cls", "<i4"), ("src", "<i4")])
assert DET_DTYPE.itemsize == C.sizeof(YfDet) == 56


class YfPostParams(C.Structure):
    _fields_ = [("anchors", C.c_double * 2 * YF_MAX_ANCHORS * 2),
                ("conf_thres", C.c_double), ("nms_thres", C.c_double),
                ("input_h", C.c_int32), ("input_w", C.c_int32), ("mode", C.c_int32), ("max_det", C.c_int32)]


# every symbol include/yf.h declares: (name, restype, argtypes)
_P = C.c_void_p
SYMBOLS = [
    ("yf_create", C.c_int, [C.POINTER(_P), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    ("yf_create_variant", C.c_int, [C.POINTER(_P), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    ("yf_destroy", None, [_P]),
    ("yf_last_error", C.c_char_p, [_P]),
    ("yf_abi_version", C.c_int, []),
    ("yf_weight_count", C.c_int64, [C.c_int, C.c_int, C.c_int]),
    ("yf_weight_count_variant", C.c_int64, [C.c_int, C.c_int, C.c_int, C.c_int]),
    ("yf_load_weights", C.c_int, [_P, _P, C.c_int64]),
    ("yf_forward", C.c_int, [_P, _P, C.c_int, _P, _P, _P]),
    ("yf_tap", C.c_int, [_P, C.c_char_p, C.c_int, _P, C.POINTER(C.c_int64), _P]),
    ("yf_postprocess", C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(YfPostParams), _P, _P, _P, _P]),
    ("yf_decode", C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(YfPostParams), _P, _P, _P, _P]),
    ("yf_val_decode", C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double), C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    ("yf_val_nms", C.c_int, [_P, _P, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, _P, _P, _P, _P]),
    ("yf_nms_sorted_i32", C.c_int, [_P, _P, C.c_int, C.c_double, _P, _P, _P]),
    ("yf_nms_sorted_f32", C.c_int, [_P, _P, C.c_int, C.c_float, _P, _P, _P]),
    ("yf_detect", C.c_int, [_P, _P, C.c_int, C.POINTER(YfPostParams), _P, _P, _P, _P]),
    ("yf_detect_host", C.c_int, [_P, _P, C.c_int, C.POINTER(YfPostParams), _P, _P, _P, _P]),
    ("yf_detect_host_u8", C.c_int, [_P, _P, C.c_int, C.POINTER(YfPostParams), _P, _P, _P, _P]),
    ("yf_detect_submit_u8", C.c_int, [_P, C.c_int, _P, C.c_int, C.POINTER(YfPostParams), _P, _P, _P]),
    ("yf_detect_wait", C.c_int, [_P, C.c_int]),
    ("yf_detect_submit_u8_dev", C.c_int, [_P, C.c_int, _P, C.c_int, C.POINTER(YfPostParams), _P, _P, _P]),
    ("yf_preprocess_bgr", C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P]),
    ("yf_detect_host_bgr", C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.POINTER(YfPostParams), _P, _P, _P, _P]),
    ("yf_preprocess_frames", C.c_int, [_P, _P, C.c_int, _P, _P, _P, _P, _P]),
    ("yf_detect_host_frames", C.c_int, [_P, _P, C.c_int64, C.c_int, _P, _P, _P, C.POINTER(YfPostParams), _P, _P, _P, _P]),
    ("yf_jpeg_probe", C.c_int, [_P, C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    ("yf_decode_jpeg", C.c_int, [_P, _P, C.c_int64, C.c_int, _P, _P, _P, _P, C.c_int64, _P, _P]),
    ("yf_detect_host_jpeg", C.c_int, [_P, _P, C.c_int64, C.c_int, _P, _P, _P, C.POINTER(YfPostParams), _P, _P, _P, _P, _P]),
    ("yf_compact_dets", C.c_int, [_P, _P, _P, C.c_int, C.c_int, _P, C.c_int, C.c_int, _P]),
    ("yf_launch_count", C.c_int64, [_P]),
    ("yf_profile_forward", C.c_int, [_P, _P, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_float), C.c_int]),
]

_lib = None


def lib():
    """Load the shared library (once). Raises YfError if it has not been built — there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise YfError("%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(the B200 path has no CPU or PyTorch fallback)" % LIB_PATH)
        l = C.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        if l.yf_abi_version() != 1:
            raise YfError("libyf_b200.so ABI version %d, expected 1" % l.yf_abi_version())
        _lib = l
    return _lib


def check(rc, ctx=None):
    if rc != 0:
        msg = lib().yf_last_error(ctx)
        raise YfError("yf error %d: %s" % (rc, msg.decode() if msg else "?"))


def make_params(anchors, conf_thres, nms_thres, input_h, input_w, mode, max_det):
    """anchors: [[(w,h)]*A for head_large, [(w,h)]*A for head_small] in input pixels."""
    p = YfPostParams()
    for hd in range(2):
        for a, (w, h) in enumerate(anchors[hd]):
            p.anchors[hd][a][0] = float(w)
            p.anchors[hd][a][1] = float(h)
    p.conf_thres = float(conf_thres)
    p.nms_thres = float(nms_thres)
    p.input_h = int(input_h)
    p.input_w = int(input_w)
    p.mode = int(mode)
    p.max_det = int(max_det)
    return p


class Ctx:
    """Owner of one yf_ctx (one device, one input size, a maximum batch)."""

    def __init__(self, device_index, in_ch, num_cls, num_anchors, max_batch, H, W, variant=0):
        self.handle = _P()
        self.variant = variant
        self.device_index, self.in_ch, self.num_cls, self.num_anchors = device_index, in_ch, num_cls, num_anchors
        self.max_batch, self.H, self.W = max_batch, H, W
        self.nout = num_anchors * (5 + num_cls)
        self.ncand = num_anchors * ((H // 16) * (W // 16) + (H // 32) * (W // 32))
        self.pending = set()          # slots of the asynchronous path holding a submitted, not yet collected batch
        l = lib()
        check(l.yf_create_variant(C.byref(self.handle), device_index, in_ch, num_cls, num_anchors, max_batch, H, W, variant), None)

    def close(self):
        if self.handle:
            lib().yf_destroy(self.handle)
            self.handle = _P()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def load_weights(self, blob):
        blob = np.ascontiguousarray(blob, dtype=np.float32)
        check(lib().yf_load_weights(self.handle, blob.ctypes.data_as(_P), blob.size), self.handle)

    def launch_count(self):
        return int(lib().yf_launch_count(self.handle))
