"""B200-native YOLO-Fastest detection hot path: the reference's Python API over libyf_b200.so.

    from yolo_fastest_b200 import YoloFastest, YOLO_post_process, Detect_YOLO, config_for

Importing the package does not need a GPU; any compute call does (there is no CPU fallback).
"""
from ._lib import LIB_PATH, YfError, lib  # noqa: F401
from .config import COCO_ANCHORS, config_for, config_params  # noqa: F401
from .detector import (Detect_YOLO, YOLO_post_process, frame_layout, jpeg_encode_bound, jpeg_encode_header, jpeg_probe,  # noqa: F401
                       plot_one_box, yuv_layout)
from .model import YoloFastest, YoloFastest_lite  # noqa: F401
from .val import YOLOLossV3, non_max_suppression  # noqa: F401
from .validate import Validation  # noqa: F401
