"""CPU oracle for YUV 4:2:0 frames.  TEST INFRASTRUCTURE ONLY (same rules as yolo_oracle.py: only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s CPU legs may import it).

Restates ``cv2.cvtColor(frame, cv2.COLOR_YUV2BGR_NV12)`` and ``cv2.COLOR_YUV2BGR_I420`` for 8-bit frames (OpenCV 4.x, imgproc
color_yuv): BT.601 limited range in 20-bit fixed point, no chroma interpolation (pixel (r, c) takes chroma sample (r / 2, c / 2)):

    y = max(Y - 16, 0) * 1220542 + 2^19;   u = U - 128;   v = V - 128
    R = sat((y + 1673527 * v) >> 20);   G = sat((y - 852492 * v - 409993 * u) >> 20);   B = sat((y + 2116026 * u) >> 20)

Parity pin: tests/test_yuv_cpu.py checks it against live cv2 for every (Y, U, V) triple, in both formats.
"""
import numpy as np


def yuv_to_bgr(Y, U, V):
    """Y uint8 [h, w], U and V uint8 [h / 2, w / 2] (any strides) -> BGR uint8 [h, w, 3]. Every intermediate fits in int32."""
    y = np.maximum(Y.astype(np.int32) - 16, 0) * 1220542 + (1 << 19)
    u = np.repeat(np.repeat(U.astype(np.int32) - 128, 2, 0), 2, 1)
    v = np.repeat(np.repeat(V.astype(np.int32) - 128, 2, 0), 2, 1)
    r = (y + 1673527 * v) >> 20
    g = (y - 852492 * v - 409993 * u) >> 20
    b = (y + 2116026 * u) >> 20
    return np.clip(np.stack([b, g, r], -1), 0, 255).astype(np.uint8)


def planes(frame, fmt):
    """cv2's single-array form uint8 [3h / 2, w] -> (Y [h, w], U [h / 2, w / 2], V [h / 2, w / 2]) views of it.
    nv12: the interleaved UV rows follow the luma rows; i420: the U plane, then the V plane, each (h / 2) * (w / 2) bytes."""
    h, w = frame.shape[0] * 2 // 3, frame.shape[1]
    Y = frame[:h]
    if fmt == "nv12":
        uv = frame[h:].reshape(h // 2, w // 2, 2)
        return Y, uv[:, :, 0], uv[:, :, 1]
    c = np.ascontiguousarray(frame[h:]).reshape(-1)
    n = (h // 2) * (w // 2)
    return Y, c[:n].reshape(h // 2, w // 2), c[n:2 * n].reshape(h // 2, w // 2)


def to_bgr(frame, fmt):
    """cv2.cvtColor(frame, COLOR_YUV2BGR_NV12 / COLOR_YUV2BGR_I420) of a frame in cv2's form."""
    return yuv_to_bgr(*planes(frame, fmt))


def from_planes(Y, U, V, fmt):
    """(Y, U, V) -> cv2's single-array form [3h / 2, w] in the given format."""
    h, w = Y.shape
    if fmt == "nv12":
        return np.concatenate([Y, np.stack([U, V], -1).reshape(h // 2, w)], 0)
    return np.concatenate([Y.reshape(-1), U.reshape(-1), V.reshape(-1)]).reshape(h * 3 // 2, w)
