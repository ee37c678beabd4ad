"""Drop-ins for the reference detection driver (src/detect.py:14-192).

``YOLO_post_process`` and ``Detect_YOLO`` keep the reference's constructor arguments, method names
(including the spelling ``non_maxium_supression``) and return types — lists of
``[x1, y1, x2, y2, conf, cls_score, cls_index]`` with Python-int coordinates — while every number is
produced by libyf_b200.so on the GPU.  The batched entry points (``postprocess_batch``,
``Detect_YOLO.detect_batch``) are what the reference's per-image Python loops turn into at B > 1.
"""
import ctypes as C
import os
import time

import numpy as np
import torch

from . import _lib
from .model import YoloFastest


def _rows_from_dets(dets):
    """structured array of yf_det -> the reference's list-of-lists rows (detect.py:65-66)."""
    return [[int(d["x1"]), int(d["y1"]), int(d["x2"]), int(d["y2"]), float(d["conf"]), float(d["cls_score"]),
             int(d["cls"])] for d in dets]


class YOLO_post_process:
    def __init__(self, conf_thres, nms_thres, num_anchors, num_class, anchors, input_shape):
        self.conf_thres = conf_thres
        self.nms_thres = nms_thres
        self.num_anchors = num_anchors
        self.num_class = num_class
        self.bbox_attrs = 5 + num_class
        self.anchors = anchors
        self.input_shape = input_shape
        self._ctx = None

    # ---- plumbing ----------------------------------------------------------------------------
    def _context(self, device, batch):
        idx = device.index if device.index is not None else torch.cuda.current_device()
        H, W = self.input_shape[0], self.input_shape[1]
        c = self._ctx
        if c is None or c.device_index != idx or c.max_batch < batch:
            if c is not None:
                torch.cuda.synchronize(c.device_index)
                c.close()
            with torch.cuda.device(idx):
                c = _lib.Ctx(idx, 1, self.num_class, self.num_anchors, batch, H, W)
            self._ctx = c
        return c

    def _params(self, mode, max_det, conf_thres=None):
        return _lib.make_params(self.anchors, self.conf_thres if conf_thres is None else conf_thres, self.nms_thres,
                                self.input_shape[0], self.input_shape[1], mode, max_det)

    @staticmethod
    def _to_cuda(t):
        if not isinstance(t, torch.Tensor):
            t = torch.as_tensor(np.asarray(t))
        if not t.is_cuda:
            if not torch.cuda.is_available():
                raise _lib.YfError("post-processing runs on the GPU only (no CPU fallback) and no CUDA device is available")
            t = t.cuda()
        return t.contiguous().float()

    DEFAULT_CAP = 256     # result slots per image of the first attempt; the call is repeated with the exact size when an image has more

    def _run(self, pred, nms, mode=_lib.MODE_DETECT, max_det=None, check_status=True):
        """-> (per-image structured arrays, true counts, status). The reference has no cap on the list length (detect.py:155-169);
        `max_det=None` reproduces that: a first pass with DEFAULT_CAP slots per image, repeated with the largest true count when
        some image holds more. An explicit `max_det` is a hard capacity: an image with more detections raises instead of being cut."""
        hl, hs = self._to_cuda(pred[0]), self._to_cuda(pred[1])
        B = hl.shape[0]
        if hl.shape[1] != self.num_anchors * self.bbox_attrs or hs.shape[1] != hl.shape[1] or hs.shape[0] != B:
            raise _lib.YfError("head shapes %s / %s do not match %d anchors x %d attrs"
                               % (tuple(hl.shape), tuple(hs.shape), self.num_anchors, self.bbox_attrs))
        ctx = self._context(hl.device, B)
        ncand = self.num_anchors * (hl.shape[2] * hl.shape[3] + hs.shape[2] * hs.shape[3])
        cap = min(ncand, self.DEFAULT_CAP) if max_det is None else max_det
        fn = _lib.lib().yf_postprocess if nms else _lib.lib().yf_decode
        stream = torch.cuda.current_stream(hl.device).cuda_stream
        while True:
            out = torch.empty((B, cap, _lib.DET_DTYPE.itemsize), dtype=torch.uint8, device=hl.device)
            counts = torch.empty((B,), dtype=torch.int32, device=hl.device)
            status = torch.empty((B,), dtype=torch.int32, device=hl.device)
            p = self._params(mode, cap)
            with torch.cuda.device(hl.device):
                _lib.check(fn(ctx.handle, hl.data_ptr(), hs.data_ptr(), B, hl.shape[2], hl.shape[3], hs.shape[2], hs.shape[3],
                              C.byref(p), out.data_ptr(), counts.data_ptr(), status.data_ptr(), C.c_void_p(stream)), ctx.handle)
            counts_h = counts.cpu().numpy()
            status_h = status.cpu().numpy()
            if check_status and (status_h & 1).any():      # decode and decode + NMS alike
                raise _lib.YfError("decoded box coordinates beyond 2^25: outside the exact-arithmetic domain of the GPU path")
            most = int(counts_h.max()) if B else 0
            if most <= cap:
                break
            if max_det is not None:
                raise _lib.YfError("an image holds %d detections, more than max_det=%d: nothing is cut silently, pass a larger max_det" % (most, max_det))
            cap = most
        kmax = max(most, 1)
        dets = out[:, :kmax].contiguous().cpu().numpy().view(_lib.DET_DTYPE).reshape(B, kmax)      # only the filled part travels
        return [dets[b, :int(counts_h[b])] for b in range(B)], counts_h, status_h

    # ---- reference API (detect.py:41-84) --------------------------------------------------------
    def decode_box(self, pred):
        """Candidates of batch element 0 with conf > conf_thres, in the reference's visiting order."""
        dets, _, _ = self._run((pred[0][0:1], pred[1][0:1]), nms=False)
        return _rows_from_dets(dets[0])

    def non_maxium_supression(self, bbox_list):
        """Greedy NMS of one class's list, already sorted by conf descending; returns the kept rows."""
        n = len(bbox_list)
        if n == 0:
            return []
        if not torch.cuda.is_available():
            raise _lib.YfError("NMS runs on the GPU only (no CPU fallback) and no CUDA device is available")
        dev = torch.device("cuda", torch.cuda.current_device())
        ctx = self._context(dev, 1)
        boxes = torch.tensor([[int(b[0]), int(b[1]), int(b[2]), int(b[3])] for b in bbox_list], dtype=torch.int32, device=dev)
        keep = torch.empty((n,), dtype=torch.int32, device=dev)
        n_keep = torch.zeros((1,), dtype=torch.int32, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().yf_nms_sorted_i32(ctx.handle, boxes.data_ptr(), n, float(self.nms_thres), keep.data_ptr(),
                                                   n_keep.data_ptr(), C.c_void_p(stream)), ctx.handle)
        k = int(n_keep.item())
        return [bbox_list[i] for i in keep[:k].cpu().tolist()]

    # ---- batched form ------------------------------------------------------------------------------
    def decode_box_batch(self, pred):
        dets, _, _ = self._run(pred, nms=False)
        return [_rows_from_dets(d) for d in dets]

    def postprocess_batch(self, pred, max_det=None, raw=False):
        """decode -> class split -> stable sort -> per-class NMS for every image (detect.py:155-169).
        Returns one list of rows per image (or the structured arrays with ``raw=True``)."""
        dets, counts, status = self._run(pred, nms=True, max_det=max_det)
        return dets if raw else [_rows_from_dets(d) for d in dets]


def plot_one_box(xyxy, img, color=None, label=None, line_thickness=None):
    """Box with an optional filled caption above its top-left corner, drawn into `img` (host-side, cv2). Call-compatible with the
    helper the reference driver uses (utils/general.py:56-67: same arguments, line width scaled with the image, anti-aliased)."""
    import cv2
    h, w = img.shape[:2]
    width = int(line_thickness) if line_thickness else int(round(0.001 * (h + w))) + 1
    if color is None:
        color = np.random.randint(0, 255, 3).tolist()
    left, top, right, bottom = (int(v) for v in xyxy[:4])
    cv2.rectangle(img, (left, top), (right, bottom), color, width, cv2.LINE_AA)
    if not label:
        return
    scale, stroke = width / 5.0, max(min(width - 1, 2), 1)
    (tw, th), _ = cv2.getTextSize(label, cv2.FONT_HERSHEY_SIMPLEX, scale, stroke)
    cv2.rectangle(img, (left, top), (left + tw, top - th - 3), color, -1, cv2.LINE_AA)          # caption background
    cv2.putText(img, label, (left, top - 2), cv2.FONT_HERSHEY_SIMPLEX, scale, (225, 255, 255), stroke, cv2.LINE_AA)


def _finish(pin_out, pin_cnt, pin_st, B, max_det, rerun):
    """Host tail of every batched detect call: status check, and NO silent truncation (the reference's lists have no cap,
    detect.py:155-169): when an image holds more than `max_det` detections the batch is run again with room for all of them."""
    if (pin_st.numpy() & 1).any():
        raise _lib.YfError("decoded box coordinates beyond 2^25: outside the exact-arithmetic domain of the GPU path")
    counts = pin_cnt.numpy()
    most = int(counts.max()) if B else 0
    if most > max_det:
        return rerun(most)
    dets = pin_out.numpy().view(_lib.DET_DTYPE).reshape(B, max_det)
    return [dets[b, :int(counts[b])].copy() for b in range(B)]


def _check_u8_host(t, input_shape, what):
    """Shared validation of the asynchronous entry points: a contiguous host uint8 tensor [B, H, W] at the network input size."""
    if not (isinstance(t, torch.Tensor) and t.dtype == torch.uint8 and t.is_contiguous() and not t.is_cuda and t.dim() == 3):
        raise _lib.YfError("%s takes a contiguous host uint8 tensor [B, H, W] (pinned for asynchronous copies)" % what)
    if list(t.shape[1:]) != list(input_shape[0:2]):
        raise _lib.YfError("images are %dx%d, the network input is %s" % (t.shape[1], t.shape[2], input_shape[0:2]))
    if input_shape[2] != 1:
        raise _lib.YfError("%s serves the single-channel networks" % what)


FRAME_ALIGN = 16          # byte alignment of every packed frame (32-bit row loads in the pre-processing kernel need 4)
MAX_FRAME_SIDE = 16384


def frame_layout(frames):
    """Validate a list of BGR uint8 frames [h, w, 3] (numpy arrays or torch tensors, sizes may differ) and lay them out back to back:
    -> (off int64 [B], Ho int32 [B], Wo int32 [B], nbytes), frame b at byte offset off[b], every offset a multiple of FRAME_ALIGN."""
    if not isinstance(frames, (list, tuple)) or len(frames) == 0:
        raise _lib.YfError("frames: a non-empty list of uint8 BGR frames [h, w, 3]")
    B = len(frames)
    off, Ho, Wo = np.zeros(B, np.int64), np.zeros(B, np.int32), np.zeros(B, np.int32)
    pos = 0
    for b, f in enumerate(frames):
        if isinstance(f, torch.Tensor):
            u8 = f.dtype == torch.uint8
        elif isinstance(f, np.ndarray):
            u8 = f.dtype == np.uint8
        else:
            raise _lib.YfError("frame %d is a %s, not a numpy array or torch tensor" % (b, type(f).__name__))
        if not u8:
            raise _lib.YfError("frame %d is %s, frames are uint8" % (b, f.dtype))
        if f.ndim != 3 or f.shape[2] != 3:
            raise _lib.YfError("frame %d has shape %s, frames are BGR [h, w, 3]" % (b, tuple(f.shape)))
        h, w = int(f.shape[0]), int(f.shape[1])
        if not (1 <= h <= MAX_FRAME_SIDE and 1 <= w <= MAX_FRAME_SIDE):
            raise _lib.YfError("frame %d is %dx%d, sizes must lie in [1, %d]" % (b, h, w, MAX_FRAME_SIDE))
        off[b], Ho[b], Wo[b] = pos, h, w
        pos += -(-h * w * 3 // FRAME_ALIGN) * FRAME_ALIGN
    return off, Ho, Wo, int(off[-1]) + int(Ho[-1]) * int(Wo[-1]) * 3


def jpeg_probe(data):
    """-> (h, w) if the device JPEG decoder takes this file (bytes / uint8 buffer), else YfError with the header parser's reason
    (progressive, arithmetic, 12-bit, CMYK, 4:1:1, several scans, RGB, EXIF-rotated, truncated, not a JPEG ...). Host only."""
    buf = np.frombuffer(data, np.uint8) if isinstance(data, (bytes, bytearray, memoryview)) else np.ascontiguousarray(data, np.uint8).reshape(-1)
    h, w = C.c_int32(), C.c_int32()
    if _lib.lib().yf_jpeg_probe(buf.ctypes.data if buf.size else None, buf.size, C.byref(h), C.byref(w)) != 0:
        raise _lib.YfError(_lib.lib().yf_last_error(None).decode())
    return h.value, w.value


def _file_bytes(f):
    """a path, bytes or a uint8 numpy buffer -> bytes"""
    if isinstance(f, (str, os.PathLike)):
        with open(f, "rb") as fh:
            return fh.read()
    if isinstance(f, (bytes, bytearray, memoryview)):
        return bytes(f)
    if isinstance(f, np.ndarray) and f.dtype == np.uint8:
        return f.tobytes()
    raise _lib.YfError("a JPEG file is a path, bytes or a uint8 numpy buffer, not %s" % type(f).__name__)


def jpeg_layout(datas):
    """Probe every file and lay the files and their decoded frames out back to back -> (files uint8 [nbytes], off int64 [B],
    len int64 [B], frame_off int64 [B], Ho int32 [B], Wo int32 [B], frames_bytes). Raises YfError naming the first file not taken."""
    if not datas:
        raise _lib.YfError("files: a non-empty list")
    B = len(datas)
    off, ln, foff = np.zeros(B, np.int64), np.zeros(B, np.int64), np.zeros(B, np.int64)
    Ho, Wo = np.zeros(B, np.int32), np.zeros(B, np.int32)
    pos = fpos = 0
    for b, d in enumerate(datas):
        try:
            Ho[b], Wo[b] = jpeg_probe(d)
        except _lib.YfError as e:
            raise _lib.YfError("file %d: %s" % (b, e)) from None
        off[b], ln[b], foff[b] = pos, len(d), fpos
        pos += len(d)
        fpos += -(-int(Ho[b]) * int(Wo[b]) * 3 // FRAME_ALIGN) * FRAME_ALIGN
    files = np.frombuffer(b"".join(datas), np.uint8)
    return files, off, ln, foff, Ho, Wo, int(foff[-1]) + int(Ho[-1]) * int(Wo[-1]) * 3


def pack_frames(frames, dst, off):
    """Copy host frames into the uint8 numpy buffer `dst` at the offsets of frame_layout (any strides)."""
    for f, o in zip(frames, off):
        a = f.numpy() if isinstance(f, torch.Tensor) else f
        dst[int(o):int(o) + a.size].reshape(a.shape)[...] = a


class Detect_YOLO:
    def __init__(self, device, model_path, config_params, logger):
        device = torch.device(device)
        if device.type != "cuda":
            raise _lib.YfError("Detect_YOLO of the B200 path needs a CUDA device (no CPU fallback), got %s" % device)
        io = config_params["io_params"]
        self.model = YoloFastest(io).to(device).eval()
        net_param = torch.load(model_path, map_location="cpu")
        self.model.load_state_dict(net_param)
        self.logger = logger
        self.device = device
        self.class_names = io["class_names"]
        self.num_cls = io["num_cls"]
        self.nms_thres = io["nms_thre"]
        self.conf_thres = io["conf_thre"]
        self.input_shape = io["input_shape"]
        self.origin_img_shape = io["origin_img_shape"]
        self.post_process = YOLO_post_process(conf_thres=self.conf_thres, nms_thres=self.nms_thres,
                                              num_anchors=io["num_anchors"], anchors=io["anchors"],
                                              input_shape=self.input_shape, num_class=self.num_cls)
        self.colors = [[106, 90, 205], [199, 97, 20], [112, 128, 105]]
        self._pinned = {}
        self._slots = {}
        self._frames_pin = None        # grow-only pinned staging of packed host frames (pre_process_frames / detect_frames)
        self._frames_ev = None         # end of the last asynchronous copy out of it

    # ---- host-side image handling (unchanged semantics, detect.py:107-139) ------------------------
    def _load_gray(self, img_path):
        """imread -> (gray) -> resize: the uint8 network input, [H, W] for the single-channel models, [3, H, W] in RGB plane
        order for 3-channel ones (detect.py:107-122: cvtColor only when the network is single-channel, then `[:, :, ::-1]` and
        HWC -> CHW)."""
        import cv2
        ori_img = cv2.imread(img_path)
        if self.input_shape[2] == 1 and self.origin_img_shape[2] != 1:
            img = cv2.cvtColor(ori_img, cv2.COLOR_BGR2GRAY)
        else:
            img = ori_img
        if list(self.input_shape[0:2]) != list(self.origin_img_shape[0:2]):
            img = cv2.resize(img, (self.input_shape[1], self.input_shape[0]))
        if self.input_shape[2] == 1:
            if img.ndim != 2:
                raise _lib.YfError("a single-channel network needs gray input: origin_img_shape[2] must not be 1 for 3-channel files")
            return np.ascontiguousarray(img), ori_img
        return np.ascontiguousarray(img[:, :, ::-1].transpose(2, 0, 1)), ori_img

    def pre_process(self, img_path):
        """imread -> gray -> resize -> (x - 128) / 255 -> [1, C, H, W] on the device (detect.py:107-129)."""
        u8, ori_img = self._load_gray(img_path)
        img = torch.from_numpy(u8[None] if u8.ndim == 2 else u8).to(self.device).float()
        img = (img - 128.0) / 255.0
        return img.unsqueeze(0), ori_img

    def adjust_coord(self, rows):
        """round(coord * origin/input) in place, after NMS (detect.py:131-139)."""
        scale_h = self.origin_img_shape[0] / self.input_shape[0]
        scale_w = self.origin_img_shape[1] / self.input_shape[1]
        for r in rows:
            r[0] = round(r[0] * scale_w)
            r[2] = round(r[2] * scale_w)
            r[1] = round(r[1] * scale_h)
            r[3] = round(r[3] * scale_h)

    # ---- pre-processing on the device (SURVEY 8f-1; detect.py:107-122) ------------------------------------
    def pre_process_batch(self, bgr):
        """BGR uint8 frames [B, Ho, Wo, 3] as cv2.imread returns them (host numpy / torch, or a cuda uint8 tensor) ->
        cuda uint8 [B, H, W]: cv2.cvtColor(BGR2GRAY) + cv2.resize(INTER_LINEAR) computed on the device, byte-identical
        to the host path (yf_preprocess_bgr). The normalisation is applied by the first convolution of the u8 paths."""
        t = bgr if isinstance(bgr, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(bgr, dtype=np.uint8))
        if t.dtype != torch.uint8 or t.dim() != 4 or t.shape[3] != 3:
            raise _lib.YfError("pre_process_batch takes uint8 frames [B, Ho, Wo, 3]")
        t = t.to(self.device).contiguous()
        B, Ho, Wo, _ = t.shape
        H, W = self.input_shape[0:2]
        ctx = self.model.context(self.device, H, W, B)
        out = torch.empty((B, H, W), dtype=torch.uint8, device=self.device)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().yf_preprocess_bgr(ctx.handle, t.data_ptr(), B, Ho, Wo, out.data_ptr(), C.c_void_p(stream)), ctx.handle)
        return out

    def detect_bgr_batch(self, bgr, max_det=64, raw=False, adjust=True):
        """Frames as cv2.imread returns them, uint8 [B, Ho, Wo, 3] on the host -> per-image rows: one yf_detect_host_bgr
        call (H2D of the frames, gray + resize + normalisation + forward + decode + NMS on the device, D2H of the result
        slab). With adjust=True the boxes are mapped back to the frame like Detect_YOLO.__adjust_coord (detect.py:131-139,
        applied when the frame and network sizes differ, as batch_detect does)."""
        t = bgr if isinstance(bgr, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(bgr, dtype=np.uint8))
        if t.dtype != torch.uint8 or t.dim() != 4 or t.shape[3] != 3 or t.is_cuda:
            raise _lib.YfError("detect_bgr_batch takes host uint8 frames [B, Ho, Wo, 3]")
        t = t.contiguous()
        B, Ho, Wo, _ = t.shape
        H, W = self.input_shape[0:2]
        ctx = self.model.context(self.device, H, W, B)
        pin_out = torch.empty((B, max_det, _lib.DET_DTYPE.itemsize), dtype=torch.uint8).pin_memory()
        pin_cnt = torch.empty((B,), dtype=torch.int32).pin_memory()
        pin_st = torch.empty((B,), dtype=torch.int32).pin_memory()
        p = self.post_process._params(_lib.MODE_DETECT, max_det)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().yf_detect_host_bgr(ctx.handle, t.data_ptr(), B, Ho, Wo, C.byref(p), pin_out.data_ptr(),
                                                    pin_cnt.data_ptr(), pin_st.data_ptr(), C.c_void_p(stream)), ctx.handle)
        res = _finish(pin_out, pin_cnt, pin_st, B, max_det, lambda need: self.detect_bgr_batch(bgr, max_det=need, raw=True, adjust=False))
        if raw:
            return res
        rows = [_rows_from_dets(d) for d in res]
        if adjust and [Ho, Wo] != [H, W]:
            scale_h, scale_w = Ho / H, Wo / W
            for rr in rows:
                for r in rr:
                    r[0] = round(r[0] * scale_w)
                    r[2] = round(r[2] * scale_w)
                    r[1] = round(r[1] * scale_h)
                    r[3] = round(r[3] * scale_h)
        return rows

    # ---- frames of mixed sizes, gray or colour networks (yf_preprocess_frames / yf_detect_host_frames) --------------------------
    def _frames_pinned(self, nbytes):
        if self._frames_ev is not None:
            self._frames_ev.synchronize()           # the previous copy out of the buffer has finished before it is rewritten
            self._frames_ev = None
        if self._frames_pin is None or self._frames_pin.numel() < nbytes:
            self._frames_pin = None
            self._frames_pin = torch.empty((nbytes,), dtype=torch.uint8).pin_memory()
        return self._frames_pin

    def pre_process_frames(self, frames):
        """A list of BGR uint8 frames [h_i, w_i, 3] as cv2.imread returns them, sizes free (all numpy / host torch, or all cuda
        tensors) -> cuda uint8 [B, H, W] gray for single-channel networks, [B, 3, H, W] R, G, B planes for 3-channel ones: the
        image half of detect.py:107-122 for each frame, byte-identical to OpenCV, in one kernel launch per 512 frames. Host frames
        are packed into a pinned buffer and copied once; cuda frames are packed on the device."""
        off, Ho, Wo, nbytes = frame_layout(frames)
        on_dev = [isinstance(f, torch.Tensor) and f.is_cuda for f in frames]
        if any(on_dev) and not all(on_dev):
            raise _lib.YfError("pre_process_frames: frames must be all on the host or all on the device")
        B = len(frames)
        H, W, chans = self.input_shape[0:3]
        ctx = self.model.context(self.device, H, W, B)
        out = torch.empty((B, H, W) if chans == 1 else (B, chans, H, W), dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device)
            packed = torch.empty((nbytes,), dtype=torch.uint8, device=self.device)
            if all(on_dev):
                for f, o in zip(frames, off):
                    packed[int(o):int(o) + f.numel()].view(f.shape).copy_(f)
            else:
                pin = self._frames_pinned(nbytes)
                pack_frames(frames, pin.numpy(), off)
                packed.copy_(pin[:nbytes], non_blocking=True)
                self._frames_ev = torch.cuda.Event()
                self._frames_ev.record(stream)
            _lib.check(_lib.lib().yf_preprocess_frames(ctx.handle, packed.data_ptr(), B, off.ctypes.data, Ho.ctypes.data, Wo.ctypes.data,
                                                      out.data_ptr(), C.c_void_p(stream.cuda_stream)), ctx.handle)
        return out

    def detect_frames(self, frames, max_det=64, raw=False, adjust=True):
        """Host BGR uint8 frames [h_i, w_i, 3] of any sizes (a list) -> per-image rows: one yf_detect_host_frames call (one copy of
        the packed frames, pre-processing, forward, decode, NMS, the result slab back), for gray and colour networks alike.
        With adjust=True each frame's boxes are mapped back to THAT frame's size with the arithmetic of adjust_coord
        (round(v * (h_i / H)), round(v * (w_i / W)); detect.py:131-139), which is batch_detect's result for a frame of
        origin_img_shape."""
        off, Ho, Wo, nbytes = frame_layout(frames)
        if any(isinstance(f, torch.Tensor) and f.is_cuda for f in frames):
            raise _lib.YfError("detect_frames takes host frames (pre_process_frames serves cuda frames)")
        B = len(frames)
        H, W = self.input_shape[0:2]
        ctx = self.model.context(self.device, H, W, B)
        pin = self._frames_pinned(nbytes)
        pack_frames(frames, pin.numpy(), off)
        pin_out = torch.empty((B, max_det, _lib.DET_DTYPE.itemsize), dtype=torch.uint8).pin_memory()
        pin_cnt = torch.empty((B,), dtype=torch.int32).pin_memory()
        pin_st = torch.empty((B,), dtype=torch.int32).pin_memory()
        p = self.post_process._params(_lib.MODE_DETECT, max_det)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().yf_detect_host_frames(ctx.handle, pin.data_ptr(), nbytes, B, off.ctypes.data, Ho.ctypes.data,
                                                       Wo.ctypes.data, C.byref(p), pin_out.data_ptr(), pin_cnt.data_ptr(),
                                                       pin_st.data_ptr(), C.c_void_p(stream)), ctx.handle)
        res = _finish(pin_out, pin_cnt, pin_st, B, max_det, lambda need: self.detect_frames(frames, max_det=need, raw=True, adjust=False))
        if raw:
            return res
        rows = [_rows_from_dets(d) for d in res]
        if adjust:
            for rr, h, w in zip(rows, Ho, Wo):
                if [int(h), int(w)] == [H, W]:
                    continue
                scale_h, scale_w = int(h) / H, int(w) / W
                for r in rr:
                    r[0] = round(r[0] * scale_w)
                    r[2] = round(r[2] * scale_w)
                    r[1] = round(r[1] * scale_h)
                    r[3] = round(r[3] * scale_h)
        return rows

    # ---- JPEG files decoded on the device (yf_decode_jpeg / yf_detect_host_jpeg) ---------------------------------------------------
    def decode_jpeg(self, files):
        """JPEG files (paths, bytes or uint8 numpy buffers) -> list of cuda uint8 [h, w, 3] BGR tensors, byte-identical to
        cv2.imread / cv2.imdecode(IMREAD_COLOR). Every header is checked first (jpeg_probe); a file the decoder does not take raises
        YfError naming its index before anything runs on the device, and a file whose scan data is corrupt raises after the decode."""
        datas = [_file_bytes(f) for f in files]
        files_u8, off, ln, foff, Ho, Wo, fbytes = jpeg_layout(datas)
        B = len(datas)
        H, W = self.input_shape[0:2]
        ctx = self.model.context(self.device, H, W, B)
        frames = torch.empty((fbytes,), dtype=torch.uint8, device=self.device)
        status = torch.zeros((B,), dtype=torch.int32, device=self.device)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().yf_decode_jpeg(ctx.handle, files_u8.ctypes.data, files_u8.size, B, off.ctypes.data, ln.ctypes.data,
                                                frames.data_ptr(), foff.ctypes.data, fbytes, status.data_ptr(), C.c_void_p(stream)),
                       ctx.handle)
        st = status.cpu().numpy()         # synchronises the stream, so files_u8 may go
        bad = np.nonzero(st & _lib.STATUS_JPEG_CORRUPT)[0]
        if bad.size:
            raise _lib.YfError("file %d: corrupt JPEG entropy-coded data" % int(bad[0]))
        return [frames[int(o):int(o) + int(h) * int(w) * 3].view(int(h), int(w), 3) for o, h, w in zip(foff, Ho, Wo)]

    def detect_jpeg(self, files, max_det=64, raw=False, adjust=True, return_frames=False):
        """JPEG files (paths, bytes or uint8 numpy buffers) -> per-image rows equal to detect_frames([cv2.imread(f) ...]): one
        yf_detect_host_jpeg call (one copy of the files, decode, pre-processing, forward, decode, NMS, the result slab back), for gray
        and colour networks. adjust as in detect_frames. With return_frames=True also returns the decoded BGR frames (host numpy), for
        drawing. A file the decoder does not take raises YfError naming its index; nothing is launched then."""
        datas = [_file_bytes(f) for f in files]
        files_u8, off, ln, foff, Ho, Wo, fbytes = jpeg_layout(datas)
        rows, frames = self._detect_jpeg(files_u8, off, ln, foff, Ho, Wo, fbytes, max_det, return_frames)
        if not raw:
            rows = [_rows_from_dets(d) for d in rows]
            if adjust:
                H, W = self.input_shape[0:2]
                for rr, h, w in zip(rows, Ho, Wo):
                    if [int(h), int(w)] == [H, W]:
                        continue
                    scale_h, scale_w = int(h) / H, int(w) / W
                    for r in rr:
                        r[0] = round(r[0] * scale_w)
                        r[2] = round(r[2] * scale_w)
                        r[1] = round(r[1] * scale_h)
                        r[3] = round(r[3] * scale_h)
        return (rows, frames) if return_frames else rows

    def _detect_jpeg(self, files_u8, off, ln, foff, Ho, Wo, fbytes, max_det, want_frames):
        B = len(off)
        H, W = self.input_shape[0:2]
        ctx = self.model.context(self.device, H, W, B)
        pin_out = torch.empty((B, max_det, _lib.DET_DTYPE.itemsize), dtype=torch.uint8).pin_memory()
        pin_cnt = torch.empty((B,), dtype=torch.int32).pin_memory()
        pin_st = torch.empty((B,), dtype=torch.int32).pin_memory()
        frames = np.empty((fbytes,), np.uint8) if want_frames else None
        p = self.post_process._params(_lib.MODE_DETECT, max_det)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().yf_detect_host_jpeg(ctx.handle, files_u8.ctypes.data, files_u8.size, B, off.ctypes.data, ln.ctypes.data,
                                                     foff.ctypes.data, C.byref(p), pin_out.data_ptr(), pin_cnt.data_ptr(), pin_st.data_ptr(),
                                                     frames.ctypes.data if want_frames else None, C.c_void_p(stream)), ctx.handle)
        bad = np.nonzero(pin_st.numpy() & _lib.STATUS_JPEG_CORRUPT)[0]
        if bad.size:
            raise _lib.YfError("file %d: corrupt JPEG entropy-coded data" % int(bad[0]))
        res = _finish(pin_out, pin_cnt, pin_st, B, max_det,
                      lambda need: self._detect_jpeg(files_u8, off, ln, foff, Ho, Wo, fbytes, need, False)[0])
        if want_frames:
            frames = [frames[int(o):int(o) + int(h) * int(w) * 3].reshape(int(h), int(w), 3) for o, h, w in zip(foff, Ho, Wo)]
        return res, frames

    # ---- batched detection through the C ABI with host buffers -----------------------------------------
    def detect_batch(self, u8_batch, max_det=64, raw=False):
        """uint8 images [B, H, W] (gray) or [B, 3, H, W] (RGB planes, 3-channel networks), host numpy array or host torch
        tensor at the network input size -> per-image rows.

        One yf_detect_host_u8 call: H2D copy of the bytes, fused normalisation + forward + decode +
        NMS, D2H copy of the fixed-capacity result slab.  This is the end-to-end call bench.py times."""
        direct = isinstance(u8_batch, torch.Tensor) and u8_batch.dtype == torch.uint8 and not u8_batch.is_cuda \
            and u8_batch.is_contiguous()
        if not direct:
            u8_batch = np.ascontiguousarray(u8_batch, dtype=np.uint8)
        B, H, W = u8_batch.shape[0], u8_batch.shape[-2], u8_batch.shape[-1]
        chans = 1 if u8_batch.ndim == 3 else u8_batch.shape[1]
        if [H, W] != list(self.input_shape[0:2]) or chans != self.input_shape[2] or u8_batch.ndim not in (3, 4):
            raise _lib.YfError("images are %s, the network input is %s" % (tuple(u8_batch.shape[1:]), self.input_shape))
        ctx = self.model.context(self.device, H, W, B)
        key = (B, max_det)
        if key not in self._pinned:
            self._pinned = {key: (torch.empty((B, chans, H, W), dtype=torch.uint8).pin_memory(),
                                  torch.empty((B, max_det, _lib.DET_DTYPE.itemsize), dtype=torch.uint8).pin_memory(),
                                  torch.empty((B,), dtype=torch.int32).pin_memory(),
                                  torch.empty((B,), dtype=torch.int32).pin_memory())}
        pin_in, pin_out, pin_cnt, pin_st = self._pinned[key]
        if direct:
            pin_in = u8_batch            # a host tensor (ideally pinned) is handed to the C ABI as is
        else:
            pin_in.numpy()[...] = u8_batch.reshape(B, chans, H, W)
        p = self.post_process._params(_lib.MODE_DETECT, max_det)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().yf_detect_host_u8(ctx.handle, pin_in.data_ptr(), B, C.byref(p), pin_out.data_ptr(),
                                                   pin_cnt.data_ptr(), pin_st.data_ptr(), C.c_void_p(stream)), ctx.handle)
        res = _finish(pin_out, pin_cnt, pin_st, B, max_det, lambda need: self.detect_batch(u8_batch, max_det=need, raw=True))
        return res if raw else [_rows_from_dets(d) for d in res]

    def submit_batch(self, u8_pinned, slot, max_det=64):
        """Asynchronous form of detect_batch for serving loops (yf_detect_submit_u8): `u8_pinned` is a pinned host
        uint8 tensor [B, H, W] that must stay untouched until `collect(slot)`. Submitting the next batch into the
        other slot before collecting this one overlaps its host-to-device copy with this batch's compute."""
        _check_u8_host(u8_pinned, self.input_shape, "submit_batch")
        B, H, W = u8_pinned.shape
        ctx = self.model.context(self.device, H, W, B)
        st = self._slots.get(slot)
        if st is None or st[0] != (B, max_det):
            st = ((B, max_det), torch.empty((B, max_det, _lib.DET_DTYPE.itemsize), dtype=torch.uint8).pin_memory(),
                  torch.empty((B,), dtype=torch.int32).pin_memory(), torch.empty((B,), dtype=torch.int32).pin_memory())
            self._slots[slot] = st
        _, pin_out, pin_cnt, pin_st = st
        p = self.post_process._params(_lib.MODE_DETECT, max_det)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().yf_detect_submit_u8(ctx.handle, slot, u8_pinned.data_ptr(), B, C.byref(p), pin_out.data_ptr(),
                                                     pin_cnt.data_ptr(), pin_st.data_ptr()), ctx.handle)
        self._slot_ref = getattr(self, "_slot_ref", {})
        self._slot_ref[slot] = u8_pinned          # keep the input alive until collected
        ctx.pending.add(slot)

    def submit_batch_device(self, u8_pinned, slot, max_det=64):
        """As submit_batch, but the results stay on the device: returns (dets uint8 [B, max_det, 56], counts int32 [B])
        cuda tensors that are complete once `wait(slot)` has returned (multi-GPU jobs gather them with NCCL). counts[b] may exceed
        max_det: the slab then holds the first max_det records of image b in (class, conf) order — check it where that can happen."""
        _check_u8_host(u8_pinned, self.input_shape, "submit_batch_device")
        B, H, W = u8_pinned.shape
        ctx = self.model.context(self.device, H, W, B)
        key = ("dev", slot)
        st = self._slots.get(key)
        if st is None or st[0] != (B, max_det):
            st = ((B, max_det), torch.empty((B, max_det, _lib.DET_DTYPE.itemsize), dtype=torch.uint8, device=self.device),
                  torch.empty((B,), dtype=torch.int32, device=self.device))
            self._slots[key] = st
        _, out, cnt = st
        p = self.post_process._params(_lib.MODE_DETECT, max_det)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().yf_detect_submit_u8_dev(ctx.handle, slot, u8_pinned.data_ptr(), B, C.byref(p), out.data_ptr(),
                                                         cnt.data_ptr(), None), ctx.handle)
        self._slot_ref = getattr(self, "_slot_ref", {})
        self._slot_ref[slot] = u8_pinned
        ctx.pending.add(slot)
        return out, cnt

    def wait(self, slot):
        ctx = self.model._ctx
        _lib.check(_lib.lib().yf_detect_wait(ctx.handle, slot), ctx.handle)
        self._slot_ref.pop(slot, None)
        ctx.pending.discard(slot)

    def collect(self, slot, raw=False):
        """Wait for the batch submitted into `slot` and return its per-image detections."""
        ctx = self.model._ctx
        (B, max_det), pin_out, pin_cnt, pin_st = self._slots[slot]
        _lib.check(_lib.lib().yf_detect_wait(ctx.handle, slot), ctx.handle)
        src = self._slot_ref.pop(slot, None)
        ctx.pending.discard(slot)
        res = _finish(pin_out, pin_cnt, pin_st, B, max_det, lambda need: self.detect_batch(src, max_det=need, raw=True))
        return res if raw else [_rows_from_dets(d) for d in res]

    def detect_device(self, x, max_det=64):
        """Device-resident form: x cuda fp32 [B, 1, H, W] (already normalised) -> (dets uint8 [B, max_det, 56],
        counts int32 [B], status int32 [B]) cuda tensors, enqueued on the current stream, no synchronisation."""
        self.model._check_input(x)
        x = x.contiguous().float()
        B, _, H, W = x.shape
        ctx = self.model.context(x.device, H, W, B)
        out = torch.empty((B, max_det, _lib.DET_DTYPE.itemsize), dtype=torch.uint8, device=x.device)
        counts = torch.empty((B,), dtype=torch.int32, device=x.device)
        status = torch.empty((B,), dtype=torch.int32, device=x.device)
        p = self.post_process._params(_lib.MODE_DETECT, max_det)
        stream = torch.cuda.current_stream(x.device).cuda_stream
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().yf_detect(ctx.handle, x.data_ptr(), B, C.byref(p), out.data_ptr(), counts.data_ptr(),
                                           status.data_ptr(), C.c_void_p(stream)), ctx.handle)
        return out, counts, status

    # ---- reference driver (detect.py:141-192) ------------------------------------------------------------
    def batch_detect(self, data_path, result_path):
        import cv2
        with torch.no_grad():
            img_list = os.listdir(data_path)
            num = len(img_list)
            avg_time = 0
            for filename in img_list:
                img_path = os.path.join(data_path, filename)
                img, ori_img = self.pre_process(img_path)

                torch.cuda.synchronize(self.device)
                start_time = time.time()
                pred = self.model(img)
                torch.cuda.synchronize(self.device)     # the reference omits this, so its GPU numbers would be launch times
                time_mark = time.time()
                infer_time = float(time_mark - start_time) * 1000

                all_bbox_rects = self.post_process.postprocess_batch(pred)[0]
                post_process_time = float(time.time() - time_mark) * 1000
                total_time = infer_time + post_process_time
                avg_time += total_time

                if len(all_bbox_rects) == 0:
                    cv2.imwrite(os.path.join(result_path, 'result_' + filename), ori_img)
                    self.logger.info("image_name:%s -> no targets, infer time:%.2fms, post_process time:%.2fms, total time:%.2fms"
                                     % (filename, infer_time, post_process_time, total_time))
                    continue

                if list(self.input_shape[0:2]) != list(self.origin_img_shape[0:2]):
                    self.adjust_coord(all_bbox_rects)

                for *xyxy, conf, cls_score, cls_pred in all_bbox_rects:
                    label = '%s %.2f' % (self.class_names[int(cls_pred)], conf * cls_score)
                    plot_one_box(xyxy, ori_img, label=label, color=self.colors[int(cls_pred)], line_thickness=3)

                cv2.imwrite(os.path.join(result_path, 'result_' + filename), ori_img)
                self.logger.info("image_name:%s -> detect finished, infer time:%.2fms, post_process time:%.2fms, total time:%.2fms"
                                 % (filename, infer_time, post_process_time, total_time))

            self.logger.info("detect avg_time: %.2fms" % (avg_time / num))

    # Smallest batch the file driver decodes on the device. One thread decodes a whole file, so a batch costs at least one file's
    # decode (12 ms for a shipped 640x512 file, DESIGN.md §5.7): on 1024 files the device path took 1.80 s against 2.42 s for
    # cv2.imread at batch 32, and 2.87 s against 2.05 s at batch 8 (profiles/r04_jpeg.txt).
    JPEG_MIN_BATCH = 32

    def batch_detect_batched(self, data_path, result_path, batch_size=32):
        """batch_detect with the per-file loop turned into batches (SURVEY 8f-1). When a batch holds at least JPEG_MIN_BATCH files and
        the device decoder takes every one of them (jpeg_probe), the batch is ONE yf_detect_host_jpeg call: JPEG decode, gray / resize, normalisation, forward, decode and NMS on
        the device, the decoded frames back for drawing. Any other batch (PNGs, progressive or EXIF-rotated JPEGs, ...) is decoded on
        the host (cv2.imread) and is one yf_detect_host_bgr call, or one detect_frames call when its frames differ in size or the
        network is 3-channel (boxes scaled to each frame's own size). Same result files and log lines as batch_detect
        (detect.py:141-192); the two per-image times of the log line are the batch's time divided by its size, and include the
        decode on the device path."""
        import cv2
        img_list = os.listdir(data_path)
        num = len(img_list)
        avg_time = 0
        for i0 in range(0, num, batch_size):
            names = img_list[i0:i0 + batch_size]
            datas = []
            for n in names:
                with open(os.path.join(data_path, n), "rb") as f:
                    datas.append(f.read())
            on_device = len(names) >= self.JPEG_MIN_BATCH
            if on_device:
                try:
                    jpeg_layout(datas)
                except _lib.YfError:
                    on_device = False
            if not on_device:
                frames = [cv2.imread(os.path.join(data_path, n)) for n in names]
            torch.cuda.synchronize(self.device)
            start_time = time.time()
            if on_device:
                rows, frames = self.detect_jpeg(datas, return_frames=True)
            elif self.input_shape[2] == 1 and all(f.shape == frames[0].shape for f in frames):
                rows = self.detect_bgr_batch(np.stack(frames))
            else:
                rows = self.detect_frames(frames)
            total_time = float(time.time() - start_time) * 1000 / len(names)
            avg_time += total_time * len(names)
            for filename, ori_img, all_bbox_rects in zip(names, frames, rows):
                if len(all_bbox_rects) == 0:
                    cv2.imwrite(os.path.join(result_path, 'result_' + filename), ori_img)
                    self.logger.info("image_name:%s -> no targets, infer time:%.2fms, post_process time:%.2fms, total time:%.2fms"
                                     % (filename, total_time, 0.0, total_time))
                    continue
                for *xyxy, conf, cls_score, cls_pred in all_bbox_rects:
                    label = '%s %.2f' % (self.class_names[int(cls_pred)], conf * cls_score)
                    plot_one_box(xyxy, ori_img, label=label, color=self.colors[int(cls_pred)], line_thickness=3)
                cv2.imwrite(os.path.join(result_path, 'result_' + filename), ori_img)
                self.logger.info("image_name:%s -> detect finished, infer time:%.2fms, post_process time:%.2fms, total time:%.2fms"
                                 % (filename, total_time, 0.0, total_time))
        self.logger.info("detect avg_time: %.2fms" % (avg_time / max(num, 1)))
