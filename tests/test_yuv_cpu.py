"""YUV 4:2:0 frames without a GPU: the oracle against live cv2 for every (Y, U, V) triple in both formats and on pitched, odd-aligned
layouts; descriptors built from host frames; every refusal with its reason; the bound C entry points and the descriptor size."""
import ctypes as C

import numpy as np
import pytest
import torch

import yolo_fastest_b200 as yf
from oracle import yuv_oracle as yo
from yolo_fastest_b200 import _lib
from yolo_fastest_b200.detector import FRAME_ALIGN, pack_yuv, yuv_layout

FMTS = ["nv12", "i420"]
CODE = {"nv12": "COLOR_YUV2BGR_NV12", "i420": "COLOR_YUV2BGR_I420"}


def all_triples():
    """One 4096x4096 frame holding every (Y, U, V) triple: 2x2 block k carries chroma pair k mod 2^16 and luma values 4 (k >> 16) ..
    4 (k >> 16) + 3, so each of the 2^16 (U, V) pairs meets all 256 luma values."""
    k = np.arange(1 << 22, dtype=np.int64).reshape(2048, 2048)
    U, V = (k & 255).astype(np.uint8), ((k >> 8) & 255).astype(np.uint8)
    base = (4 * (k >> 16)).astype(np.uint8)
    Y = np.empty((4096, 4096), np.uint8)
    for a in range(2):
        for b in range(2):
            Y[a::2, b::2] = base + 2 * a + b
    return Y, U, V


@pytest.mark.parametrize("fmt", FMTS)
def test_oracle_every_triple_matches_live_cv2(fmt):
    cv2 = pytest.importorskip("cv2")
    Y, U, V = all_triples()
    frame = yo.from_planes(Y, U, V, fmt)
    want = cv2.cvtColor(frame, getattr(cv2, CODE[fmt]))
    got = yo.to_bgr(frame, fmt)
    assert got.shape == want.shape == (4096, 4096, 3)
    assert np.array_equal(got, want)
    key = (Y.astype(np.int64)[::2, ::2] >> 2) << 16 | V.astype(np.int64) << 8 | U       # every triple present exactly once per block
    assert np.unique(key).size == 1 << 22


def _read_planes(buf, d):
    """The planes a yf_yuv420 descriptor names in a byte buffer, read with its offsets, pitches and chroma step."""
    h, w = int(d["h"]), int(d["w"])
    Y = np.stack([buf[int(d["y_off"]) + r * int(d["y_pitch"]):][:w] for r in range(h)])
    idx = np.arange(w // 2) * int(d["c_step"])
    U = np.stack([buf[int(d["u_off"]) + r * int(d["c_pitch"]) + idx] for r in range(h // 2)])
    V = np.stack([buf[int(d["v_off"]) + r * int(d["c_pitch"]) + idx] for r in range(h // 2)])
    return Y, U, V


def _pitched(rng, h, w, fmt, y_off, y_pitch, c_gap, c_pitch_pad):
    """A buffer with the planes of a random frame at odd offsets and pitches, like a decoder surface -> (buf, descriptor, frame)."""
    Y = rng.integers(0, 256, (h, w), dtype=np.uint8)
    U = rng.integers(0, 256, (h // 2, w // 2), dtype=np.uint8)
    V = rng.integers(0, 256, (h // 2, w // 2), dtype=np.uint8)
    d = np.zeros(1, _lib.YUV_DTYPE)[0]
    step = 2 if fmt == "nv12" else 1
    c_pitch = (w // 2) * step + c_pitch_pad
    u_off = y_off + h * y_pitch + c_gap
    v_off = u_off + 1 if fmt == "nv12" else u_off + (h // 2) * c_pitch + c_gap
    d["y_off"], d["u_off"], d["v_off"], d["y_pitch"], d["c_pitch"], d["c_step"], d["h"], d["w"] = \
        y_off, u_off, v_off, y_pitch, c_pitch, step, h, w
    buf = rng.integers(0, 256, v_off + (h // 2) * c_pitch + 7, dtype=np.uint8)
    for r in range(h):
        buf[y_off + r * y_pitch:][:w] = Y[r]
    idx = np.arange(w // 2) * step
    for r in range(h // 2):
        buf[u_off + r * c_pitch + idx] = U[r]
        buf[v_off + r * c_pitch + idx] = V[r]
    return buf, d, yo.from_planes(Y, U, V, fmt)


@pytest.mark.parametrize("fmt", FMTS)
def test_oracle_on_pitched_and_odd_layouts(fmt):
    """The descriptor's reading of a surface (odd offsets, pitches wider than the row, chroma after a padded height) gives planes whose
    oracle conversion is cv2's conversion of the same frame in cv2's own form."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(31)
    for (h, w, y_off, y_pitch, c_gap, c_pad) in [(8, 6, 1, 7, 3, 1), (1080, 1920, 3, 2048, 8 * 2048, 128), (2, 2, 0, 2, 0, 0),
                                                  (34, 50, 5, 61, 1, 3), (6, 1922, 2, 1923, 5, 2)]:
        buf, d, frame = _pitched(rng, h, w, fmt, y_off, y_pitch, c_gap, c_pad)
        assert _lib.lib().yf_yuv420_check(buf.size, 1, d.tobytes()) == 0
        Y, U, V = _read_planes(buf, d)
        assert np.array_equal(yo.yuv_to_bgr(Y, U, V), cv2.cvtColor(frame, getattr(cv2, CODE[fmt]))), (fmt, h, w)


@pytest.mark.parametrize("fmt", FMTS)
def test_descriptors_of_host_frames(fmt):
    """Host frames in cv2's form: packed back to back at FRAME_ALIGN, descriptors in cv2's layout, and the packed bytes read back
    through the descriptors are the frames' planes (a strided NV12 view is packed as its values)."""
    rng = np.random.default_rng(5)
    sizes = [(2, 2), (6, 10), (480, 640), (8, 4)]
    frames = [rng.integers(0, 256, (h * 3 // 2, w), dtype=np.uint8) for h, w in sizes]
    frames[3] = torch.from_numpy(frames[3])
    if fmt == "nv12":
        frames[1] = rng.integers(0, 256, (9, 20), dtype=np.uint8)[:, ::2]
    desc, on_dev, base, nbytes = yuv_layout(frames, fmt)
    assert not on_dev and base is None and desc.dtype == _lib.YUV_DTYPE
    assert list(desc["h"]) == [h for h, _ in sizes] and list(desc["w"]) == [w for _, w in sizes]
    assert desc["y_off"][0] == 0 and all(o % FRAME_ALIGN == 0 for o in desc["y_off"])
    assert nbytes == desc["y_off"][-1] + 8 * 3 // 2 * 4
    for d in desc:
        h, w, o = int(d["h"]), int(d["w"]), int(d["y_off"])
        assert d["y_pitch"] == w and d["u_off"] == o + h * w
        if fmt == "nv12":
            assert (d["v_off"], d["c_pitch"], d["c_step"]) == (o + h * w + 1, w, 2)
        else:
            assert (d["v_off"], d["c_pitch"], d["c_step"]) == (o + h * w + (h // 2) * (w // 2), w // 2, 1)
    buf = np.zeros(nbytes, np.uint8)
    pack_yuv(frames, buf, desc)
    for f, d in zip(frames, desc):
        a = f.numpy() if isinstance(f, torch.Tensor) else f
        for got, want in zip(_read_planes(buf, d), yo.planes(np.ascontiguousarray(a), fmt)):
            assert np.array_equal(got, want)


@pytest.mark.parametrize("bad, fmt, reason", [
    ([np.zeros((6, 4), np.uint8)], "yuv444", "fmt"),
    ([np.zeros((6, 4), np.uint8)], "NV12", "fmt"),
    ([], "nv12", "non-empty"),
    ([np.zeros((6, 5), np.uint8)], "nv12", "even"),                    # odd width (cv2's form cannot hold an odd height)
    ([np.zeros((7, 4), np.uint8)], "nv12", "[3h / 2, w]"),             # rows not a multiple of 3
    ([np.zeros((6, 4, 1), np.uint8)], "nv12", "[3h / 2, w]"),
    ([np.zeros((6, 4), np.float32)], "nv12", "uint8"),
    ([np.zeros((24579, 2), np.uint8)], "nv12", "even and in [2, 16384]"),          # h = 16386
    ([[0, 1, 2]], "nv12", "not a numpy array"),
    ([np.zeros((12, 8), np.uint8)[:, :4]], "i420", "contiguous"),     # a row-padded i420 view
    ([np.zeros((6, 4), np.uint8), (torch.zeros(4, 4, dtype=torch.uint8), torch.zeros(2, 4, dtype=torch.uint8))], "nv12",
     "all on the host or all on the device"),
    ([(torch.zeros(4, 4, dtype=torch.uint8), torch.zeros(2, 4, dtype=torch.uint8))], "nv12", "cuda"),
])
def test_layout_refusals(bad, fmt, reason):
    with pytest.raises(yf.YfError) as e:
        yuv_layout(bad, fmt)
    assert reason in str(e.value)


def test_layout_refusal_names_the_frame():
    ok = np.zeros((6, 4), np.uint8)
    with pytest.raises(yf.YfError, match=r"frame 1 is 6x5: YUV 4:2:0 sizes are even"):
        yuv_layout([ok, np.zeros((9, 5), np.uint8)], "nv12")
    with pytest.raises(yf.YfError, match=r"frame 2 has shape \(8, 4\)"):
        yuv_layout([ok, ok, np.zeros((8, 4), np.uint8)], "i420")


def _check(desc, nbytes):
    d = np.array(desc, _lib.YUV_DTYPE) if not isinstance(desc, np.ndarray) else desc
    rc = _lib.lib().yf_yuv420_check(nbytes, d.size, d.ctypes.data)
    return rc, _lib.lib().yf_last_error(None).decode()


def _desc(**kw):
    d = np.zeros(1, _lib.YUV_DTYPE)
    f = dict(y_off=0, u_off=32, v_off=33, y_pitch=8, c_pitch=8, c_step=2, h=4, w=8)
    f.update(kw)
    for k, v in f.items():
        d[0][k] = v
    return d


def test_library_checks_and_reasons():
    """yf_yuv420_check holds the checks of the three entry points: each refusal carries its reason and names the frame."""
    assert _check(_desc(), 48)[0] == 0                                  # NV12 4x8 in exactly 48 bytes
    cases = [
        (dict(h=3), "size 3x8: YUV 4:2:0 sizes are even"), (dict(w=0), "size 4x0"), (dict(w=16386, y_pitch=16386), "size 4x16386"),
        (dict(y_pitch=7), "luma pitch 7 below the width 8"), (dict(c_step=0), "chroma step 0 below 1"),
        (dict(c_pitch=7), "chroma pitch 7 below 4 samples of step 2"),
        (dict(y_off=-1), "luma plane bytes [-1, 31)"), (dict(u_off=33, v_off=34), "V plane bytes [34, 49) outside the 48-byte buffer"),
        (dict(u_off=34), "U plane bytes [34, 49)"),
    ]
    for kw, reason in cases:
        rc, msg = _check(np.concatenate([_desc(), _desc(**kw)]), 48)
        assert rc == -1 and msg.startswith("frame 1: ") and reason in msg, (kw, msg)
    assert _check(_desc(), 47)[0] == -1
    assert _lib.lib().yf_yuv420_check(48, 0, _desc().ctypes.data) == -1
    # I420 4x8 in cv2's layout: 32 luma bytes, then 2x4 U and 2x4 V
    assert _check(_desc(u_off=32, v_off=40, c_pitch=4, c_step=1), 48)[0] == 0
    assert _check(_desc(u_off=32, v_off=41, c_pitch=4, c_step=1), 48)[0] == -1


def test_yuv_symbols_and_struct_size():
    assert C.sizeof(_lib.YfYuv420) == 48 and _lib.YUV_DTYPE.itemsize == 48
    assert [f[0] for f in _lib.YfYuv420._fields_] == list(_lib.YUV_DTYPE.names)
    assert _lib.YUV_DTYPE.fields["h"][1] == 36 and _lib.YUV_DTYPE.fields["w"][1] == 40
    l = _lib.lib()
    names = [s[0] for s in _lib.SYMBOLS]
    for name, nargs, i64 in (("yf_yuv420_check", 3, (0,)), ("yf_yuv420_to_bgr", 9, (2, 7)), ("yf_preprocess_yuv420", 7, (2,)),
                             ("yf_detect_yuv420", 10, (2,))):
        assert name in names
        fn = getattr(l, name)
        assert fn.restype is C.c_int and len(fn.argtypes) == nargs
        for i in i64:
            assert fn.argtypes[i] is C.c_int64, (name, i)
    assert l.yf_detect_yuv420.argtypes[5] is C.POINTER(_lib.YfPostParams)
