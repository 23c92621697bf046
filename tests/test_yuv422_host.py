"""CPU checks of the packed YUV 4:2:2 formats (FDT_FMT_YUYV / _UYVY / _YVYU): the constants against the C header, the
frame-size math, the argument checks that must fail before any call into the library, and the numpy restatement of the pixel
rule that the GPU tests' references rest on, pinned against cv2.cvtColor."""
import re
from pathlib import Path

import cv2
import numpy as np
import pytest

from face_detection_tflite_b200 import _ffi
from face_detection_tflite_b200.face_detector import _frame_geometry, _row_step

HEADER = Path(__file__).resolve().parents[1] / "include" / "fdt_api.h"
NEW = (_ffi.FDT_FMT_YUYV, _ffi.FDT_FMT_UYVY, _ffi.FDT_FMT_YVYU)
CV = {_ffi.FDT_FMT_YUYV: cv2.COLOR_YUV2BGR_YUYV, _ffi.FDT_FMT_UYVY: cv2.COLOR_YUV2BGR_UYVY, _ffi.FDT_FMT_YVYU: cv2.COLOR_YUV2BGR_YVYU}
# byte offsets of (Y from 2x, U and V from the macropixel at 4 * (x / 2)), as include/fdt_api.h states them
RULE = {_ffi.FDT_FMT_YUYV: (0, 1, 3), _ffi.FDT_FMT_UYVY: (1, 0, 2), _ffi.FDT_FMT_YVYU: (0, 3, 1)}


def yuv422_to_bgr(frame: np.ndarray, w: int, h: int, mt: int, stride: int) -> np.ndarray:
    """The header's pixel rule and the library's BT.601 fixed-point conversion (kernels.h yuv_to_bgr), in numpy."""
    rows = np.frombuffer(np.ascontiguousarray(frame).tobytes(), np.uint8)[:h * stride].reshape(h, stride).astype(np.int64)
    yo, uo, vo = RULE[mt]
    x = np.arange(w)
    m = 4 * (x // 2)
    Y, U, V = rows[:, 2 * x + yo], rows[:, m + uo], rows[:, m + vo]
    yy = np.maximum(Y - 16, 0) * 1220542 + (1 << 19)
    u, v = U - 128, V - 128
    b = (yy + 2116026 * u) >> 20
    g = (yy - 852492 * v - 409993 * u) >> 20
    r = (yy + 1673527 * v) >> 20
    return np.clip(np.stack([b, g, r], -1), 0, 255).astype(np.uint8)


def test_constants_match_header():
    text = HEADER.read_text()
    for name in ("FDT_FMT_YUYV", "FDT_FMT_UYVY", "FDT_FMT_YVYU"):
        m = re.search(r"\b%s = (0x[0-9A-Fa-f]+|\d+)" % name, text)
        assert m, name
        assert getattr(_ffi, name) == int(m.group(1), 0), name
    assert _ffi.YUV422_FORMATS == NEW == (0x1020, 0x1021, 0x1022)
    # no cv MatType (at most 4095) and no other FDT_FMT_* value collides
    others = {int(v, 0) for k, v in re.findall(r"\b(FDT_FMT_\w+) = (0x[0-9A-Fa-f]+|\d+)", text) if k not in
              ("FDT_FMT_YUYV", "FDT_FMT_UYVY", "FDT_FMT_YVYU")}
    assert others and not others & set(NEW) and min(NEW) > 4095
    assert not set(NEW) & set(_ffi.YUV_FORMATS + _ffi.RGB_FORMATS + (_ffi.FDT_MAT_8UC1, _ffi.FDT_MAT_8UC3, _ffi.FDT_MAT_8UC4))


@pytest.mark.parametrize("w,h", [(1280, 720), (1920, 1080), (130, 97), (6, 4), (2, 1)])
def test_frame_geometry(w, h):
    for mt in NEW:
        assert _row_step(mt) == 2
        assert _frame_geometry(0, w, h, mt, None) == (2 * w, 2 * w * h)
        assert _frame_geometry(0, w, h, mt, 2 * w + 3) == (2 * w + 3, (2 * w + 3) * h)     # odd strides are allowed
        assert _frame_geometry(0, w, h, mt, 2 * w + 64) == (2 * w + 64, (2 * w + 64) * h)
        with pytest.raises(ValueError):
            _frame_geometry(0, w, h, mt, 2 * w - 1)
        with pytest.raises(ValueError):
            _frame_geometry(0, w + 1, h, mt, None)                                           # odd width
    # the existing formats are unchanged
    assert _frame_geometry(0, w, h, _ffi.FDT_MAT_8UC3, None) == (3 * w, 3 * w * h)
    assert _frame_geometry(0, w, h, _ffi.FDT_FMT_RGB_PLANAR, None) == (w, 3 * w * h)


@pytest.mark.parametrize("w,h", [(1280, 720), (1920, 1080), (14, 34), (130, 97), (6, 3), (2, 1)])
@pytest.mark.parametrize("mt", NEW)
def test_pixel_rule_equals_cv2(mt, w, h):
    """The GPU tests' reference is the BGR call on cv2.cvtColor(frame); this pins that it is the header's rule, including odd
    heights and padded, odd row strides."""
    rng = np.random.default_rng(w * 7 + h + mt)
    img = rng.integers(0, 256, (h, w, 2), dtype=np.uint8)
    want = cv2.cvtColor(img, CV[mt])
    assert np.array_equal(yuv422_to_bgr(img, w, h, mt, 2 * w), want)
    for pad in (3, 16):
        buf = rng.integers(0, 256, (h, 2 * w + pad), dtype=np.uint8)
        buf[:, :2 * w] = img.reshape(h, 2 * w)
        assert np.array_equal(yuv422_to_bgr(buf, w, h, mt, 2 * w + pad), want)


class _NoLibrary:
    def __getattr__(self, name):
        raise AssertionError("the argument checks must fail before %s is called" % name)


@pytest.fixture
def detector(lib):
    import face_detection_tflite_b200 as fdt
    d = fdt.FaceDetector()
    d._lib = _NoLibrary()
    d._ready = True             # past the state check: only the argument checks stand between the call and the library
    return d


@pytest.mark.parametrize("layout", ["yuyv", "uyvy", "yvyu"])
@pytest.mark.parametrize("shape", [(4, 6, 3), (4, 6), (4, 6, 1), (4, 12), (4, 5, 2), (0, 6, 2), (4, 0, 2), (2, 4, 6, 2)])
def test_wrong_shape_for_layout(detector, layout, shape):
    m = np.zeros(shape, np.uint8)
    with pytest.raises(ValueError):
        detector.detectFacesFromMat(m, layout=layout)
    with pytest.raises(ValueError):
        detector.detectFacesFromMats([np.zeros((4, 6, 2), np.uint8), m], layout=layout)


@pytest.mark.parametrize("layout", ["yuyv", "uyvy", "yvyu"])
def test_wrong_dtype(detector, layout):
    for dt in (np.uint16, np.float32, np.int8):
        with pytest.raises(ValueError):
            detector.detectFacesFromMat(np.zeros((4, 6, 2), dt), layout=layout)
    with pytest.raises(ValueError):
        detector.detectFacesFromMat(np.zeros((4, 6, 2), np.uint8), layout="YUYV")


@pytest.mark.parametrize("mt", NEW)
def test_raw_call_checks(detector, mt):
    data = np.zeros(4 * 64, np.uint8)
    # odd width
    with pytest.raises(ValueError):
        detector.detectFramesRaw([(data[:4 * 10], 5, 4, mt)])
    with pytest.raises(ValueError):
        detector.detectBatchRaw(data[:4 * 10], count=1, width=5, height=4, matType=mt)
    with pytest.raises(ValueError):
        detector.detectFacesFromMatBytes(data[:4 * 10], width=5, height=4, matType=mt)
    with pytest.raises(ValueError):
        detector.detectFacesFromMatBytes(data[:4 * 10], width=5, height=4, matType=mt, orientation=6)
    # a row stride below 2 * width
    with pytest.raises(ValueError):
        detector.detectFramesRaw([(data[:4 * 11], 6, 4, mt, 11)])
    with pytest.raises(ValueError):
        detector.detectBatchRaw(data[:4 * 11], count=1, width=6, height=4, matType=mt, rowStride=11)
    # a data length that is not the frame size
    for n in (4 * 12 - 1, 4 * 12 + 1, 6 * 4 * 3 // 2, 6 * 4 * 3):
        with pytest.raises(ValueError):
            detector.detectFramesRaw([(data[:n], 6, 4, mt)])
        with pytest.raises(ValueError):
            detector.detectBatchRaw(data[:n], count=1, width=6, height=4, matType=mt)
        with pytest.raises(ValueError):
            detector.detectFacesFromMatBytes(data[:n], width=6, height=4, matType=mt)
    with pytest.raises(ValueError):
        detector.detectFramesRaw([(data[:4 * 15], 6, 4, mt, 16)])                  # 4 rows of stride 16 are 64 bytes
