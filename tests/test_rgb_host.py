"""CPU checks of the RGB, RGBA and planar RGB formats' Python mirror: the constants against the C header, the frame-size math,
and the argument checks that must fail before any call into the library."""
import re
from pathlib import Path

import numpy as np
import pytest

from face_detection_tflite_b200 import _ffi
from face_detection_tflite_b200.face_detector import _frame_geometry

HEADER = Path(__file__).resolve().parents[1] / "include" / "fdt_api.h"


def test_constants_match_header():
    text = HEADER.read_text()
    for name in ("FDT_FMT_RGB", "FDT_FMT_RGBA", "FDT_FMT_RGB_PLANAR", "FDT_FMT_YUV_NV12"):
        m = re.search(r"\b%s = (0x[0-9A-Fa-f]+|\d+)" % name, text)
        assert m, name
        assert getattr(_ffi, name) == int(m.group(1), 0), name
    assert _ffi.RGB_FORMATS == (_ffi.FDT_FMT_RGB, _ffi.FDT_FMT_RGBA, _ffi.FDT_FMT_RGB_PLANAR)
    assert not set(_ffi.RGB_FORMATS) & set(_ffi.YUV_FORMATS) and min(_ffi.RGB_FORMATS) > 4095   # no cv MatType collides


@pytest.mark.parametrize("w,h", [(1280, 720), (641, 359), (1, 1)])
def test_frame_geometry(w, h):
    assert _frame_geometry(0, w, h, _ffi.FDT_FMT_RGB, None) == (3 * w, 3 * w * h)
    assert _frame_geometry(0, w, h, _ffi.FDT_FMT_RGBA, None) == (4 * w, 4 * w * h)
    assert _frame_geometry(0, w, h, _ffi.FDT_FMT_RGB_PLANAR, None) == (w, 3 * w * h)
    assert _frame_geometry(0, w, h, _ffi.FDT_FMT_RGB, 3 * w + 5) == (3 * w + 5, (3 * w + 5) * h)
    assert _frame_geometry(0, w, h, _ffi.FDT_FMT_RGBA, 4 * w + 64) == (4 * w + 64, (4 * w + 64) * h)
    assert _frame_geometry(0, w, h, _ffi.FDT_FMT_RGB_PLANAR, w + 7) == (w + 7, 3 * (w + 7) * h)
    # the existing formats are unchanged
    assert _frame_geometry(0, w, h, _ffi.FDT_MAT_8UC3, None) == (3 * w, 3 * w * h)
    assert _frame_geometry(0, w, h, _ffi.FDT_MAT_8UC1, None) == (w, w * h)


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


@pytest.mark.parametrize("layout,shape", [("rgb", (4, 6, 2)), ("rgb", (4, 6, 5)), ("rgb", (4,)), ("rgb_planar", (4, 6, 3)),
                                          ("rgb_planar", (4, 6)), ("rgb_planar", (3, 0, 6)), ("rgb_planar", (1, 4, 6)),
                                          ("bgr", (4, 6, 2))])
def test_wrong_shape_for_layout(detector, layout, shape):
    m = np.zeros(shape, np.uint8)
    with pytest.raises(ValueError):
        detector.detectFacesFromMat(m, layout=layout)
    with pytest.raises(ValueError):
        detector.detectFacesFromMats([np.zeros((4, 6, 3), np.uint8) if layout != "rgb_planar" else np.zeros((3, 4, 6), np.uint8), m],
                                     layout=layout)


@pytest.mark.parametrize("layout", ["RGB", "chw", "", None, 1, "planar"])
def test_unknown_layout(detector, layout):
    with pytest.raises(ValueError):
        detector.detectFacesFromMat(np.zeros((4, 6, 3), np.uint8), layout=layout)
    with pytest.raises(ValueError):
        detector.detectFacesFromMats([np.zeros((4, 6, 3), np.uint8)], layout=layout)
    with pytest.raises(ValueError):
        detector.detectFacesFromMats([], layout=layout)


def test_wrong_dtype(detector):
    with pytest.raises(ValueError):
        detector.detectFacesFromMat(np.zeros((3, 4, 6), np.float32), layout="rgb_planar")
    with pytest.raises(ValueError):
        detector.detectFacesFromMat(np.zeros((4, 6, 3), np.uint16), layout="rgb")


@pytest.mark.parametrize("mt,minimum", [(_ffi.FDT_FMT_RGB, 18), (_ffi.FDT_FMT_RGBA, 24), (_ffi.FDT_FMT_RGB_PLANAR, 6)])
def test_short_row_stride(detector, mt, minimum):
    data = np.zeros(3 * 4 * 32, np.uint8)
    with pytest.raises(ValueError):
        detector.detectFramesRaw([(data[:4 * (minimum - 1) * (3 if mt == _ffi.FDT_FMT_RGB_PLANAR else 1)], 6, 4, mt, minimum - 1)])
    with pytest.raises(ValueError):
        detector.detectBatchRaw(data, count=1, width=6, height=4, matType=mt, rowStride=minimum - 1)
    # a data length that does not match the format's frame size
    n = 4 * minimum * (3 if mt == _ffi.FDT_FMT_RGB_PLANAR else 1)
    with pytest.raises(ValueError):
        detector.detectFramesRaw([(data[:n - 1], 6, 4, mt)])
    with pytest.raises(ValueError):
        detector.detectBatchRaw(data[:n + 1], count=1, width=6, height=4, matType=mt)
