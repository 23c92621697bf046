"""CPU checks of separate-plane YUV 4:2:0 frames (fdt_detect_yuv_planes): the ctypes struct against the C header, the sampled
extents, and the argument checks of the Python mirror that must fail before any call into the library.  (The C checks need a
handle, so their codes are tested on the GPU, tests/test_gpu_yuv_planes.py; without one the call returns FDT_ERR_NOT_READY.)"""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

from face_detection_tflite_b200 import _ffi
from face_detection_tflite_b200.face_detector import _plane_extents

HEADER = Path(__file__).resolve().parents[1] / "include" / "fdt_api.h"


def test_struct_layout():
    S = _ffi.FdtYuvPlanes
    assert C.sizeof(S) == 56
    assert [(n, getattr(S, n).offset) for n in ("plane", "row_stride", "width", "height", "pixel_stride", "reserved")] == \
        [("plane", 0), ("row_stride", 24), ("width", 36), ("height", 40), ("pixel_stride", 44), ("reserved", 48)]
    text = HEADER.read_text()
    m = re.search(r"typedef struct fdt_yuv_planes \{(.*?)\} fdt_yuv_planes;\s*/\* (\d+) bytes", text, re.S)
    assert m and int(m.group(2)) == 56
    fields = re.findall(r"(const uint8_t\*|int32_t) ([\w\[\]0-9, ]+);", m.group(1))
    assert fields == [("const uint8_t*", "plane[3]"), ("int32_t", "row_stride[3]"), ("int32_t", "width, height"),
                      ("int32_t", "pixel_stride"), ("int32_t", "reserved")]


def test_entry_point_declared(lib):
    assert "fdt_detect_yuv_planes" in HEADER.read_text()
    fn = lib.fdt_detect_yuv_planes
    assert fn.argtypes[1] == C.POINTER(_ffi.FdtYuvPlanes)
    buf = np.zeros(64, np.uint8)
    arr = (_ffi.FdtYuvPlanes * 1)()
    arr[0].plane = (C.c_void_p * 3)(buf.ctypes.data, buf.ctypes.data, buf.ctypes.data)
    faces = (_ffi.FdtFace * 100)()
    counts = (C.c_int32 * 1)()
    assert fn(None, arr, None, 1, 0, 0, faces, counts, None, None) == _ffi.FDT_ERR_NOT_READY
    assert b"null handle" in lib.fdt_last_error(None)


@pytest.mark.parametrize("w,h,ps,strides", [(1920, 1080, 2, (2048, 2048, 2048)), (1920, 1080, 1, (1984, 1024, 1056)),
                                            (2, 2, 2, (2, 1, 1)), (640, 480, 2, (656, 639, 639)), (640, 480, 1, (640, 320, 320))])
def test_extents(w, h, ps, strides):
    cc = (w // 2 - 1) * ps + 1
    assert _plane_extents(0, strides, w, h, ps) == ((h - 1) * strides[0] + w, (h // 2 - 1) * strides[1] + cc,
                                                    (h // 2 - 1) * strides[2] + cc)


@pytest.mark.parametrize("strides,w,h,ps", [((64, 64, 64), 63, 48, 2), ((64, 64, 64), 64, 47, 2), ((64, 64, 64), 0, 48, 2),
                                            ((64, 64, 64), 64, 48, 3), ((64, 64, 64), 64, 48, 0), ((-64, 64, 64), 64, 48, 2),
                                            ((64, 0, 64), 64, 48, 2), ((63, 64, 64), 64, 48, 2), ((64, 62, 64), 64, 48, 2),
                                            ((64, 64, 31), 64, 48, 1), ((64, 64), 64, 48, 2), ((64, 64, 64.0), 64, 48, 2),
                                            ((64, 64, 64), 64, 48, True)])
def test_extents_refuse(strides, w, h, ps):
    with pytest.raises(ValueError):
        _plane_extents(0, strides, w, h, ps)


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


def planes(h=48, w=64):
    return np.zeros((h, w), np.uint8), np.zeros((h // 2, w // 2), np.uint8), np.zeros((h // 2, w // 2), np.uint8)


def bad_frames():
    y, u, v = planes()
    uv = np.zeros((24, 64), np.uint8)
    wide = np.zeros((24, 96), np.uint8)
    oy, ou, ov = planes(47, 64)
    return [
        (y, u),                                          # two planes
        (y, u, v.astype(np.int16)),                      # wrong dtype
        (y, u, v.reshape(-1)),                           # 1-D plane
        (y, u[:, :31], v),                               # U narrower than width / 2
        (y, u, v[:23]),                                  # V shorter than height / 2
        (np.zeros((48, 64, 1), np.uint8)[..., 0][:, ::-1], u, v),   # negative Y pixel step
        (np.zeros((48, 128), np.uint8)[:, ::2], u, v),   # Y pixel step 2
        (y, uv[:, 0::2], v),                             # U pixel stride 2, V 1
        (y, wide[:, 0::3], wide[:, 1::3]),               # pixel stride 3
        (y[::-1], u, v),                                 # bottom-up Y
        (y, u[::-1], v[::-1]),                           # bottom-up chroma
        (oy, ou, ov),                                    # odd height
        (np.zeros((48, 63), np.uint8), np.zeros((24, 31), np.uint8), np.zeros((24, 31), np.uint8)),   # odd width
        "not a frame",
    ]


@pytest.mark.parametrize("k", range(len(bad_frames())))
def test_python_argument_checks(detector, k):
    good = planes()
    with pytest.raises(ValueError):
        detector.detectFacesFromYuvPlanes([good, bad_frames()[k]])


def test_views_are_accepted(detector):
    """NV12 chroma views, pitched Y views, and orientations, up to the library call."""
    y = np.zeros((48, 96), np.uint8)[:, :64]
    uv = np.zeros((24, 64), np.uint8)
    with pytest.raises(AssertionError, match="fdt_detect_yuv_planes"):
        detector.detectFacesFromYuvPlanes([(y, uv[:, 0::2], uv[:, 1::2])], orientations=[6])


@pytest.mark.parametrize("orientations", [[1], [1, 2, 3], [0, 1], [1, 9], "12", [1.0, 2]])
def test_orientation_list(detector, orientations):
    with pytest.raises(ValueError):
        detector.detectFacesFromYuvPlanes([planes(), planes()], orientations=orientations)


def test_raw_argument_checks(detector):
    y, u, v = (np.zeros(n, np.uint8) for n in (48 * 64, 24 * 32, 24 * 32))
    ok = ((y, u, v), (64, 32, 32), 64, 48, 1)
    bad = [
        ((y, u), (64, 32, 32), 64, 48, 1),                       # two planes
        ((y, u, v), (64, 32), 64, 48, 1),                        # two strides
        ((y, u, v), (64, 32, 32), 64, 48),                       # no pixel stride
        ((y, u, v[:-1]), (64, 32, 32), 64, 48, 1),               # V shorter than its extent
        ((y, u, v), (64, 32, 32), 64, 48, 2),                    # ps 2 extents do not fit 24 x 32 buffers
        ((y, u, v), (64, 31, 32), 64, 48, 1),                    # short chroma stride
        ((y, u, v), (64, 32, 32), 65, 48, 1),                    # odd width
        ((1, 2, 3), (64, 32, 32), 64, 48, 1),                    # pointers for host memory
        ((y, u, v.astype(np.int16)), (64, 32, 32), 64, 48, 1),  # wrong dtype
        ((y, u, v.reshape(24, 32)[:, ::2]), (64, 32, 32), 64, 48, 1),   # not contiguous
    ]
    for fr in bad:
        with pytest.raises(ValueError):
            detector.detectYuvPlanesRaw([ok, fr])
    with pytest.raises(ValueError):
        detector.detectYuvPlanesRaw([((y, 2, 3), (64, 32, 32), 64, 48, 1)], memKind=_ffi.FDT_MEM_DEVICE)
    with pytest.raises(ValueError):
        detector.detectYuvPlanesRaw([ok], memKind=5)
    with pytest.raises(ValueError):
        detector.detectYuvPlanesRaw([ok], orientations=[1, 1])
    # a buffer that ends at its last sample is enough
    ends = ((y[:47 * 64 + 64], u[:23 * 32 + 32], v[:23 * 32 + 32]), (64, 32, 32), 64, 48, 1)
    with pytest.raises(AssertionError, match="fdt_detect_yuv_planes"):
        detector.detectYuvPlanesRaw([ok, ends])
