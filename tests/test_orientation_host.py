"""CPU checks of the oriented entry points (fdt_detect_batch_oriented, fdt_detect_frames_oriented) and their Python mirror:
the null-handle status, the argument checks that must fail before any call into the library, and the orientation convention
(oracle.jpeg_ops.exif_transform) against OpenCV's rotate / flip / transpose."""
import ctypes as C

import cv2
import numpy as np
import pytest

from face_detection_tflite_b200 import _ffi
from oracle.jpeg_ops import exif_transform


def test_null_handle_is_not_ready(lib):
    frames = (_ffi.FdtFrame * 1)()
    faces = (_ffi.FdtFace * 100)()
    counts = (C.c_int32 * 1)()
    orients = (C.c_int32 * 1)(6)
    buf = (C.c_uint8 * 12)()
    assert lib.fdt_detect_batch_oriented(None, buf, 1, 2, 2, 6, 16, 6, 0, 0, faces, counts, None, None) == _ffi.FDT_ERR_NOT_READY
    assert lib.fdt_detect_frames_oriented(None, frames, orients, 1, 0, 0, faces, counts, None, None) == _ffi.FDT_ERR_NOT_READY
    assert lib.fdt_detect_frames_oriented(None, frames, None, 1, 0, 0, faces, counts, None, None) == _ffi.FDT_ERR_NOT_READY


def test_constants():
    assert (_ffi.FDT_ORIENT_UPRIGHT, _ffi.FDT_ORIENT_ROT180, _ffi.FDT_ORIENT_ROT90_CW, _ffi.FDT_ORIENT_ROT90_CCW) == (1, 3, 6, 8)


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


BAD = [0, 9, -1, 2.0, "6", None, True]


@pytest.mark.parametrize("o", BAD)
def test_uniform_calls_reject_bad_orientation(detector, o):
    frame = np.zeros((2, 2, 3), np.uint8)
    with pytest.raises(ValueError):
        detector.detectBatchRaw(frame, count=1, width=2, height=2, orientation=o)
    with pytest.raises(ValueError):
        detector.detectFacesBatch(frame, count=1, width=2, height=2, orientation=o)
    with pytest.raises(ValueError):
        detector.detectFacesFromMatBytes(frame.tobytes(), width=2, height=2, orientation=o)
    with pytest.raises(ValueError):
        detector.detectFacesFromMat(frame, orientation=o)


@pytest.mark.parametrize("orients", [[0], [1, 9], [6], [1, 2, 3], "12", 6, [6.0, 1], [np.int32(1), None]])
def test_frame_lists_reject_bad_orientations(detector, orients):
    frames = [(np.zeros(12, np.uint8), 2, 2, 16), (np.zeros(12, np.uint8), 2, 2, 16)]
    with pytest.raises(ValueError):
        detector.detectFramesRaw(frames, orientations=orients)
    with pytest.raises(ValueError):
        detector.detectFacesFromMats([np.zeros((2, 2, 3), np.uint8)] * 2, orientations=orients)


def _cv2_composition(img, o):
    """The EXIF meaning spelled with OpenCV's own operations."""
    return {1: lambda m: m,
            2: lambda m: cv2.flip(m, 1),
            3: lambda m: cv2.rotate(m, cv2.ROTATE_180),
            4: lambda m: cv2.flip(m, 0),
            5: lambda m: cv2.transpose(m),
            6: lambda m: cv2.rotate(m, cv2.ROTATE_90_CLOCKWISE),
            7: lambda m: cv2.rotate(cv2.transpose(m), cv2.ROTATE_180),
            8: lambda m: cv2.rotate(m, cv2.ROTATE_90_COUNTERCLOCKWISE)}[o](img)


@pytest.mark.parametrize("o", range(1, 9))
@pytest.mark.parametrize("shape", [(5, 7), (6, 4, 3), (3, 8, 4), (1, 9, 1)])
def test_exif_transform_matches_cv2(o, shape):
    img = np.random.default_rng(o).integers(0, 256, shape, dtype=np.uint8)
    want = _cv2_composition(img, o)
    if img.ndim == 3 and img.shape[2] == 1:
        want = want.reshape(want.shape[0], want.shape[1], 1)
    if img.ndim == 2:
        got = exif_transform(img[..., None], o)[..., 0]
    else:
        got = exif_transform(img, o)
    assert got.shape == want.shape and np.array_equal(got, want)
    if o >= 5:
        assert got.shape[:2] == img.shape[1::-1]
