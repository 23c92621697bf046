"""CPU checks of the mixed-batch entry points (fdt_detect_frames, fdt_detect_jpeg_batch) and their Python mirror: the wire
layout of fdt_frame, the null-handle status, and the argument checks that must fail before any call into the library."""
import ctypes as C

import numpy as np
import pytest

from face_detection_tflite_b200 import _ffi


def test_frame_struct_layout():
    assert C.sizeof(_ffi.FdtFrame) == 24                      # static_assert in csrc/fdt_api.cu
    assert [f[0] for f in _ffi.FdtFrame._fields_] == ["data", "width", "height", "row_stride", "mat_type"]
    assert _ffi.FdtFrame.width.offset == 8 and _ffi.FdtFrame.mat_type.offset == 20


def test_null_handle_is_not_ready(lib):
    frames = (_ffi.FdtFrame * 1)()
    faces = (_ffi.FdtFace * 100)()
    counts = (C.c_int32 * 1)()
    assert lib.fdt_detect_frames(None, frames, 1, 0, 0, faces, counts, None, None) == _ffi.FDT_ERR_NOT_READY
    ptrs = (C.c_void_p * 1)()
    sizes = (C.c_size_t * 1)()
    status = (C.c_int32 * 1)()
    assert lib.fdt_detect_jpeg_batch(None, ptrs, sizes, 1, 0, faces, counts, None, None, None, status) == _ffi.FDT_ERR_NOT_READY


class _NoLibrary:
    def __getattr__(self, name):
        raise AssertionError("the argument checks must fail before %s is called" % name)


@pytest.fixture
def detector(lib):
    import face_detection_tflite_b200 as fdt
    d = fdt.FaceDetector()
    d._lib = _NoLibrary()
    return d


@pytest.mark.parametrize("frames", [
    [("not a tuple")],
    [(np.zeros(12, np.uint8), 2, 2)],                                   # too short
    [(np.zeros(12, np.uint8), 0, 2, 16)],                               # zero width
    [(np.zeros(12, np.uint8), 2, 2, 99)],                               # unknown format
    [(np.zeros(12, np.uint8), 2, 2, 16, 5)],                            # row stride below width * channels
    [(np.zeros(11, np.uint8), 2, 2, 16)],                               # short buffer
    [(np.zeros(12, np.uint8), 2, 2, 16), (np.zeros(6, np.uint8), 3, 2, _ffi.FDT_FMT_YUV_NV12)],   # odd YUV width
    [(12345, 2, 2, 16)],                                                # a device pointer as a host frame
])
def test_frames_argument_checks(detector, frames):
    with pytest.raises(ValueError):
        detector.detectFramesRaw(frames)


def test_device_frames_need_pointers(detector):
    with pytest.raises(ValueError):
        detector.detectFramesRaw([(np.zeros(12, np.uint8), 2, 2, 16)], memKind=_ffi.FDT_MEM_DEVICE)
    with pytest.raises(ValueError):
        detector.detectFramesRaw([], memKind=7)


@pytest.mark.parametrize("mats", [[np.zeros((4, 4), np.float32)], [np.zeros((4, 4, 2), np.uint8)], [np.zeros((0, 4, 3), np.uint8)],
                                  ["image"]])
def test_mats_argument_checks(detector, mats):
    with pytest.raises(ValueError):
        detector.detectFacesFromMats(mats)


def test_bytes_batch_argument_checks(detector):
    with pytest.raises(ValueError):
        detector.detectFacesFromBytesBatch([b"\xff\xd8", 17])
    with pytest.raises(ValueError):
        detector.detectBytesBatchRaw(["a path, not bytes"])
