"""CPU checks of the 16-bit YUV 4:2:0 inputs (FDT_FMT_P010 and fdt_detect_yuv_planes16): the constant and the header's text,
the frame-size and plane-extent math, the argument checks that must fail before any call into the library, and the sm_100a
build's new kernel instantiations."""
import os
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

from face_detection_tflite_b200 import _ffi
from face_detection_tflite_b200.face_detector import _frame_geometry, _plane_extents, _row_step

ROOT = Path(__file__).resolve().parents[1]
HEADER = ROOT / "include" / "fdt_api.h"
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
P010 = _ffi.FDT_FMT_P010


def reduce8(s, bits):
    """The header's sample rule."""
    return ((s.astype(np.uint32) >> (bits - 8)) & 0xFF).astype(np.uint8)


def test_constant_and_header_text():
    text = HEADER.read_text()
    m = re.search(r"\bFDT_FMT_P010 = (0x[0-9A-Fa-f]+|\d+)", text)
    assert m and int(m.group(1), 0) == P010 == 0x1003
    others = {int(v, 0) for k, v in re.findall(r"\b(FDT_FMT_\w+) = (0x[0-9A-Fa-f]+|\d+)", text) if k != "FDT_FMT_P010"}
    assert P010 not in others and P010 > 4095
    assert re.search(r"fdt_detect_yuv_planes16\(fdt_handle\* h, const fdt_yuv_planes\* frames, const int32_t\* orientations, "
                     r"int32_t n,\s+int32_t sample_bits, int32_t mode, int32_t mem_kind,", text)
    # the rule, and that the colour is not an HDR-correct conversion
    assert "(s >> (bits - 8)) & 0xFF" in text and "(s >> (sample_bits - 8)) & 0xFF" in text
    assert "BT.2020" in text and "PQ / HLG" in text and "552,960" in text
    assert _ffi.SAMPLE_BITS == (10, 12, 16)
    assert '"fdt_detect_yuv_planes16"' in Path(_ffi.__file__).read_text()


@pytest.mark.parametrize("bits", [10, 12, 16])
def test_sample_rule_truncates_and_ignores_other_bits(bits):
    rng = np.random.default_rng(bits)
    v8 = rng.integers(0, 256, 4096, dtype=np.uint16)
    low = rng.integers(0, 1 << (bits - 8), 4096, dtype=np.uint16)
    high = (rng.integers(0, 1 << (16 - bits), 4096, dtype=np.uint16) << bits) if bits < 16 else 0
    s = (v8 << (bits - 8)) | low | high
    assert np.array_equal(reduce8(s, bits), v8.astype(np.uint8))
    # P010 (bits 16) is the high byte: what a caller's (t >> 8).to(uint8) computes
    assert np.array_equal(reduce8(s, 16), (s >> 8).astype(np.uint8))


@pytest.mark.parametrize("w,h", [(1280, 720), (1920, 1080), (6, 4), (2, 2)])
def test_frame_geometry(w, h):
    assert _row_step(P010) == 2
    assert _frame_geometry(0, w, h, P010, None) == (2 * w, 3 * w * h)
    assert _frame_geometry(0, w, h, P010, 2 * w + 64) == (2 * w + 64, (2 * w + 64) * h * 3 // 2)
    for bad in ((w, h, 2 * w - 2), (w, h, 2 * w + 1), (w + 1, h, 2 * w + 2), (w, h + 1, 2 * w)):
        with pytest.raises(ValueError):
            _frame_geometry(0, *bad[:2], P010, bad[2])
    assert _frame_geometry(0, w, h, _ffi.FDT_FMT_YUV_NV12, None) == (w, w * h * 3 // 2)


def test_plane_extents_16():
    # 8-bit extents are unchanged
    assert _plane_extents(0, (1280, 1280, 1280), 1280, 720, 2) == (719 * 1280 + 1280, 359 * 1280 + 1279, 359 * 1280 + 1279)
    # 16-bit: samples x 2 bytes (NVDEC P016 surface: pitch 2560 + padding, chroma interleaved)
    assert _plane_extents(0, (2688, 2688, 2688), 1280, 720, 2, 2) == (719 * 2688 + 2560, 359 * 2688 + 2558, 359 * 2688 + 2558)
    assert _plane_extents(0, (2560, 1280, 1280), 1280, 720, 1, 2) == (719 * 2560 + 2560, 359 * 1280 + 1280, 359 * 1280 + 1280)
    for strides in ((2558, 1280, 1280), (2560, 1278, 1280), (2560, 1280, 1278), (2561, 1281, 1281), (2560, 1281, 1280)):
        with pytest.raises(ValueError):
            _plane_extents(0, strides, 1280, 720, 1, 2)


class _NoLibrary:
    def __getattr__(self, name):
        raise AssertionError("the argument checks must fail before %s is called" % name)


class _Recorder:
    """Records the library function a call reaches, then stops it."""

    def __init__(self):
        self.called = []

    def __getattr__(self, name):
        def f(*a):
            self.called.append(name)
            raise _Stop()
        return f


class _Stop(Exception):
    pass


@pytest.fixture
def detector(lib):
    import face_detection_tflite_b200 as fdt
    d = fdt.FaceDetector()
    d._lib = _NoLibrary()
    d._ready = True             # past the state check: only the argument checks stand between the call and the library
    return d


@pytest.mark.parametrize("shape,dt", [((6, 4), np.uint8), ((6, 4), np.float32), ((6, 4, 1), np.uint16), ((4, 4), np.uint16),
                                      ((5, 4), np.uint16), ((6, 5), np.uint16), ((0, 4), np.uint16), ((6, 0), np.uint16)])
def test_mat_checks(detector, shape, dt):
    m = np.zeros(shape, dt)
    with pytest.raises(ValueError):
        detector.detectFacesFromMat(m, layout="p010")
    with pytest.raises(ValueError):
        detector.detectFacesFromMats([np.zeros((6, 4), np.uint16), m], layout="p010")


@pytest.mark.parametrize("h", [2, 4, 270, 720, 1050, 1080])
def test_mat_accepts_every_even_height(lib, h):
    """(3H/2) x W uint16 arrays of every even H reach the library, H = 2 (mod 4) included (1680x1050 screen captures)."""
    import face_detection_tflite_b200 as fdt
    from face_detection_tflite_b200.face_detector import _mat_type
    m = np.zeros((h * 3 // 2, 64), np.uint16)
    assert _mat_type(m, 0, "p010") == P010
    d = fdt.FaceDetector()
    d._lib = rec = _Recorder()
    d._ready = True
    d._h = None
    with pytest.raises(_Stop):
        d.detectFacesFromMat(m, layout="p010")
    with pytest.raises(_Stop):
        d.detectFacesFromMats([m, m[:, :32]], layout="p010")
    assert rec.called == ["fdt_detect_one", "fdt_detect_frames"]


def test_raw_call_checks(detector):
    data = np.zeros(64 * 48 * 3, np.uint8)
    for w, h in ((63, 48), (64, 47)):                     # odd width or height
        with pytest.raises(ValueError):
            detector.detectFramesRaw([(data, w, h, P010)])
        with pytest.raises(ValueError):
            detector.detectBatchRaw(data, count=1, width=w, height=h, matType=P010)
        with pytest.raises(ValueError):
            detector.detectFacesFromMatBytes(data, width=w, height=h, matType=P010)
        with pytest.raises(ValueError):
            detector.detectFacesFromMatBytes(data, width=w, height=h, matType=P010, orientation=6)
    for stride in (126, 129):                             # below 2 * width, odd
        with pytest.raises(ValueError):
            detector.detectFramesRaw([(np.zeros(48 * stride * 3 // 2, np.uint8), 64, 48, P010, stride)])
        with pytest.raises(ValueError):
            detector.detectBatchRaw(np.zeros(48 * stride * 3 // 2, np.uint8), count=1, width=64, height=48, matType=P010,
                                    rowStride=stride)
    for n in (64 * 48 * 3 - 2, 64 * 48 * 3 + 2, 64 * 48 * 3 // 2, 64 * 48 * 2):
        with pytest.raises(ValueError):
            detector.detectFramesRaw([(np.zeros(n, np.uint8), 64, 48, P010)])
        with pytest.raises(ValueError):
            detector.detectBatchRaw(np.zeros(n, np.uint8), count=1, width=64, height=48, matType=P010)
        with pytest.raises(ValueError):
            detector.detectFacesFromMatBytes(np.zeros(n, np.uint8), width=64, height=48, matType=P010)
    with pytest.raises(ValueError):                       # a uint16 frame of the wrong length
        detector.detectBatchRaw(np.zeros(64 * 48 * 3 // 2 - 1, np.uint16), count=1, width=64, height=48, matType=P010)


def planes16(w=64, h=48, dt=np.uint16):
    return np.zeros((h, w), dt), np.zeros((h // 2, w // 2), dt), np.zeros((h // 2, w // 2), dt)


def test_planes_checks(detector):
    for bits in (None, 8, 9, 11, 15, 17, 0, 16.0, True, "10"):
        with pytest.raises(ValueError):
            detector.detectFacesFromYuvPlanes([planes16()], sampleBits=bits)
    with pytest.raises(ValueError):                                   # uint8 planes with sampleBits
        detector.detectFacesFromYuvPlanes([planes16(dt=np.uint8)], sampleBits=10)
    with pytest.raises(ValueError):                                   # mixed dtypes
        detector.detectFacesFromYuvPlanes([(np.zeros((48, 64), np.uint16), np.zeros((24, 32), np.uint8),
                                            np.zeros((24, 32), np.uint16))], sampleBits=10)
    with pytest.raises(ValueError):                                   # odd width
        detector.detectFacesFromYuvPlanes([(np.zeros((48, 63), np.uint16), np.zeros((24, 31), np.uint16),
                                            np.zeros((24, 31), np.uint16))], sampleBits=10)
    with pytest.raises(ValueError):                                   # chroma shape
        detector.detectFacesFromYuvPlanes([(np.zeros((48, 64), np.uint16), np.zeros((24, 30), np.uint16),
                                            np.zeros((24, 32), np.uint16))], sampleBits=12)
    y = np.zeros((48, 128), np.uint16)
    with pytest.raises(ValueError):                                   # Y samples not adjacent
        detector.detectFacesFromYuvPlanes([(y[:, ::2], *planes16()[1:])], sampleBits=16)
    # raw: strides in bytes, pixel stride in samples
    buf = np.zeros(64 * 48 * 3, np.uint8)
    ok = ((buf, buf, buf), (128, 64, 64), 64, 48, 1)
    for bad in (((buf, buf, buf), (127, 64, 64), 64, 48, 1), ((buf, buf, buf), (128, 63, 64), 64, 48, 1),
                ((buf, buf, buf), (126, 64, 64), 64, 48, 1), ((buf, buf, buf), (128, 62, 64), 64, 48, 1),
                ((buf, buf, buf), (128, 64, 64), 64, 48, 3), ((buf[:100], buf, buf), (128, 64, 64), 64, 48, 1),
                ((buf[1:], buf, buf), (128, 64, 64), 64, 48, 1)):
        with pytest.raises(ValueError):
            detector.detectYuvPlanesRaw([ok, bad], sampleBits=10)
    with pytest.raises(ValueError):                                   # odd device pointer
        detector.detectYuvPlanesRaw([((1 << 20, (1 << 20) + 1, 1 << 21), (128, 64, 64), 64, 48, 1)], memKind=1, sampleBits=10)
    for bits in (8, 14, 10.0):
        with pytest.raises(ValueError):
            detector.detectYuvPlanesRaw([ok], sampleBits=bits)


def test_eight_bit_calls_reach_the_functions_they_always_did(lib):
    import face_detection_tflite_b200 as fdt
    d = fdt.FaceDetector()
    d._lib = rec = _Recorder()
    d._ready = True
    d._h = None
    y, u, v = planes16(dt=np.uint8)
    for call, name in ((lambda: d.detectFacesFromYuvPlanes([(y, u, v)]), "fdt_detect_yuv_planes"),
                       (lambda: d.detectYuvPlanesRaw([((y, u, v), (64, 32, 32), 64, 48, 1)]), "fdt_detect_yuv_planes"),
                       (lambda: d.detectFacesFromYuvPlanes([planes16()], sampleBits=10), "fdt_detect_yuv_planes16"),
                       (lambda: d.detectBatchRaw(np.zeros(64 * 48 * 3, np.uint16), count=2, width=64, height=48, matType=P010),
                        "fdt_detect_batch"),
                       (lambda: d.detectFacesFromMat(np.zeros((72, 64), np.uint16), layout="p010"), "fdt_detect_one")):
        rec.called.clear()
        with pytest.raises(_Stop):
            call()
        assert rec.called == [name]


def _sass_names(obj):
    out = subprocess.run([os.path.join(CUDA, "bin", "cuobjdump"), "-sass", str(obj)], capture_output=True, text=True, check=True).stdout
    names = re.findall(r"Function : (\S+)", out)
    demangled = subprocess.run([os.path.join(CUDA, "bin", "cu++filt")], input="\n".join(names), capture_output=True, text=True,
                               check=True).stdout.split("\n")
    return out, [n for n in demangled if n]


def test_new_instantiations_build_for_sm100a(lib):
    build = ROOT / "face_detection_tflite_b200" / "build"
    out, names = _sass_names(build / "kernels_pre.cu.o")
    assert "arch = sm_100a" in out
    assert sum("k_letterbox_yuv<(bool)1>" in n for n in names) == 1
    assert sum("k_letterbox_tr<(bool)1, (bool)1>" in n for n in names) == 1
    assert sum(re.search(r"k_letterbox_multi<(\(bool\)[01], ){4}\(bool\)1>", n) is not None for n in names) == 4
    out, names = _sass_names(build / "kernels_warp16.cu.o")
    assert "arch = sm_100a" in out
    warps = [n for n in names if "yuv16::k_warp_affine<" in n]
    assert len(warps) == 16 and len(names) == 16
    # kernels_post.cu keeps exactly its twenty crop warps
    _, names = _sass_names(build / "kernels_post.cu.o")
    assert len([n for n in names if "k_warp_affine<" in n]) == 20
