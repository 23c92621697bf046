"""CPU checks of the face crops of the detect calls (fdt_set_face_crops): the ctypes struct against the C header, the Python spec
checks that must fail before any call into the library, the numpy reference of the layouts and of the float32 conversion, and the
sm_100a build of the crop warps.  (The C checks need a handle; their codes are tested on the GPU, tests/test_gpu_face_crops.py.)"""
import ctypes as C
import os
import re
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from face_detection_tflite_b200 import _ffi
from face_detection_tflite_b200.face_detector import FaceCropSpec

ROOT = Path(__file__).resolve().parents[1]
HEADER = ROOT / "include" / "fdt_api.h"
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")


def test_struct_layout():
    S = _ffi.FdtCropSpec
    assert C.sizeof(S) == 40
    assert [(n, getattr(S, n).offset) for n in ("struct_size", "kind", "out_size", "layout", "scale", "bias")] == \
        [("struct_size", 0), ("kind", 4), ("out_size", 8), ("layout", 12), ("scale", 16), ("bias", 28)]
    text = HEADER.read_text()
    m = re.search(r"typedef struct fdt_crop_spec \{(.*?)\} fdt_crop_spec;\s*/\* (\d+) bytes", text, re.S)
    assert m and int(m.group(2)) == 40
    assert re.findall(r"(int32_t|float) ([\w\[\]0-9, ]+);", m.group(1)) == [
        ("int32_t", "struct_size"), ("int32_t", "kind"), ("int32_t", "out_size"), ("int32_t", "layout"), ("float", "scale[3], bias[3]")]
    consts = dict(re.findall(r"(FDT_CROP_\w+) = (\d+)", text))
    assert {k: int(v) for k, v in consts.items()} == {"FDT_CROP_EMBEDDING": _ffi.FDT_CROP_EMBEDDING, "FDT_CROP_FACE": _ffi.FDT_CROP_FACE,
                                                      "FDT_CROP_RGB": _ffi.FDT_CROP_RGB, "FDT_CROP_CHW": _ffi.FDT_CROP_CHW,
                                                      "FDT_CROP_F32": _ffi.FDT_CROP_F32}


def test_entry_points_declared(lib):
    spec = FaceCropSpec()._struct()
    n = C.c_int64(5)
    assert lib.fdt_set_face_crops(None, C.byref(spec)) == _ffi.FDT_ERR_NOT_READY
    assert lib.fdt_get_face_crops(None, C.byref(n), None) == _ffi.FDT_ERR_NOT_READY
    assert lib.fdt_copy_face_crops(None, None, 0, 0, None) == _ffi.FDT_ERR_NOT_READY


@pytest.mark.parametrize("order,chw,dtype,layout,shape", [("bgr", False, np.uint8, 0, (2, 112, 112, 3)),
                                                          ("rgb", False, np.uint8, 1, (2, 112, 112, 3)),
                                                          ("bgr", True, np.uint8, 2, (2, 3, 112, 112)),
                                                          ("rgb", True, np.float32, 7, (2, 3, 112, 112)),
                                                          ("bgr", False, "float32", 4, (2, 112, 112, 3))])
def test_spec_fields(order, chw, dtype, layout, shape):
    s = FaceCropSpec("face", 112, order, chw, dtype, scale=0.5, bias=(1, 2, 3))
    c = s._struct()
    assert (c.struct_size, c.kind, c.out_size, c.layout) == (40, _ffi.FDT_CROP_FACE, 112, layout)
    assert list(c.scale) == [0.5] * 3 and list(c.bias) == [1.0, 2.0, 3.0]
    assert s.shape(2) == shape and s.cropBytes == 3 * 112 * 112 * np.dtype(dtype).itemsize


@pytest.mark.parametrize("kw", [dict(kind="mesh"), dict(kind=0), dict(size=0), dict(size=4097), dict(size=112.0), dict(size=True),
                                dict(order="RGB"), dict(order=None), dict(chw=1), dict(dtype=np.float64), dict(dtype=np.int8),
                                dict(dtype="nonsense"), dict(scale=(1, 2)), dict(scale=float("nan")), dict(bias=(0, float("inf"), 0)),
                                dict(scale=1e39), dict(bias="x")])
def test_spec_refuses(kw):
    with pytest.raises(ValueError):
        FaceCropSpec(**kw)


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


def test_python_argument_checks(detector):
    for bad in ("embedding", 112, {"kind": "face"}):
        with pytest.raises(ValueError):
            detector.setFaceCrops(bad)
    for args in ((1.5, 10), (0, -1), (True, 10), (0, 10, 5)):
        with pytest.raises(ValueError):
            detector.copyFaceCropsRaw(*args)
    with pytest.raises(AssertionError, match="fdt_set_face_crops"):
        detector.setFaceCrops(FaceCropSpec())


def test_numpy_f32_conversion_is_mul_then_add():
    """numpy's float32 v * s + b rounds the product and then the sum (no fused multiply-add), the kernel's __fmul_rn then
    __fadd_rn.  Emulated in float64: a u8 times a float32 is exact there, and so is the sum of two float32 of these magnitudes
    before its one rounding."""
    v = np.arange(256, dtype=np.uint8)
    rng = np.random.default_rng(0)
    for s, b in [(1 / 127.5, -1.0), (1 / 255, 0.0), (1 / 58.395, -123.675 / 58.395)] + \
                [tuple(rng.uniform(-3, 3, 2)) for _ in range(20)]:
        s32, b32 = np.float32(s), np.float32(b)
        got = v.astype(np.float32) * s32 + b32
        prod = (v.astype(np.float64) * np.float64(s32)).astype(np.float32)
        want = (prod.astype(np.float64) + np.float64(b32)).astype(np.float32)
        assert got.dtype == np.float32 and np.array_equal(got, want)


def test_layout_reference():
    """The test reference's reorder of an HWC BGR crop: RGB reverses the last axis, CHW moves it first."""
    from test_gpu_face_crops import to_layout
    crop = np.random.default_rng(1).integers(0, 256, (5, 5, 3), dtype=np.uint8)
    for layout in range(8):
        s = FaceCropSpec("embedding", 5, "rgb" if layout & 1 else "bgr", bool(layout & 2), np.float32 if layout & 4 else np.uint8,
                         (0.5, 2.0, -1.0), (1.0, 0.0, 0.25))
        out = to_layout(crop, s)
        assert out.shape == s.shape(1)[1:] and out.dtype == s.dtype
        for y, x, c in [(0, 0, 0), (1, 3, 2), (4, 2, 1)]:
            src = crop[y, x, 2 - c if layout & 1 else c]
            val = np.float32(src) * np.float32(s.scale[c]) + np.float32(s.bias[c]) if layout & 4 else src
            assert (out[c, y, x] if layout & 2 else out[y, x, c]) == val


def _sass_kernels(obj):
    out = subprocess.run([os.path.join(CUDA, "bin", "cuobjdump"), "-sass", str(obj)], capture_output=True, text=True, check=True).stdout
    names = re.findall(r"Function : (\S+)", out)
    demangled = subprocess.run([os.path.join(CUDA, "bin", "cu++filt")], input="\n".join(names), capture_output=True, text=True,
                               check=True).stdout.split("\n")
    return out, [n for n in demangled if n]


def test_crop_warps_build_for_sm100a(lib):
    """libfdt_cuda's crop warps are sm_100a SASS: the ten gathers the pipeline launches, each with and without the face-crop
    epilogue, and nothing else."""
    obj = ROOT / "face_detection_tflite_b200" / "build" / "kernels_post.cu.o"
    out, names = _sass_kernels(obj)
    assert "arch = sm_100a" in out
    warps = [n for n in names if "k_warp_affine<" in n]
    assert len(warps) == 20
    assert sum(", (bool)1>(fdt::WarpP, const fdt::YuvPlaneD *, fdt::CropOutP)" in n for n in warps) == 10


def test_sass_compare_runs_without_gpu(lib):
    """tools/sass_compare.py on the sm_100a build: a kernel equals itself, and the face-crop epilogue is a different kernel."""
    obj = str(ROOT / "face_detection_tflite_b200" / "build" / "kernels_post.cu.o")
    tool = str(ROOT / "tools" / "sass_compare.py")
    same = "k_warp_affine<(bool)0, (bool)0, (bool)0, (bool)0, (bool)0>=k_warp_affine<(bool)0, (bool)0, (bool)0, (bool)0, (bool)0>"
    r = subprocess.run([sys.executable, tool, obj, obj, same], capture_output=True, text=True)
    assert r.returncode == 0 and " 0 differ" in r.stdout, r.stdout + r.stderr
    other = "k_warp_affine<(bool)0, (bool)0, (bool)0, (bool)0, (bool)0>=k_warp_affine<(bool)0, (bool)0, (bool)0, (bool)0, (bool)1>"
    r = subprocess.run([sys.executable, tool, obj, obj, other], capture_output=True, text=True)
    assert r.returncode == 1, r.stdout + r.stderr
