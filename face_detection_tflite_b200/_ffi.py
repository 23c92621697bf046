"""ctypes binding of libfdt_cuda.so (include/fdt_api.h).  The same entry points are what a
dart:ffi binding binds (INTEGRATION.md); nothing here computes — it only marshals."""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libfdt_cuda.so"

FDT_OK, FDT_ERR_NOT_READY, FDT_ERR_BAD_ARG, FDT_ERR_SIZE_MISMATCH, FDT_ERR_MODEL, FDT_ERR_CUDA, FDT_ERR_UNSUPPORTED, FDT_ERR_FORMAT = range(8)
FDT_MAT_8UC1, FDT_MAT_8UC3, FDT_MAT_8UC4 = 0, 16, 24
FDT_FMT_YUV_NV12, FDT_FMT_YUV_NV21, FDT_FMT_YUV_I420 = 0x1000, 0x1001, 0x1002   # YUV 4:2:0, height * rowStride * 3 / 2 bytes
YUV_FORMATS = (FDT_FMT_YUV_NV12, FDT_FMT_YUV_NV21, FDT_FMT_YUV_I420)
# RGB-ordered frames: packed RGB / RGBA (height * rowStride bytes) and planar RGB, an R, a G and a B plane of height rows of
# rowStride bytes each, back to back (3 * height * rowStride bytes; a contiguous [3, H, W] tensor has rowStride = W)
FDT_FMT_RGB, FDT_FMT_RGBA, FDT_FMT_RGB_PLANAR = 0x1010, 0x1011, 0x1012
RGB_FORMATS = (FDT_FMT_RGB, FDT_FMT_RGBA, FDT_FMT_RGB_PLANAR)
# packed YUV 4:2:2 (V4L2 webcams: YUYV; capture cards: UYVY; GStreamer YUY2 / UYVY / YVYU): 2 bytes per pixel, even width,
# height * rowStride bytes with rowStride >= 2 * width (cv2's HxW CV_8UC2 Mat, an HxWx2 array)
FDT_FMT_YUYV, FDT_FMT_UYVY, FDT_FMT_YVYU = 0x1020, 0x1021, 0x1022
YUV422_FORMATS = (FDT_FMT_YUYV, FDT_FMT_UYVY, FDT_FMT_YVYU)
# 16-bit YUV 4:2:0 with the value in the high bits (P010 / P012 / P016: NVDEC, DXGI, hwdownload): NV12's layout of 16-bit words,
# even width, height and rowStride >= 2 * width, height * rowStride * 3 / 2 bytes (cv2's (3H/2) x W CV_16UC1 Mat); each sample
# is read as its high byte.  16-bit planes (yuv420p10le / p12le, P016 surfaces) go to fdt_detect_yuv_planes16 with sampleBits.
FDT_FMT_P010 = 0x1003
SAMPLE_BITS = (10, 12, 16)
FDT_MEM_HOST, FDT_MEM_DEVICE = 0, 1
# EXIF orientation of a stored frame (fdt_detect_batch_oriented / fdt_detect_frames_oriented): the upright image is
# oracle.jpeg_ops.exif_transform(stored, orientation)
(FDT_ORIENT_UPRIGHT, FDT_ORIENT_MIRROR_H, FDT_ORIENT_ROT180, FDT_ORIENT_MIRROR_V, FDT_ORIENT_TRANSPOSE, FDT_ORIENT_ROT90_CW,
 FDT_ORIENT_TRANSVERSE, FDT_ORIENT_ROT90_CCW) = range(1, 9)
# face crops of the detect calls (fdt_set_face_crops): kinds and layout flags (0 = u8 HWC BGR)
FDT_CROP_EMBEDDING, FDT_CROP_FACE = 0, 1
FDT_CROP_RGB, FDT_CROP_CHW, FDT_CROP_F32 = 1, 2, 4
FDT_MAX_FACES = 100
FDT_MESH_FLOATS = 1404
FDT_IRIS_FLOATS = 456


class FdtConfig(C.Structure):
    _fields_ = [("struct_size", C.c_int32), ("model", C.c_int32), ("device", C.c_int32),
                ("max_batch", C.c_int32), ("max_faces", C.c_int32), ("fuse_level", C.c_int32),
                ("min_score", C.c_double), ("min_face_size", C.c_double), ("min_face_presence", C.c_double)]


class FdtFace(C.Structure):
    _fields_ = [("xmin", C.c_double), ("ymin", C.c_double), ("xmax", C.c_double), ("ymax", C.c_double),
                ("score", C.c_double), ("keypoints", C.c_double * 12), ("mesh_score", C.c_double),
                ("has_mesh", C.c_int32), ("anchor_index", C.c_int32), ("has_iris", C.c_int32), ("reserved", C.c_int32)]


class FdtFrame(C.Structure):
    """fdt_frame: one frame of a mixed batch (fdt_detect_frames)."""
    _fields_ = [("data", C.c_void_p), ("width", C.c_int32), ("height", C.c_int32), ("row_stride", C.c_int32),
                ("mat_type", C.c_int32)]


class FdtYuvPlanes(C.Structure):
    """fdt_yuv_planes: one YUV 4:2:0 frame as a Y, a U and a V plane, each with its own base and row stride, U and V sharing a
    pixel stride of 1 or 2 (fdt_detect_yuv_planes)."""
    _fields_ = [("plane", C.c_void_p * 3), ("row_stride", C.c_int32 * 3), ("width", C.c_int32), ("height", C.c_int32),
                ("pixel_stride", C.c_int32), ("reserved", C.c_int32)]


class FdtCropSpec(C.Structure):
    """fdt_crop_spec: the face crops every detect call returns (fdt_set_face_crops), 40 bytes."""
    _fields_ = [("struct_size", C.c_int32), ("kind", C.c_int32), ("out_size", C.c_int32), ("layout", C.c_int32),
                ("scale", C.c_float * 3), ("bias", C.c_float * 3)]


# every symbol include/fdt_api.h declares: name -> (restype, argtypes)
P = C.c_void_p
u8p = C.POINTER(C.c_uint8)
i32p = C.POINTER(C.c_int32)
f32p = C.POINTER(C.c_float)
f64p = C.POINTER(C.c_double)
SIGNATURES = {
    "fdt_default_config": (None, [C.POINTER(FdtConfig)]),
    "fdt_create": (C.c_int32, [C.POINTER(FdtConfig), C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, C.POINTER(P)]),
    "fdt_create_ex": (C.c_int32, [C.POINTER(FdtConfig), C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t,
                                  i32p, C.c_int32, C.POINTER(P)]),
    "fdt_destroy": (C.c_int32, [P]),
    "fdt_detect_batch": (C.c_int32, [P, P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                     C.POINTER(FdtFace), i32p, f32p, f32p]),
    "fdt_detect_frames": (C.c_int32, [P, C.POINTER(FdtFrame), C.c_int32, C.c_int32, C.c_int32, C.POINTER(FdtFace), i32p, f32p, f32p]),
    "fdt_detect_batch_oriented": (C.c_int32, [P, P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                              C.c_int32, C.POINTER(FdtFace), i32p, f32p, f32p]),
    "fdt_detect_frames_oriented": (C.c_int32, [P, C.POINTER(FdtFrame), i32p, C.c_int32, C.c_int32, C.c_int32, C.POINTER(FdtFace),
                                               i32p, f32p, f32p]),
    "fdt_detect_yuv_planes": (C.c_int32, [P, C.POINTER(FdtYuvPlanes), i32p, C.c_int32, C.c_int32, C.c_int32, C.POINTER(FdtFace),
                                          i32p, f32p, f32p]),
    "fdt_detect_yuv_planes16": (C.c_int32, [P, C.POINTER(FdtYuvPlanes), i32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                            C.POINTER(FdtFace), i32p, f32p, f32p]),
    "fdt_detect_jpeg_batch": (C.c_int32, [P, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_int32, C.c_int32, C.POINTER(FdtFace),
                                          i32p, f32p, f32p, i32p, i32p]),
    "fdt_detect_one": (C.c_int32, [P, P, C.c_size_t, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(FdtFace), i32p, f32p, f32p]),
    "fdt_detect_batch_device": (C.c_int32, [P, P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                            C.POINTER(P), C.POINTER(P)]),
    "fdt_synchronize": (C.c_int32, [P]),
    "fdt_get_info": (C.c_int32, [P, i32p, i32p, i32p, i32p, i32p]),
    "fdt_get_anchors": (C.c_int32, [P, f64p]),
    "fdt_letterbox_params": (C.c_int32, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, i32p]),
    "fdt_alloc_pinned": (C.c_int32, [C.c_size_t, C.POINTER(P)]),
    "fdt_free_pinned": (C.c_int32, [P]),
    "fdt_alloc_device": (C.c_int32, [P, C.c_size_t, C.POINTER(P)]),
    "fdt_free_device": (C.c_int32, [P, P]),
    "fdt_copy_to_device": (C.c_int32, [P, P, P, C.c_size_t]),
    "fdt_copy_to_host": (C.c_int32, [P, P, P, C.c_size_t]),
    "fdt_debug_get_letterboxed": (C.c_int32, [P, C.c_int32, P]),
    "fdt_debug_get_input_tensor": (C.c_int32, [P, C.c_int32, P]),
    "fdt_debug_get_raw_heads": (C.c_int32, [P, C.c_int32, P, P]),
    "fdt_debug_get_candidates": (C.c_int32, [P, C.c_int32, P, C.c_int32, i32p]),
    "fdt_debug_get_tensor": (C.c_int32, [P, C.c_int32, C.c_int32, C.c_int32, P, C.c_size_t, i32p]),
    "fdt_debug_get_mesh_stage": (C.c_int32, [P, C.c_int32, P, P, P, i32p]),
    "fdt_debug_get_iris_stage": (C.c_int32, [P, C.c_int32, P, P, P, P, i32p]),
    "fdt_debug_decode": (C.c_int32, [P, P, P, P, C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_double, P,
                                     C.POINTER(FdtFace), i32p, P, i32p]),
    "fdt_debug_nms": (C.c_int32, [P, P, C.c_int32, C.c_double, C.c_double, P, C.POINTER(FdtFace), i32p]),
    "fdt_extract_aligned_squares": (C.c_int32, [P, P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, P, C.c_int32, C.c_int32, P, i32p]),
    "fdt_profile_net": (C.c_int32, [P, C.c_int32, C.c_int32, C.c_int32, f32p, C.c_int32, i32p]),
    "fdt_get_net_step_info": (C.c_int32, [P, C.c_int32, C.c_int32, C.c_char_p, C.c_char_p, C.c_int32, f64p, f64p]),
    "fdt_num_devices": (C.c_int32, [P]),
    "fdt_detect_jpeg": (C.c_int32, [P, P, C.c_size_t, C.c_int32, C.POINTER(FdtFace), i32p, f32p, f32p, i32p]),
    "fdt_decode_jpeg": (C.c_int32, [P, P, C.c_size_t, P, C.c_size_t, i32p]),
    "fdt_get_decoded_frame": (C.c_int32, [P, P, C.c_size_t]),
    "fdt_host_jpeg_info": (C.c_int32, [P, C.c_size_t, i32p]),
    "fdt_host_jpeg_coefficients": (C.c_int32, [P, C.c_size_t, C.c_int32, P, C.c_size_t, i32p, P]),
    "fdt_host_eye_rois": (C.c_int32, [P, P]),
    "fdt_host_embedding_roi": (C.c_int32, [P, P, P]),
    "fdt_last_launch_count": (C.c_int64, [P]),
    "fdt_last_h2d_bytes": (C.c_int64, [P]),
    "fdt_set_stage_timing": (C.c_int32, [P, C.c_int32]),
    "fdt_get_stage_ms": (C.c_int32, [P, C.c_int32, f32p, i32p]),
    "fdt_timer_begin": (C.c_int32, [P]),
    "fdt_timer_end": (C.c_int32, [P, f32p]),
    "fdt_profile_chunk": (C.c_int32, [P, P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, f32p, C.c_int32, i32p]),
    "fdt_get_step_info": (C.c_int32, [P, C.c_int32, C.c_char_p, C.c_char_p, C.c_int32, f64p, f64p]),
    "fdt_host_anchors": (C.c_int32, [C.c_int32, P, C.c_int32]),
    "fdt_host_plan_describe": (C.c_int32, [C.c_char_p, C.c_size_t, C.c_int32, C.c_char_p, C.c_size_t]),
    "fdt_host_resize_taps": (C.c_int32, [C.c_int32, C.c_int32, C.c_int32, P, P, P, P]),
    "fdt_host_decode_box": (C.c_int32, [P, C.c_double, C.c_double, C.c_double, P, P]),
    "fdt_host_face_roi": (C.c_int32, [P, C.c_double, C.c_double, C.c_int32, P]),
    "fdt_host_tile_walk": (C.c_int32, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, P]),
    "fdt_set_face_crops": (C.c_int32, [P, C.POINTER(FdtCropSpec)]),
    "fdt_get_face_crops": (C.c_int32, [P, C.POINTER(C.c_int64), C.POINTER(P)]),
    "fdt_copy_face_crops": (C.c_int32, [P, P, C.c_size_t, C.c_int32, i32p]),
    "fdt_last_error": (C.c_char_p, [P]),
    "fdt_version": (C.c_char_p, []),
}

_lib = None


def load():
    """Loads libfdt_cuda.so; raises (never falls back) when the CUDA library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("FDT_CUDA_LIB", LIB_PATH))
    if not path.exists():
        raise RuntimeError(
            "libfdt_cuda.so is missing (%s): build it with `python -m face_detection_tflite_b200.build`; "
            "there is no CPU fallback" % path)
    lib = C.CDLL(str(path))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the library lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
