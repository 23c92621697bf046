"""FaceDetector — host-side mirror of the reference's public API for the detection hot path
(lib/src/face_detector.dart): create / initialize / detectFacesFromMatBytes / dispose keep their
names, argument meaning and error behaviour; detectFacesBatch is the new batched entry point.

All compute happens in libfdt_cuda.so behind the C ABI (include/fdt_api.h).  The isolate RPC of
the reference (face_detector.dart:1132-1584) is replaced by one FFI call."""
from __future__ import annotations

import ctypes as C
from pathlib import Path
from typing import List, Optional, Sequence

import numpy as np

from . import _ffi
from .face_types import (IRIS_MODEL_FILE, MESH_MODEL_FILE, MODEL_FILES, Detection, Face, FaceDetectionMode,
                         FaceDetectionModel, FaceMesh, Point, RectF, Size)

ASSETS = Path(__file__).resolve().parent.parent / "assets" / "models"


class StateError(RuntimeError):
    """Dart StateError (not initialised / disposed / double initialise)."""


class FormatException(ValueError):
    """Dart FormatException: the image bytes cannot be decoded (face_detector.dart:476)."""


def _raise(lib, handle, code: int):
    msg = lib.fdt_last_error(handle)
    msg = msg.decode() if msg else "error %d" % code
    if code == _ffi.FDT_ERR_NOT_READY:
        raise StateError(msg)
    if code in (_ffi.FDT_ERR_BAD_ARG, _ffi.FDT_ERR_SIZE_MISMATCH):
        raise ValueError(msg)          # Dart ArgumentError
    if code == _ffi.FDT_ERR_FORMAT:
        raise FormatException(msg)
    if code == _ffi.FDT_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError(msg)


_PACKED = {_ffi.FDT_MAT_8UC1: 1, _ffi.FDT_MAT_8UC3: 3, _ffi.FDT_MAT_8UC4: 4, _ffi.FDT_FMT_RGB: 3, _ffi.FDT_FMT_RGBA: 4}
LAYOUTS = ("bgr", "rgb", "rgb_planar")


def _row_step(mt) -> int:
    """Bytes of one pixel within a row: the packed formats' channels, 1 for YUV and planar RGB (a row is one plane's); 0 when
    matType is unknown."""
    return 1 if mt in _ffi.YUV_FORMATS or mt == _ffi.FDT_FMT_RGB_PLANAR else _PACKED.get(mt, 0)


def _frame_bytes(mt, h, stride) -> int:
    if mt in _ffi.YUV_FORMATS:
        return h * stride * 3 // 2
    return 3 * h * stride if mt == _ffi.FDT_FMT_RGB_PLANAR else h * stride


def _layout(layout) -> str:
    if not isinstance(layout, str) or layout not in LAYOUTS:
        raise ValueError("layout must be one of %s, got %r" % (", ".join(LAYOUTS), layout))
    return layout


def _mat_type(m, i: int, layout: str = "bgr") -> int:
    """The matType of a mat in `layout`: "bgr" (cv.Mat: HxW gray, HxWx3 BGR, HxWx4 BGRA), "rgb" (HxW gray, HxWx3 RGB, HxWx4 RGBA)
    or "rgb_planar" (3xHxW, the R, G and B planes)."""
    if layout == "rgb_planar":
        if not isinstance(m, np.ndarray) or m.dtype != np.uint8 or m.ndim != 3 or m.shape[0] != 3 or m.shape[1] <= 0 or m.shape[2] <= 0:
            raise ValueError("mat %d: layout 'rgb_planar' expects a 3xHxW uint8 array" % i)
        return _ffi.FDT_FMT_RGB_PLANAR
    if not isinstance(m, np.ndarray) or m.dtype != np.uint8 or m.ndim not in (2, 3) or m.shape[0] <= 0 or m.shape[1] <= 0:
        raise ValueError("mat %d: expected an HxW, HxWx3 or HxWx4 uint8 array" % i)
    mt = {1: _ffi.FDT_MAT_8UC1, 3: _ffi.FDT_MAT_8UC3, 4: _ffi.FDT_MAT_8UC4}.get(1 if m.ndim == 2 else m.shape[2])
    if mt is None:
        raise ValueError("mat %d: unsupported Mat type" % i)
    if layout == "rgb":
        mt = {_ffi.FDT_MAT_8UC3: _ffi.FDT_FMT_RGB, _ffi.FDT_MAT_8UC4: _ffi.FDT_FMT_RGBA}.get(mt, mt)
    return mt


def _rows_in_buffer(m: np.ndarray) -> bool:
    """True when height * strides[0] bytes from the view's start stay inside the memory it views (the library reads a frame
    as height whole rows of the row stride)."""
    root = m
    while isinstance(root.base, np.ndarray):
        root = root.base
    byte_bounds = getattr(np, "byte_bounds", None) or np.lib.array_utils.byte_bounds
    return m.ctypes.data + m.shape[0] * m.strides[0] <= byte_bounds(root)[1]


def _frame_geometry(i: int, w, h, mt, stride):
    """(row stride, frame bytes) of one fdt_frame; ValueError for arguments the library cannot take."""
    if not all(isinstance(v, (int, np.integer)) for v in (w, h, mt)) or w <= 0 or h <= 0:
        raise ValueError("frame %d: width, height and matType must be positive integers" % i)
    yuv = mt in _ffi.YUV_FORMATS
    ch = _row_step(mt)
    if ch == 0:
        raise ValueError("frame %d: unknown matType %r" % (i, mt))
    stride = w * ch if stride is None else stride
    if not isinstance(stride, (int, np.integer)) or stride < w * ch:
        raise ValueError("frame %d: rowStride smaller than width * channels" % i)
    if yuv and (w % 2 or h % 2):
        raise ValueError("frame %d: YUV 4:2:0 frames need an even width and height" % i)
    return int(stride), _frame_bytes(mt, h, stride)


def _orientation(o, what: str = "orientation") -> int:
    """An EXIF orientation 1..8 as an int; ValueError otherwise."""
    if isinstance(o, bool) or not isinstance(o, (int, np.integer)) or not 1 <= o <= 8:
        raise ValueError("%s must be an EXIF orientation 1..8, got %r" % (what, o))
    return int(o)


def _orientations(orientations, n: int):
    """A per-frame orientation list as int32 [n] (None: all upright, passed on as None); ValueError otherwise."""
    if orientations is None:
        return None
    if isinstance(orientations, (str, bytes)) or not hasattr(orientations, "__len__") or len(orientations) != n:
        raise ValueError("orientations must be a list of one EXIF orientation per frame (%d)" % n)
    return np.array([_orientation(o, "orientations[%d]" % i) for i, o in enumerate(orientations)], np.int32)


def _plane_extents(i: int, strides, w, h, ps) -> tuple:
    """The sampled extent in bytes of the Y, U and V plane of a separate-plane YUV 4:2:0 frame, (rows - 1) * stride +
    (cols - 1) * step + 1; ValueError for the arguments fdt_detect_yuv_planes refuses."""
    vals = (w, h, ps, *strides)
    if len(strides) != 3 or not all(isinstance(v, (int, np.integer)) and not isinstance(v, bool) for v in vals):
        raise ValueError("frame %d: width, height, pixel stride and the three row strides must be integers" % i)
    if w <= 0 or h <= 0 or w % 2 or h % 2:
        raise ValueError("frame %d: YUV 4:2:0 frames need an even, positive width and height" % i)
    if ps not in (1, 2):
        raise ValueError("frame %d: the chroma pixel stride must be 1 or 2, got %r" % (i, ps))
    if min(strides) <= 0:
        raise ValueError("frame %d: row strides must be positive (bottom-up frames are not supported)" % i)
    cc = (w // 2 - 1) * ps + 1
    if strides[0] < w:
        raise ValueError("frame %d: Y row stride smaller than width" % i)
    if strides[1] < cc or strides[2] < cc:
        raise ValueError("frame %d: chroma row stride smaller than (width / 2 - 1) * pixelStride + 1" % i)
    return (h - 1) * int(strides[0]) + w, (h // 2 - 1) * int(strides[1]) + cc, (h // 2 - 1) * int(strides[2]) + cc


def _upright(w, h, orientation) -> tuple:
    """Size of the upright image of a w x h frame stored in `orientation`: 5-8 swap the axes."""
    return (h, w) if orientation >= 5 else (w, h)


class FaceDetector:
    modelVersion = "1.1.1"   # lib/src/face_detector.dart:54-64

    def __init__(self):
        self._lib = _ffi.load()
        self._h = C.c_void_p()
        self._ready = False
        self._max_faces = _ffi.FDT_MAX_FACES

    # -- lifecycle ------------------------------------------------------------------------------
    @classmethod
    def create(cls, model: FaceDetectionModel = FaceDetectionModel.backCamera, *, minScore: float = 0.0,
               minFaceSize: float = 0.0, minFacePresenceConfidence: float = 0.5, device: int = 0,
               maxBatch: int = 0, maxFaces: int = 0, fuseLevel: int = -1, withMesh: bool = True, withIris: bool = True,
               detectorBytes: Optional[bytes] = None, meshBytes: Optional[bytes] = None,
               irisBytes: Optional[bytes] = None, devices: Optional[Sequence[int]] = None) -> "FaceDetector":
        """FaceDetector.create (face_detector.dart:84-119).  `devices` (new): a list of CUDA device ordinals; every
        detect call then splits its batch across them inside the library (fdt_create_ex)."""
        d = cls()
        d.initialize(model, minScore=minScore, minFaceSize=minFaceSize,
                     minFacePresenceConfidence=minFacePresenceConfidence, device=device, maxBatch=maxBatch,
                     maxFaces=maxFaces, fuseLevel=fuseLevel, withMesh=withMesh, withIris=withIris,
                     detectorBytes=detectorBytes, meshBytes=meshBytes, irisBytes=irisBytes, devices=devices)
        return d

    def initialize(self, model: FaceDetectionModel = FaceDetectionModel.backCamera, *, minScore: float = 0.0,
                   minFaceSize: float = 0.0, minFacePresenceConfidence: float = 0.5, device: int = 0,
                   maxBatch: int = 0, maxFaces: int = 0, fuseLevel: int = -1, withMesh: bool = True, withIris: bool = True,
                   detectorBytes: Optional[bytes] = None, meshBytes: Optional[bytes] = None,
                   irisBytes: Optional[bytes] = None, devices: Optional[Sequence[int]] = None) -> None:
        """FaceDetector.initialize (face_detector.dart:297-415)."""
        if self._ready:
            raise StateError("FaceDetector already initialized")          # :315-317
        model = FaceDetectionModel(model)
        if detectorBytes is None:
            detectorBytes = (ASSETS / MODEL_FILES[model]).read_bytes()   # rootBundle.load (:353-372)
        if meshBytes is None and withMesh:
            meshBytes = (ASSETS / MESH_MODEL_FILE).read_bytes()
        if irisBytes is None and withMesh and withIris:
            irisBytes = (ASSETS / IRIS_MODEL_FILE).read_bytes()
        if not withMesh:
            meshBytes = irisBytes = None
        cfg = _ffi.FdtConfig()
        self._lib.fdt_default_config(C.byref(cfg))
        cfg.model, cfg.device, cfg.max_batch, cfg.max_faces, cfg.fuse_level = int(model), device, maxBatch, maxFaces, fuseLevel
        cfg.min_score, cfg.min_face_size, cfg.min_face_presence = minScore, minFaceSize, minFacePresenceConfidence
        h = C.c_void_p()
        devs = (C.c_int32 * len(devices))(*devices) if devices else None
        rc = self._lib.fdt_create_ex(C.byref(cfg), detectorBytes, len(detectorBytes), meshBytes,
                                     len(meshBytes) if meshBytes else 0, irisBytes, len(irisBytes) if irisBytes else 0,
                                     devs, len(devices) if devices else 0, C.byref(h))
        if rc != _ffi.FDT_OK:
            _raise(self._lib, None, rc)
        self._h = h
        self._ready = True
        self.model = model
        iw, ih, na, mf, mb = (C.c_int32() for _ in range(5))
        self._lib.fdt_get_info(h, C.byref(iw), C.byref(ih), C.byref(na), C.byref(mf), C.byref(mb))
        self.inputWidth, self.inputHeight, self.numAnchors = iw.value, ih.value, na.value
        self._max_faces, self.maxBatch = mf.value, mb.value

    @property
    def isReady(self) -> bool:
        return self._ready

    def dispose(self) -> None:
        """FaceDetector.dispose (face_detector.dart:1061-1081)."""
        if self._ready:
            self._lib.fdt_destroy(self._h)
        self._ready = False
        self._h = C.c_void_p()

    def __del__(self):
        try:
            self.dispose()
        except Exception:
            pass

    def _check(self):
        if not self._ready:
            raise StateError("FaceDetector not initialized. Call initialize() first.")   # :1083-1089

    # -- detection ------------------------------------------------------------------------------
    def detectFacesFromMatBytes(self, data, *, width: int, height: int, matType: int = 16,
                                mode: FaceDetectionMode = FaceDetectionMode.full, orientation: int = 1) -> List[Face]:
        """detectFacesFromMatBytes (face_detector.dart:588-609); the default mode is `full` like the reference's
        (detector + mesh + iris; the blendshape classifier is outside this path).  matType may also be one of the YUV 4:2:0
        formats FDT_FMT_YUV_NV12 / _NV21 / _I420: `data` is then width * height * 3 / 2 bytes (cv2's (3H/2) x W Mat), or one of
        the RGB formats FDT_FMT_RGB / _RGBA / _RGB_PLANAR (width * height * 3, * 4, or 3 * width * height bytes).
        orientation (EXIF 1..8, FDT_ORIENT_*): the frame is stored rotated / mirrored; width and height are the stored size,
        the faces are those of the upright image exif_transform(frame, orientation), normalised to its size."""
        if _orientation(orientation) != 1:
            self._check()
            return self.detectFacesBatch(data, count=1, width=width, height=height, matType=matType, mode=mode,
                                         orientation=orientation)[0]
        self._check()
        buf = np.ascontiguousarray(np.frombuffer(data, np.uint8) if not isinstance(data, np.ndarray) else data.reshape(-1))
        if matType in _ffi.YUV_FORMATS and buf.size != width * height * 3 // 2:
            raise ValueError("bytes length does not equal width * height * 3 / 2")        # helpers.dart:440-447
        faces = (_ffi.FdtFace * self._max_faces)()
        count = C.c_int32(0)
        mode = FaceDetectionMode(mode)
        want_mesh = mode != FaceDetectionMode.fast
        want_iris = mode == FaceDetectionMode.full
        mesh = np.empty((self._max_faces, 468, 3), np.float32) if want_mesh else None
        iris = np.empty((self._max_faces, 152, 3), np.float32) if want_iris else None
        rc = self._lib.fdt_detect_one(self._h, buf.ctypes.data, buf.size, width, height, matType, int(mode), faces,
                                      C.byref(count), mesh.ctypes.data_as(_ffi.f32p) if want_mesh else None,
                                      iris.ctypes.data_as(_ffi.f32p) if want_iris else None)
        if rc != _ffi.FDT_OK:
            _raise(self._lib, self._h, rc)
        return [self._to_face(faces[i], mesh[i] if want_mesh else None, width, height, iris[i] if want_iris else None)
                for i in range(count.value)]

    def detectFacesFromBytes(self, imageBytes, *, mode: FaceDetectionMode = FaceDetectionMode.full) -> List[Face]:
        """detectFacesFromBytes (face_detector.dart:477-485): encoded image bytes (JPEG) -> faces.  The reference decodes with
        cv.imdecode; here the host runs the Huffman decoder and the device does the rest (bit-exact with cv.imdecode, EXIF
        orientation included).  Raises FormatException when the bytes cannot be decoded, like the reference."""
        self._check()
        buf = np.frombuffer(bytes(imageBytes), np.uint8)
        faces = (_ffi.FdtFace * self._max_faces)()
        count = C.c_int32(0)
        mode = FaceDetectionMode(mode)
        want_mesh = mode != FaceDetectionMode.fast
        want_iris = mode == FaceDetectionMode.full
        mesh = np.empty((self._max_faces, 468, 3), np.float32) if want_mesh else None
        iris = np.empty((self._max_faces, 152, 3), np.float32) if want_iris else None
        wh = (C.c_int32 * 2)()
        rc = self._lib.fdt_detect_jpeg(self._h, buf.ctypes.data, buf.size, int(mode), faces, C.byref(count),
                                       mesh.ctypes.data_as(_ffi.f32p) if want_mesh else None,
                                       iris.ctypes.data_as(_ffi.f32p) if want_iris else None, wh)
        if rc != _ffi.FDT_OK:
            _raise(self._lib, self._h, rc)
        return [self._to_face(faces[i], mesh[i] if want_mesh else None, wh[0], wh[1], iris[i] if want_iris else None)
                for i in range(count.value)]

    def decodeImage(self, imageBytes) -> np.ndarray:
        """The decoder alone (cv.imdecode(bytes, IMREAD_COLOR)): HxWx3 BGR uint8."""
        self._check()
        buf = np.frombuffer(bytes(imageBytes), np.uint8)
        wh = (C.c_int32 * 2)()
        rc = self._lib.fdt_decode_jpeg(self._h, buf.ctypes.data, buf.size, None, 0, wh)
        if rc != _ffi.FDT_OK:
            _raise(self._lib, self._h, rc)
        out = np.empty((wh[1], wh[0], 3), np.uint8)
        rc = self._lib.fdt_get_decoded_frame(self._h, out.ctypes.data, out.size)
        if rc != _ffi.FDT_OK:
            _raise(self._lib, self._h, rc)
        return out

    def detectFacesFromMat(self, mat: np.ndarray, *, mode: FaceDetectionMode = FaceDetectionMode.full,
                           orientation: int = 1, layout: str = "bgr") -> List[Face]:
        """detectFacesFromMat (face_detector.dart:559-572): `mat` is an HxW[xC] uint8 array (cv.Mat), stored in EXIF
        `orientation` (see detectFacesFromMatBytes).  layout: "bgr" (cv.Mat channel order), "rgb" (HxWx3 RGB, HxWx4 RGBA, HxW
        gray: PIL, imageio, Flutter rawRgba) or "rgb_planar" (3xHxW, e.g. a decoded torchvision image moved to the host).  The
        faces equal those of the BGR image."""
        if _layout(layout) != "bgr":
            mt = _mat_type(mat, 0, layout)
            h, w = mat.shape[1:] if mt == _ffi.FDT_FMT_RGB_PLANAR else mat.shape[:2]
            return self.detectFacesFromMatBytes(np.ascontiguousarray(mat), width=w, height=h, matType=mt, mode=mode,
                                                orientation=orientation)
        ch = 1 if mat.ndim == 2 else mat.shape[2]
        mt = {1: _ffi.FDT_MAT_8UC1, 3: _ffi.FDT_MAT_8UC3, 4: _ffi.FDT_MAT_8UC4}.get(ch)
        if mt is None or mat.dtype != np.uint8:
            raise ValueError("unsupported Mat type")
        return self.detectFacesFromMatBytes(np.ascontiguousarray(mat), width=mat.shape[1], height=mat.shape[0],
                                            matType=mt, mode=mode, orientation=orientation)

    def detectFacesBatch(self, frames, *, count: int, width: int, height: int, matType: int = 16,
                         mode: FaceDetectionMode = FaceDetectionMode.fast, orientation: int = 1) -> List[List[Face]]:
        """New batched entry point: `frames` holds `count` packed frames (bytes / uint8 array), or `count` YUV 4:2:0 frames of
        width * height * 3 / 2 bytes with matType FDT_FMT_YUV_NV12 / _NV21 / _I420.  orientation: EXIF 1..8 of every frame
        (see detectBatchRaw); the faces refer to the upright image."""
        uw, uh = _upright(width, height, _orientation(orientation))
        self._check()
        faces, counts, mesh, iris = self.detectBatchRaw(frames, count=count, width=width, height=height,
                                                        matType=matType, mode=mode, withIris=True, orientation=orientation)
        out = []
        for b in range(count):
            out.append([self._to_face(faces[b * self._max_faces + j], mesh[b, j] if mesh is not None else None, uw, uh,
                                      iris[b, j] if iris is not None else None)
                        for j in range(int(counts[b]))])
        return out

    def detectBatchRaw(self, frames, *, count: int, width: int, height: int, matType: int = 16,
                       mode: FaceDetectionMode = FaceDetectionMode.fast, memKind: int = _ffi.FDT_MEM_HOST,
                       rowStride: Optional[int] = None, withIris: bool = False, orientation: int = 1):
        """fdt_detect_batch with array outputs: (FdtFace array, counts int32[count], mesh f32 or None) and, with
        withIris=True, a fourth element iris f32 [count, max_faces, 152, 3] (None unless mode is full).
        `frames` may be a numpy array / bytes (host) or an integer device pointer with memKind=FDT_MEM_DEVICE (a CUDA tensor:
        t.data_ptr()).  YUV 4:2:0 formats: rowStride is the Y-plane stride (default: width) and a frame is
        height * rowStride * 3 / 2 bytes.  FDT_FMT_RGB_PLANAR: rowStride is one plane's row stride (default: width) and a frame
        is 3 * height * rowStride bytes.
        orientation (EXIF 1..8, FDT_ORIENT_*; fdt_detect_batch_oriented): every frame is stored rotated / mirrored.  width,
        height and rowStride describe the stored frames; faces are normalised to the upright image exif_transform(frame,
        orientation) and mesh / iris points are in its pixels."""
        orientation = _orientation(orientation)
        self._check()
        yuv = matType in _ffi.YUV_FORMATS
        ch = _row_step(matType)
        stride = rowStride if rowStride is not None else width * ch
        if ch and stride < width * ch:
            raise ValueError("rowStride smaller than width * channels")
        frame_bytes = _frame_bytes(matType, height, stride)
        if isinstance(frames, int):
            ptr = frames
        else:
            buf = np.ascontiguousarray(np.frombuffer(frames, np.uint8) if not isinstance(frames, np.ndarray) else frames.reshape(-1))
            if buf.size != count * frame_bytes:
                raise ValueError("frames length does not equal count * %sheight * rowStride%s" % (
                    "3 * " if matType == _ffi.FDT_FMT_RGB_PLANAR else "", " * 3 / 2" if yuv else ""))   # helpers.dart:440-447
            ptr = buf.ctypes.data
        faces = (_ffi.FdtFace * max(1, count * self._max_faces))()
        counts = np.zeros(max(1, count), np.int32)
        mode = FaceDetectionMode(mode)
        want_mesh = mode != FaceDetectionMode.fast
        want_iris = mode == FaceDetectionMode.full
        mesh = np.zeros((count, self._max_faces, 468, 3), np.float32) if want_mesh else None
        iris = np.zeros((count, self._max_faces, 152, 3), np.float32) if want_iris else None
        outs = (faces, counts.ctypes.data_as(_ffi.i32p), mesh.ctypes.data_as(_ffi.f32p) if want_mesh else None,
                iris.ctypes.data_as(_ffi.f32p) if want_iris else None)
        if orientation == 1:
            rc = self._lib.fdt_detect_batch(self._h, ptr, count, width, height, stride, matType, int(mode), memKind, *outs)
        else:
            rc = self._lib.fdt_detect_batch_oriented(self._h, ptr, count, width, height, stride, matType, orientation, int(mode),
                                                     memKind, *outs)
        if rc != _ffi.FDT_OK:
            _raise(self._lib, self._h, rc)
        return (faces, counts[:count], mesh, iris) if withIris else (faces, counts[:count], mesh)

    # -- mixed batches: frames of different sizes and formats, and encoded images, in one call ----------------------------
    def detectFacesFromMats(self, mats, *, mode: FaceDetectionMode = FaceDetectionMode.full,
                            orientations=None, layout: str = "bgr") -> List[List[Face]]:
        """detectFacesFromMat over a list of HxW / HxWx3 / HxWx4 uint8 arrays of any sizes, in one batched call
        (fdt_detect_frames).  A row-padded view (e.g. a crop of a larger array) goes in uncopied with strides[0] as its row
        stride.  Returns one list of faces per mat, each normalised to its own mat.  orientations: one EXIF orientation 1..8
        per mat (fdt_detect_frames_oriented), or None for all upright; faces then refer to each mat's upright image.
        layout: as detectFacesFromMat, for every mat.  A 3xHxW view whose rows are padded but whose planes are height rows
        apart (e.g. a crop of the columns of a larger CHW array) goes in uncopied; any other planar view is copied."""
        mats = list(mats)
        layout = _layout(layout)
        orients = _orientations(orientations, len(mats))
        frames, keep = [], []
        for i, m in enumerate(mats):
            mt = _mat_type(m, i, layout)
            if mt == _ffi.FDT_FMT_RGB_PLANAR:
                h, w = m.shape[1:]
                if m.strides[2] != 1 or m.strides[1] < w or m.strides[0] != h * m.strides[1] or not _rows_in_buffer(m):
                    m = np.ascontiguousarray(m)
                keep.append(m)
                frames.append((m.ctypes.data, w, h, m.strides[1], mt))
                continue
            if m.strides[-1] != 1 or (m.ndim == 3 and m.strides[1] != m.shape[2]) or m.strides[0] < m.shape[1] * m.strides[1] \
                    or not _rows_in_buffer(m):
                m = np.ascontiguousarray(m)
            keep.append(m)
            frames.append((m.ctypes.data, m.shape[1], m.shape[0], m.strides[0], mt))
        self._check()
        faces, counts, mesh, iris = self._detect_frames(frames, mode, _ffi.FDT_MEM_HOST, orients)
        sizes = [_upright(f[1], f[2], 1 if orients is None else orients[i]) for i, f in enumerate(frames)]
        return self._faces_per_frame(faces, counts, mesh, iris, sizes)

    def detectFramesRaw(self, frames, *, mode: FaceDetectionMode = FaceDetectionMode.fast, memKind: int = _ffi.FDT_MEM_HOST,
                        orientations=None):
        """fdt_detect_frames with array outputs.  `frames` is a list of (data, width, height, matType[, rowStride]) tuples: data
        is a numpy array / bytes of exactly height * rowStride bytes (YUV 4:2:0: height * rowStride * 3 / 2; planar RGB:
        3 * height * rowStride), or an integer device pointer with memKind=FDT_MEM_DEVICE.  rowStride defaults to
        width * channels (YUV and planar RGB: width).  Returns
        (FdtFace array [n * max_faces], counts int32 [n], mesh f32 [n, max_faces, 468, 3] or None,
        iris f32 [n, max_faces, 152, 3] or None).  orientations: one EXIF orientation 1..8 per frame
        (fdt_detect_frames_oriented; results refer to each frame's upright image), or None for all upright."""
        if memKind not in (_ffi.FDT_MEM_HOST, _ffi.FDT_MEM_DEVICE):
            raise ValueError("memKind must be FDT_MEM_HOST or FDT_MEM_DEVICE")
        frames = list(frames)
        orients = _orientations(orientations, len(frames))
        descs, keep = [], []
        for i, fr in enumerate(frames):
            if not isinstance(fr, (tuple, list)) or len(fr) not in (4, 5):
                raise ValueError("frame %d: expected (data, width, height, matType[, rowStride])" % i)
            data, w, h, mt = fr[:4]
            stride, nbytes = _frame_geometry(i, w, h, mt, fr[4] if len(fr) == 5 else None)
            if memKind == _ffi.FDT_MEM_DEVICE:
                if not isinstance(data, int):
                    raise ValueError("frame %d: FDT_MEM_DEVICE frames are integer device pointers" % i)
                ptr = data
            else:
                if isinstance(data, int):
                    raise ValueError("frame %d: host frames are numpy arrays or bytes" % i)
                buf = np.ascontiguousarray(np.frombuffer(data, np.uint8) if not isinstance(data, np.ndarray) else data.reshape(-1))
                if buf.dtype != np.uint8 or buf.size != nbytes:
                    raise ValueError("frame %d: data length does not equal %sheight * rowStride%s" % (
                        i, "3 * " if mt == _ffi.FDT_FMT_RGB_PLANAR else "", " * 3 / 2" if mt in _ffi.YUV_FORMATS else ""))
                keep.append(buf)
                ptr = buf.ctypes.data
            descs.append((ptr, w, h, stride, mt))
        self._check()
        return self._detect_frames(descs, mode, memKind, orients)

    # -- YUV 4:2:0 frames as three separate planes: decoder surfaces, AVFrames, Android YUV_420_888 images --------------------
    def detectFacesFromYuvPlanes(self, frames, *, mode: FaceDetectionMode = FaceDetectionMode.full,
                                 orientations=None) -> List[List[Face]]:
        """Faces in YUV 4:2:0 frames given as (y, u, v) triples of 2-D uint8 arrays (fdt_detect_yuv_planes): Y is height x width,
        U and V are height / 2 x width / 2.  strides[0] of each plane is its row stride; strides[1] is 1 for Y and the chroma
        pixel stride, 1 or 2 and the same for U and V.  NumPy views describe every layout without a copy: an NV12 chroma plane
        uv gives uv[:, 0::2], uv[:, 1::2]; an AVFrame gives its three planes; an Android YUV_420_888 image its three buffers
        (pixelStride 2: U and V views into one interleaved buffer, or buffers that end at their last sample).  Returns one list
        of faces per frame, normalised to its upright image.  orientations: one EXIF orientation 1..8 per frame, or None."""
        frames = list(frames)
        orients = _orientations(orientations, len(frames))
        descs = []
        for i, fr in enumerate(frames):
            if not isinstance(fr, (tuple, list)) or len(fr) != 3 or \
                    not all(isinstance(p, np.ndarray) and p.dtype == np.uint8 and p.ndim == 2 for p in fr):
                raise ValueError("frame %d: expected (y, u, v), three 2-D uint8 arrays" % i)
            y, u, v = fr
            h, w = y.shape
            if u.shape != (h // 2, w // 2) or v.shape != (h // 2, w // 2):
                raise ValueError("frame %d: U and V must be height / 2 x width / 2 (Y is %d x %d)" % (i, h, w))
            if y.strides[1] != 1:
                raise ValueError("frame %d: the Y plane's pixels must be adjacent (strides[1] == 1)" % i)
            if u.strides[1] != v.strides[1]:
                raise ValueError("frame %d: U and V need the same pixel stride" % i)
            strides = (y.strides[0], u.strides[0], v.strides[0])
            _plane_extents(i, strides, w, h, u.strides[1])
            descs.append(((y.ctypes.data, u.ctypes.data, v.ctypes.data), strides, w, h, u.strides[1]))
        self._check()
        faces, counts, mesh, iris = self._detect_planes(descs, mode, _ffi.FDT_MEM_HOST, orients)
        sizes = [_upright(d[2], d[3], 1 if orients is None else orients[i]) for i, d in enumerate(descs)]
        return self._faces_per_frame(faces, counts, mesh, iris, sizes)

    def detectYuvPlanesRaw(self, frames, *, mode: FaceDetectionMode = FaceDetectionMode.fast, memKind: int = _ffi.FDT_MEM_HOST,
                           orientations=None):
        """fdt_detect_yuv_planes with array outputs, as detectFramesRaw.  `frames` is a list of
        ((y, u, v), (yStride, uStride, vStride), width, height, pixelStride) tuples: the planes are integer device pointers with
        memKind=FDT_MEM_DEVICE (e.g. torch CUDA tensors' data_ptr()), else numpy arrays or bytes, each holding at least its
        plane's sampled extent from its first byte."""
        if memKind not in (_ffi.FDT_MEM_HOST, _ffi.FDT_MEM_DEVICE):
            raise ValueError("memKind must be FDT_MEM_HOST or FDT_MEM_DEVICE")
        frames = list(frames)
        orients = _orientations(orientations, len(frames))
        descs, keep = [], []
        for i, fr in enumerate(frames):
            if not isinstance(fr, (tuple, list)) or len(fr) != 5 or not isinstance(fr[0], (tuple, list)) or len(fr[0]) != 3 \
                    or not isinstance(fr[1], (tuple, list)):
                raise ValueError("frame %d: expected ((y, u, v), (yStride, uStride, vStride), width, height, pixelStride)" % i)
            planes, strides, w, h, ps = fr
            extents = _plane_extents(i, tuple(strides), w, h, ps)
            ptrs = []
            for k, (p, ext) in enumerate(zip(planes, extents)):
                if memKind == _ffi.FDT_MEM_DEVICE:
                    if isinstance(p, bool) or not isinstance(p, int):
                        raise ValueError("frame %d: FDT_MEM_DEVICE planes are integer device pointers" % i)
                    ptrs.append(p)
                    continue
                if isinstance(p, int):
                    raise ValueError("frame %d: host planes are numpy arrays or bytes" % i)
                buf = np.frombuffer(p, np.uint8) if not isinstance(p, np.ndarray) else p
                if buf.dtype != np.uint8 or not buf.flags.c_contiguous or buf.size < ext:
                    raise ValueError("frame %d: plane %s is not a contiguous uint8 buffer of at least its sampled extent (%d bytes)"
                                     % (i, "YUV"[k], ext))
                keep.append(buf)
                ptrs.append(buf.ctypes.data)
            descs.append((tuple(ptrs), tuple(int(s) for s in strides), int(w), int(h), int(ps)))
        self._check()
        return self._detect_planes(descs, mode, memKind, orients)

    def _detect_planes(self, descs, mode, memKind, orients):
        n = len(descs)
        arr = (_ffi.FdtYuvPlanes * max(1, n))()
        for k, (ptrs, strides, w, h, ps) in enumerate(descs):
            arr[k].plane = (C.c_void_p * 3)(*ptrs)
            arr[k].row_stride = (C.c_int32 * 3)(*strides)
            arr[k].width, arr[k].height, arr[k].pixel_stride = w, h, ps
        faces, counts, mesh, iris = self._outputs(n, mode)
        rc = self._lib.fdt_detect_yuv_planes(self._h, arr, orients.ctypes.data_as(_ffi.i32p) if orients is not None else None, n,
                                             int(FaceDetectionMode(mode)), memKind, faces, counts.ctypes.data_as(_ffi.i32p),
                                             mesh.ctypes.data_as(_ffi.f32p) if mesh is not None else None,
                                             iris.ctypes.data_as(_ffi.f32p) if iris is not None else None)
        if rc != _ffi.FDT_OK:
            _raise(self._lib, self._h, rc)
        return faces, counts[:n], mesh, iris

    def detectFacesFromBytesBatch(self, images, *, mode: FaceDetectionMode = FaceDetectionMode.full) -> List[Optional[List[Face]]]:
        """detectFacesFromBytes over a list of encoded images (JPEG) in one call (fdt_detect_jpeg_batch).  An image that
        cannot be decoded gives None in its place instead of raising, so one bad photo does not discard the batch."""
        faces, counts, mesh, iris, wh, status = self.detectBytesBatchRaw(images, mode=mode)
        out = self._faces_per_frame(faces, counts, mesh, iris, [tuple(x) for x in wh])
        return [f if status[i] == _ffi.FDT_OK else None for i, f in enumerate(out)]

    def detectBytesBatchRaw(self, images, *, mode: FaceDetectionMode = FaceDetectionMode.full):
        """fdt_detect_jpeg_batch with array outputs: (FdtFace array, counts, mesh or None, iris or None, wh int32 [n, 2],
        status int32 [n]); status is FDT_OK, FDT_ERR_FORMAT or FDT_ERR_UNSUPPORTED per image."""
        bufs = []
        for i, im in enumerate(images):
            if not isinstance(im, (bytes, bytearray, memoryview, np.ndarray)):
                raise ValueError("image %d: expected encoded bytes" % i)
            bufs.append(np.frombuffer(bytes(im), np.uint8) if not isinstance(im, np.ndarray) else np.ascontiguousarray(im, np.uint8).reshape(-1))
        self._check()
        n = len(bufs)
        ptrs = (C.c_void_p * max(1, n))(*[b.ctypes.data if b.size else None for b in bufs])
        sizes = (C.c_size_t * max(1, n))(*[b.size for b in bufs])
        faces, counts, mesh, iris = self._outputs(n, mode)
        wh = np.zeros((max(1, n), 2), np.int32)
        status = np.zeros(max(1, n), np.int32)
        rc = self._lib.fdt_detect_jpeg_batch(self._h, ptrs, sizes, n, int(mode), faces, counts.ctypes.data_as(_ffi.i32p),
                                             mesh.ctypes.data_as(_ffi.f32p) if mesh is not None else None,
                                             iris.ctypes.data_as(_ffi.f32p) if iris is not None else None,
                                             wh.ctypes.data_as(_ffi.i32p), status.ctypes.data_as(_ffi.i32p))
        if rc != _ffi.FDT_OK:
            _raise(self._lib, self._h, rc)
        return faces, counts[:n], mesh, iris, wh[:n], status[:n]

    def _outputs(self, n: int, mode):
        mode = FaceDetectionMode(mode)
        faces = (_ffi.FdtFace * max(1, n * self._max_faces))()
        counts = np.zeros(max(1, n), np.int32)
        mesh = np.zeros((n, self._max_faces, 468, 3), np.float32) if mode != FaceDetectionMode.fast else None
        iris = np.zeros((n, self._max_faces, 152, 3), np.float32) if mode == FaceDetectionMode.full else None
        return faces, counts, mesh, iris

    def _detect_frames(self, descs, mode, memKind, orients=None):
        n = len(descs)
        arr = (_ffi.FdtFrame * max(1, n))(*[_ffi.FdtFrame(*d) for d in descs])   # (data, width, height, row_stride, mat_type)
        faces, counts, mesh, iris = self._outputs(n, mode)
        outs = (faces, counts.ctypes.data_as(_ffi.i32p), mesh.ctypes.data_as(_ffi.f32p) if mesh is not None else None,
                iris.ctypes.data_as(_ffi.f32p) if iris is not None else None)
        if orients is None:
            rc = self._lib.fdt_detect_frames(self._h, arr, n, int(FaceDetectionMode(mode)), memKind, *outs)
        else:
            rc = self._lib.fdt_detect_frames_oriented(self._h, arr, orients.ctypes.data_as(_ffi.i32p), n,
                                                      int(FaceDetectionMode(mode)), memKind, *outs)
        if rc != _ffi.FDT_OK:
            _raise(self._lib, self._h, rc)
        return faces, counts[:n], mesh, iris

    def _faces_per_frame(self, faces, counts, mesh, iris, sizes):
        mf = self._max_faces
        return [[self._to_face(faces[b * mf + j], mesh[b, j] if mesh is not None else None, w, h, iris[b, j] if iris is not None else None)
                 for j in range(int(counts[b]))] for b, (w, h) in enumerate(sizes)]

    @staticmethod
    def _to_face(f, mesh, width, height, iris=None) -> Face:
        size = Size(float(width), float(height))
        det = Detection(RectF(f.xmin, f.ymin, f.xmax, f.ymax), f.score, [f.keypoints[k] for k in range(12)], size)
        fm = FaceMesh(np.array(mesh, np.float32), f.mesh_score) if (mesh is not None and f.has_mesh) else None
        pts, packed = [], None
        if iris is not None and f.has_iris:
            packed = np.array(iris, np.float32)
            pts = [Point(float(p[0]), float(p[1]), float(p[2])) for p in packed]
        return Face(det, fm, size, irisPoints=pts, anchorIndex=f.anchor_index, irisPacked=packed)

    # -- embedding alignment (lib/src/models/face_embedding.dart:362-384, face_detector_core.dart:419-452) ----------
    def extractAlignedSquares(self, mat: np.ndarray, rois, outSize: int):
        """extractAlignedSquare (helpers.dart:583-625) on the device for ROIs (cx, cy, size, theta) of one frame.
        Returns (crops u8 [n, outSize, outSize, 3], ok bool[n])."""
        self._check()
        mat = np.ascontiguousarray(mat)
        ch = 1 if mat.ndim == 2 else mat.shape[2]
        mt = {1: _ffi.FDT_MAT_8UC1, 3: _ffi.FDT_MAT_8UC3, 4: _ffi.FDT_MAT_8UC4}[ch]
        r = np.ascontiguousarray(np.asarray(rois, np.float64).reshape(-1, 4))
        out = np.empty((r.shape[0], outSize, outSize, 3), np.uint8)
        ok = np.zeros(r.shape[0], np.int32)
        self._rc(self._lib.fdt_extract_aligned_squares(self._h, mat.ctypes.data, mat.shape[1], mat.shape[0], mat.shape[1] * ch, mt,
                                                       r.ctypes.data, r.shape[0], outSize, out.ctypes.data, ok.ctypes.data_as(_ffi.i32p)))
        return out, ok.astype(bool)

    def embeddingCrop(self, face: Face, mat: np.ndarray, outSize: int = 112) -> np.ndarray:
        """The aligned 112x112 crop getFaceEmbeddingFromEyesDirect feeds MobileFaceNet (face_detector_core.dart:419-452):
        computeEmbeddingAlignment on the (iris-refined) eye keypoints, then extractAlignedSquare(..., -theta).  The
        embedding model itself is not shipped by the reference."""
        lm = face.landmarks
        le, re = lm[0], lm[1]
        out4 = (C.c_double * 4)()
        self._lib.fdt_host_embedding_roi((C.c_double * 2)(le.x, le.y), (C.c_double * 2)(re.x, re.y), out4)
        theta, cx, cy, size = out4
        crops, ok = self.extractAlignedSquares(mat, [[cx, cy, size, -theta]], outSize)
        if not ok[0]:
            raise StateError("Failed to extract aligned face crop for embedding")
        return crops[0]

    # -- parity taps (tests only) -----------------------------------------------------------------
    # The detector taps describe the first n frames of the last call's first chunk (min(count, maxBatch) frames).  After a
    # call of more than two chunks (count > 2 * maxBatch) a later chunk has overwritten that chunk's buffers, and
    # debugLetterboxed, debugInputTensor, debugRawHeads and debugTensor(0, ...) raise ValueError; debugCandidates
    # keeps the first chunk's index sets for any count.
    def debugLetterboxed(self, n: int) -> np.ndarray:
        out = np.empty((n, self.inputHeight, self.inputWidth, 3), np.uint8)
        self._rc(self._lib.fdt_debug_get_letterboxed(self._h, n, out.ctypes.data))
        return out

    def debugInputTensor(self, n: int) -> np.ndarray:
        out = np.empty((n, self.inputHeight, self.inputWidth, 3), np.float32)
        self._rc(self._lib.fdt_debug_get_input_tensor(self._h, n, out.ctypes.data))
        return out

    def debugRawHeads(self, n: int):
        boxes = np.empty((n, self.numAnchors, 16), np.float32)
        scores = np.empty((n, self.numAnchors), np.float32)
        self._rc(self._lib.fdt_debug_get_raw_heads(self._h, n, boxes.ctypes.data, scores.ctypes.data))
        return boxes, scores

    def debugCandidates(self, image: int) -> np.ndarray:
        idx = np.empty(self.numAnchors, np.int32)
        n = C.c_int32(0)
        self._rc(self._lib.fdt_debug_get_candidates(self._h, image, idx.ctypes.data, idx.size, C.byref(n)))
        return idx[:n.value].copy()

    def debugTensor(self, which: int, tensor: int, n: int) -> np.ndarray:
        """A materialised activation of the detector (which=0, first chunk), mesh (1) or iris (2) graph, dense NHWC f32.
        The mesh and iris tensors hold the last call's last mesh / iris pass."""
        dims = (C.c_int32 * 4)()
        self._rc(self._lib.fdt_debug_get_tensor(self._h, which, tensor, n, None, 0, dims))
        out = np.empty(tuple(dims), np.float32)
        self._rc(self._lib.fdt_debug_get_tensor(self._h, which, tensor, n, out.ctypes.data, out.size, dims))
        return out

    def debugMeshStage(self, n: int):
        """The first min(n, m) faces of the last call's LAST mesh pass, m being that pass's size (a pass holds up to
        2 * maxBatch faces of one chunk, in frame then detection order): (crops u8 [., 192, 192, 3], raw mesh outputs
        f32 [., 1404], face-flag logits f32 [.])."""
        crops = np.empty((n, 192, 192, 3), np.uint8)
        raw = np.empty((n, 1404), np.float32)
        flag = np.empty((n,), np.float32)
        got = C.c_int32(0)
        self._rc(self._lib.fdt_debug_get_mesh_stage(self._h, n, crops.ctypes.data, raw.ctypes.data, flag.ctypes.data, C.byref(got)))
        m = min(n, got.value)
        return crops[:m], raw[:m], flag[:m]

    def debugIrisStage(self, n: int):
        """The first m = min(n, faces) faces of the last call's LAST iris pass (the faces of the last mesh pass that passed
        the presence gate and have two valid eye ROIs): (eye crops u8 [2m,64,64,3], rois f64 [2m,4] = cx,cy,size,theta,
        contours f32 [2m,213], iris f32 [2m,15])."""
        crops = np.empty((2 * n, 64, 64, 3), np.uint8)
        rois = np.empty((2 * n, 4), np.float64)
        cont = np.empty((2 * n, 213), np.float32)
        ir = np.empty((2 * n, 15), np.float32)
        got = C.c_int32(0)
        self._rc(self._lib.fdt_debug_get_iris_stage(self._h, n, crops.ctypes.data, rois.ctypes.data, cont.ctypes.data, ir.ctypes.data, C.byref(got)))
        m = 2 * min(n, got.value)
        return crops[:m], rois[:m], cont[:m], ir[:m]

    def debugDecode(self, rawBoxes, rawScores, *, anchors=None, scale: float, scoreThresh: float = 0.5, iouThresh: float = 0.3,
                    padding=None):
        """k_decode_nms on caller-supplied raw heads: boxes [B,N,16], scores [B,N] -> (list of list of FdtFace-like
        dicts, decoded candidates [B][n_cand, 18])."""
        boxes = np.ascontiguousarray(np.asarray(rawBoxes, np.float32))
        scores = np.ascontiguousarray(np.asarray(rawScores, np.float32))
        if boxes.ndim == 2:
            boxes, scores = boxes[None], scores[None]
        B, N = scores.shape
        anc = np.ascontiguousarray(np.asarray(anchors, np.float64).reshape(N, 2)) if anchors is not None else None
        pad = (C.c_double * 4)(*padding) if padding is not None else None
        faces = (_ffi.FdtFace * (B * _ffi.FDT_MAX_FACES))()
        counts = np.zeros(B, np.int32)
        dec = np.zeros((B, N, 18), np.float64)
        ndec = np.zeros(B, np.int32)
        self._rc(self._lib.fdt_debug_decode(self._h, boxes.ctypes.data, scores.ctypes.data, anc.ctypes.data if anc is not None else None,
                                            B, N, float(scale), float(scoreThresh), float(iouThresh), pad, faces,
                                            counts.ctypes.data_as(_ffi.i32p), dec.ctypes.data, ndec.ctypes.data_as(_ffi.i32p)))
        out = [[self._face_row(faces[b * _ffi.FDT_MAX_FACES + j]) for j in range(int(counts[b]))] for b in range(B)]
        return out, [dec[b, :int(ndec[b])] for b in range(B)]

    def debugNms(self, dets17, *, scoreThresh: float, iouThresh: float, padding=None):
        """weightedNms + letterbox removal on the device for detections [n,17] = xmin,ymin,xmax,ymax,score,kp12."""
        d = np.ascontiguousarray(np.asarray(dets17, np.float64).reshape(-1, 17))
        pad = (C.c_double * 4)(*padding) if padding is not None else None
        faces = (_ffi.FdtFace * _ffi.FDT_MAX_FACES)()
        count = C.c_int32(0)
        self._rc(self._lib.fdt_debug_nms(self._h, d.ctypes.data if d.shape[0] else None, d.shape[0], float(scoreThresh), float(iouThresh), pad, faces, C.byref(count)))
        return [self._face_row(faces[j]) for j in range(count.value)]

    @staticmethod
    def _face_row(f) -> dict:
        return {"box": (f.xmin, f.ymin, f.xmax, f.ymax), "score": f.score, "kp": [f.keypoints[k] for k in range(12)], "index": f.anchor_index}

    def numDevices(self) -> int:
        return int(self._lib.fdt_num_devices(self._h))

    def anchors(self) -> np.ndarray:
        a = np.empty((self.numAnchors, 2), np.float64)
        self._rc(self._lib.fdt_get_anchors(self._h, a.ctypes.data_as(_ffi.f64p)))
        return a

    def lastLaunchCount(self) -> int:
        return int(self._lib.fdt_last_launch_count(self._h))

    def _rc(self, rc):
        if rc != _ffi.FDT_OK:
            _raise(self._lib, self._h, rc)
