/// FaceDetector façade over libfdt_cuda.so: the names, argument meaning and error behaviour of
/// `lib/src/face_detector.dart` (create / initialize / detectFacesFromMatBytes / dispose / isReady) for the
/// detection hot path, plus the new batched entry point `detectFacesBatch`.
///
/// The isolate worker of the reference (`_FaceDetectorWorker`, face_detector.dart:1830-1885) is not needed on this
/// path: one FFI call does letterbox -> BlazeFace -> decode -> weighted NMS [-> warp -> mesh [-> eye warps -> iris]]
/// for the whole batch on the GPU.  For single-frame UI use wrap a call in `Isolate.run`.
library;

import 'dart:ffi';
import 'dart:typed_data';

import 'package:ffi/ffi.dart';
import 'package:flutter/services.dart' show rootBundle;

import '../shared/face_model_config.dart' show faceDetectionModelFile;
import '../shared/face_types.dart';
import 'fdt_ffi.dart';

const String _kAssetRoot = 'packages/face_detection_tflite/assets/models';
const String _kMeshModel = 'face_landmark.tflite';
const String _kIrisModel = 'iris_landmark.tflite';

class FdtFaceDetector {
  FdtFaceDetector._();

  final FdtLibrary _lib = FdtLibrary.instance;
  Pointer<Void> _h = nullptr;
  int _maxFaces = kFdtMaxFaces;

  /// face_detector.dart:210
  bool get isReady => _h != nullptr;

  /// Number of CUDA devices a detect call is split across (1 unless [create] was given `devices`).
  int get numDevices => _h == nullptr ? 0 : _lib.numDevices(_h);

  /// FaceDetector.create (face_detector.dart:84-119).  `devices`: optional CUDA device ordinals; with more than one the
  /// library splits every batch across them (fdt_create_ex).
  static Future<FdtFaceDetector> create({
    FaceDetectionModel model = FaceDetectionModel.backCamera,
    double minScore = 0.0,
    double minFaceSize = 0.0,
    double minFacePresenceConfidence = 0.5,
    List<int>? devices,
    int maxBatch = 0,
  }) async {
    final d = FdtFaceDetector._();
    await d.initialize(
      model: model,
      minScore: minScore,
      minFaceSize: minFaceSize,
      minFacePresenceConfidence: minFacePresenceConfidence,
      devices: devices,
      maxBatch: maxBatch,
    );
    return d;
  }

  /// FaceDetector.initialize (face_detector.dart:297-415): loads the bundled models and creates the native handle.
  Future<void> initialize({
    FaceDetectionModel model = FaceDetectionModel.backCamera,
    double minScore = 0.0,
    double minFaceSize = 0.0,
    double minFacePresenceConfidence = 0.5,
    List<int>? devices,
    int maxBatch = 0,
  }) async {
    if (_h != nullptr) {
      throw StateError('FaceDetector already initialized'); // :315-317
    }
    final ByteData det = await rootBundle.load('$_kAssetRoot/${faceDetectionModelFile(model)}');
    final ByteData mesh = await rootBundle.load('$_kAssetRoot/$_kMeshModel');
    final ByteData iris = await rootBundle.load('$_kAssetRoot/$_kIrisModel');
    final arena = Arena();
    try {
      final Pointer<FdtConfig> cfg = arena<FdtConfig>();
      _lib.defaultConfig(cfg);
      cfg.ref
        ..model = model.index
        ..maxBatch = maxBatch
        ..minScore = minScore
        ..minFaceSize = minFaceSize
        ..minFacePresence = minFacePresenceConfidence;
      Pointer<Uint8> copy(ByteData b) {
        final Pointer<Uint8> p = arena<Uint8>(b.lengthInBytes);
        p.asTypedList(b.lengthInBytes).setAll(0, b.buffer.asUint8List(b.offsetInBytes, b.lengthInBytes));
        return p;
      }

      Pointer<Int32> devs = nullptr;
      final int nDev = devices?.length ?? 0;
      if (nDev > 0) {
        devs = arena<Int32>(nDev);
        for (int i = 0; i < nDev; i++) {
          devs[i] = devices![i];
        }
      }
      final Pointer<Pointer<Void>> out = arena<Pointer<Void>>();
      final int rc = _lib.createEx(cfg, copy(det), det.lengthInBytes, copy(mesh), mesh.lengthInBytes, copy(iris),
          iris.lengthInBytes, devs, nDev, out);
      if (rc != FdtStatus.ok) {
        _lib.throwFor(rc, nullptr); // ArgumentError for gates outside [0, 1], like validateFaceGates
      }
      _h = out.value;
      final Pointer<Int32> mf = arena<Int32>();
      _lib.getInfo(_h, nullptr, nullptr, nullptr, mf, nullptr);
      _maxFaces = mf.value;
    } finally {
      arena.releaseAll();
    }
  }

  /// An EXIF orientation (kFdtOrient*) must be 1..8; checked before any library call.
  static void _checkOrientation(int orientation) {
    if (orientation < 1 || orientation > 8) {
      throw ArgumentError.value(orientation, 'orientation', 'must be an EXIF orientation 1..8');
    }
  }

  void _check() {
    if (_h == nullptr) {
      throw StateError('FaceDetector not initialized. Call initialize() first.'); // :1083-1089
    }
  }

  /// detectFacesFromMatBytes (face_detector.dart:588-609): same signature and default mode (full).
  Future<List<Face>> detectFacesFromMatBytes(
    Uint8List bytes, {
    required int width,
    required int height,
    int matType = 16,
    FaceDetectionMode mode = FaceDetectionMode.full,
    int orientation = kFdtOrientUpright,
  }) async {
    _checkOrientation(orientation);
    if (orientation != kFdtOrientUpright) {
      // a stored-rotated frame: fdt_detect_batch_oriented with one frame; faces refer to the upright image
      return (await detectFacesBatch(bytes, count: 1, width: width, height: height, matType: matType, mode: mode,
          orientation: orientation))[0];
    }
    _check();
    final arena = Arena();
    try {
      final Pointer<Uint8> src = arena<Uint8>(bytes.length);
      src.asTypedList(bytes.length).setAll(0, bytes);
      final Pointer<FdtFace> faces = arena<FdtFace>(_maxFaces);
      final Pointer<Int32> count = arena<Int32>();
      final bool wantMesh = mode != FaceDetectionMode.fast;
      final bool wantIris = mode == FaceDetectionMode.full;
      final Pointer<Float> mesh = wantMesh ? arena<Float>(_maxFaces * kFdtMeshFloats) : nullptr;
      final Pointer<Float> iris = wantIris ? arena<Float>(_maxFaces * kFdtIrisFloats) : nullptr;
      final int rc = _lib.detectOne(_h, src, bytes.length, width, height, matType, mode.index, faces, count, mesh, iris);
      if (rc != FdtStatus.ok) {
        _lib.throwFor(rc, _h); // ArgumentError on a byte-length mismatch (helpers.dart:440-447)
      }
      return <Face>[for (int i = 0; i < count.value; i++) _toFace(faces[i], mesh, iris, i, width, height)];
    } finally {
      arena.releaseAll();
    }
  }

  /// detectFacesFromBytes (face_detector.dart:477-485): encoded image bytes (JPEG) -> faces; same default mode (full).
  /// The reference decodes with cv.imdecode on the host; here the host only runs the Huffman decoder, the IDCT, chroma
  /// upsampling, colour conversion and EXIF orientation run on the GPU (byte-equal to cv.imdecode).  Throws
  /// [FormatException] when the bytes cannot be decoded, like the reference.
  Future<List<Face>> detectFacesFromBytes(
    Uint8List imageBytes, {
    FaceDetectionMode mode = FaceDetectionMode.full,
  }) async {
    _check();
    final arena = Arena();
    try {
      final Pointer<Uint8> src = arena<Uint8>(imageBytes.length);
      src.asTypedList(imageBytes.length).setAll(0, imageBytes);
      final Pointer<FdtFace> faces = arena<FdtFace>(_maxFaces);
      final Pointer<Int32> count = arena<Int32>();
      final Pointer<Int32> wh = arena<Int32>(2);
      final bool wantMesh = mode != FaceDetectionMode.fast;
      final bool wantIris = mode == FaceDetectionMode.full;
      final Pointer<Float> mesh = wantMesh ? arena<Float>(_maxFaces * kFdtMeshFloats) : nullptr;
      final Pointer<Float> iris = wantIris ? arena<Float>(_maxFaces * kFdtIrisFloats) : nullptr;
      final int rc = _lib.detectJpeg(_h, src, imageBytes.length, mode.index, faces, count, mesh, iris, wh);
      if (rc != FdtStatus.ok) {
        _lib.throwFor(rc, _h); // FormatException for undecodable bytes
      }
      return <Face>[for (int i = 0; i < count.value; i++) _toFace(faces[i], mesh, iris, i, wh[0], wh[1])];
    } finally {
      arena.releaseAll();
    }
  }

  /// New batched entry point: [frames] holds [count] packed frames (count * height * width * channels bytes), or [count]
  /// YUV 4:2:0 frames of width * height * 3 / 2 bytes with matType kFdtFmtYuvNv12 / kFdtFmtYuvNv21 / kFdtFmtYuvI420, or RGB
  /// frames with kFdtFmtRgb / kFdtFmtRgba / kFdtFmtRgbPlanar (a Flutter `ui.Image.toByteData(format: rawRgba)` buffer is one
  /// kFdtFmtRgba frame as it is).
  /// One `fdt_detect_batch` call; results come back in frame order.  [orientation]: the EXIF orientation (kFdtOrient*) every
  /// frame is stored in (`fdt_detect_batch_oriented`); width / height are the stored size, faces refer to the upright image.  For sustained throughput keep the frames in a
  /// buffer from `fdt_alloc_pinned` (see [FdtPinnedFrames]) so the upload runs at PCIe speed.
  Future<List<List<Face>>> detectFacesBatch(
    Uint8List frames, {
    required int count,
    required int width,
    required int height,
    int matType = 16,
    FaceDetectionMode mode = FaceDetectionMode.fast,
    int orientation = kFdtOrientUpright,
  }) async {
    _checkOrientation(orientation);
    _check();
    final int frameBytes = fdtFrameBytes(matType, width, height);
    if (frames.length != count * frameBytes) {
      throw ArgumentError('frames length ${frames.length} does not equal count * frame size ($frameBytes bytes)');
    }
    if (count == 0) return <List<Face>>[];
    final arena = Arena();
    try {
      final Pointer<Uint8> src = arena<Uint8>(frames.length);
      src.asTypedList(frames.length).setAll(0, frames);
      return _detectBatchPtr(arena, src, count, width, height, fdtRowStride(matType, width), matType, mode, orientation);
    } finally {
      arena.releaseAll();
    }
  }

  /// As [detectFacesBatch] on frames already resident in pinned host memory (no copy on the Dart side).
  Future<List<List<Face>>> detectFacesPinned(
    FdtPinnedFrames frames, {
    required int count,
    required int width,
    required int height,
    int matType = 16,
    FaceDetectionMode mode = FaceDetectionMode.fast,
    int orientation = kFdtOrientUpright,
  }) async {
    _checkOrientation(orientation);
    _check();
    if (count * fdtFrameBytes(matType, width, height) > frames.lengthInBytes) {
      throw ArgumentError('pinned buffer smaller than count * frame size');
    }
    final arena = Arena();
    try {
      return _detectBatchPtr(
          arena, frames.pointer, count, width, height, fdtRowStride(matType, width), matType, mode, orientation);
    } finally {
      arena.releaseAll();
    }
  }

  List<List<Face>> _detectBatchPtr(Arena arena, Pointer<Uint8> src, int count, int width, int height, int rowStride,
      int matType, FaceDetectionMode mode, int orientation) {
    final Pointer<FdtFace> faces = arena<FdtFace>(count * _maxFaces);
    final Pointer<Int32> counts = arena<Int32>(count);
    final bool wantMesh = mode != FaceDetectionMode.fast;
    final bool wantIris = mode == FaceDetectionMode.full;
    final Pointer<Float> mesh = wantMesh ? arena<Float>(count * _maxFaces * kFdtMeshFloats) : nullptr;
    final Pointer<Float> iris = wantIris ? arena<Float>(count * _maxFaces * kFdtIrisFloats) : nullptr;
    final int rc = orientation == kFdtOrientUpright
        ? _lib.detectBatch(_h, src, count, width, height, rowStride, matType, mode.index, kFdtMemHost, faces, counts, mesh, iris)
        : _lib.detectBatchOriented(
            _h, src, count, width, height, rowStride, matType, orientation, mode.index, kFdtMemHost, faces, counts, mesh, iris);
    if (rc != FdtStatus.ok) {
      _lib.throwFor(rc, _h);
    }
    // faces are normalised to the upright image: orientations 5-8 swap its axes
    final int uw = orientation >= 5 ? height : width, uh = orientation >= 5 ? width : height;
    final List<List<Face>> out = <List<Face>>[];
    for (int b = 0; b < count; b++) {
      final int n = counts[b];
      out.add(<Face>[
        for (int j = 0; j < n; j++) _toFace(faces[b * _maxFaces + j], mesh, iris, b * _maxFaces + j, uw, uh),
      ]);
    }
    return out;
  }

  /// detectFacesFromMat over a list of frames of any sizes and formats (photos, mixed camera feeds) in one batched
  /// `fdt_detect_frames` call.  Each mat is packed bytes of its own width, height and matType (kFdtFmtYuv* included);
  /// each result list is normalised to its own mat.  [orientations]: one EXIF orientation (kFdtOrient*) per mat, or null
  /// for all upright (`fdt_detect_frames_oriented`); each result list then refers to its mat's upright image.
  Future<List<List<Face>>> detectFacesFromMats(
    List<({Uint8List bytes, int width, int height, int matType})> mats, {
    FaceDetectionMode mode = FaceDetectionMode.full,
    List<int>? orientations,
  }) async {
    if (orientations != null) {
      if (orientations.length != mats.length) {
        throw ArgumentError('orientations: one EXIF orientation per mat (${mats.length})');
      }
      orientations.forEach(_checkOrientation);
    }
    _check();
    for (int i = 0; i < mats.length; i++) {
      final m = mats[i];
      if (m.bytes.length != fdtFrameBytes(m.matType, m.width, m.height)) {
        throw ArgumentError('mat $i: bytes length does not equal its frame size');
      }
    }
    final int n = mats.length;
    if (n == 0) return <List<Face>>[];
    final arena = Arena();
    try {
      final Pointer<FdtFrame> frames = arena<FdtFrame>(n);
      for (int i = 0; i < n; i++) {
        final m = mats[i];
        final Pointer<Uint8> src = arena<Uint8>(m.bytes.length);
        src.asTypedList(m.bytes.length).setAll(0, m.bytes);
        frames[i].data = src;
        frames[i].width = m.width;
        frames[i].height = m.height;
        frames[i].rowStride = fdtRowStride(m.matType, m.width);
        frames[i].matType = m.matType;
      }
      final out = _outputs(arena, n, mode);
      final int rc;
      if (orientations == null) {
        rc = _lib.detectFrames(_h, frames, n, mode.index, kFdtMemHost, out.faces, out.counts, out.mesh, out.iris);
      } else {
        final Pointer<Int32> ors = arena<Int32>(n);
        ors.asTypedList(n).setAll(0, orientations);
        rc = _lib.detectFramesOriented(_h, frames, ors, n, mode.index, kFdtMemHost, out.faces, out.counts, out.mesh, out.iris);
      }
      if (rc != FdtStatus.ok) {
        _lib.throwFor(rc, _h); // ArgumentError naming the first bad mat
      }
      return <List<Face>>[
        for (int b = 0; b < n; b++)
          (orientations != null && orientations[b] >= 5)
              ? _facesOf(out, b, mats[b].height, mats[b].width)
              : _facesOf(out, b, mats[b].width, mats[b].height),
      ];
    } finally {
      arena.releaseAll();
    }
  }

  /// Faces in YUV 4:2:0 frames given as three planes (`fdt_detect_yuv_planes`): an Android `YUV_420_888` CameraImage maps
  /// planes[0..2].bytes to [y], [u], [v], their bytesPerRow to the row strides and planes[1].bytesPerPixel (1 or 2) to
  /// [pixelStride]; the buffers may end at their last sample (pixelStride 2 leaves the last chroma row short).  The sample of
  /// pixel (x, y) is y[y * yStride + x], u[(y ~/ 2) * uStride + (x ~/ 2) * pixelStride], likewise v.  [orientations]: one
  /// EXIF orientation (kFdtOrient*) per frame, or null for all upright; each result list refers to its frame's upright image.
  Future<List<List<Face>>> detectFacesFromYuvPlanes(
    List<({Uint8List y, Uint8List u, Uint8List v, int yStride, int uStride, int vStride, int pixelStride, int width, int height})> frames, {
    FaceDetectionMode mode = FaceDetectionMode.full,
    List<int>? orientations,
  }) async {
    if (orientations != null) {
      if (orientations.length != frames.length) {
        throw ArgumentError('orientations: one EXIF orientation per frame (${frames.length})');
      }
      orientations.forEach(_checkOrientation);
    }
    _check();
    for (int i = 0; i < frames.length; i++) {
      final f = frames[i];
      if (f.width <= 0 || f.height <= 0 || f.width.isOdd || f.height.isOdd) {
        throw ArgumentError('frame $i: YUV 4:2:0 frames need an even, positive width and height');
      }
      if (f.pixelStride != 1 && f.pixelStride != 2) throw ArgumentError('frame $i: pixelStride must be 1 or 2');
      final int cols = (f.width ~/ 2 - 1) * f.pixelStride + 1;
      if (f.yStride < f.width || f.uStride < cols || f.vStride < cols) throw ArgumentError('frame $i: row stride too small');
      if (f.y.length < (f.height - 1) * f.yStride + f.width ||
          f.u.length < (f.height ~/ 2 - 1) * f.uStride + cols ||
          f.v.length < (f.height ~/ 2 - 1) * f.vStride + cols) {
        throw ArgumentError('frame $i: a plane is shorter than its sampled extent');
      }
    }
    final int n = frames.length;
    if (n == 0) return <List<Face>>[];
    final arena = Arena();
    try {
      final Pointer<FdtYuvPlanes> desc = arena<FdtYuvPlanes>(n);
      for (int i = 0; i < n; i++) {
        final f = frames[i];
        final planes = [f.y, f.u, f.v];
        final strides = [f.yStride, f.uStride, f.vStride];
        for (int k = 0; k < 3; k++) {
          final Pointer<Uint8> src = arena<Uint8>(planes[k].length);
          src.asTypedList(planes[k].length).setAll(0, planes[k]);
          desc[i].plane[k] = src;
          desc[i].rowStride[k] = strides[k];
        }
        desc[i].width = f.width;
        desc[i].height = f.height;
        desc[i].pixelStride = f.pixelStride;
        desc[i].reserved = 0;
      }
      final out = _outputs(arena, n, mode);
      Pointer<Int32> ors = nullptr;
      if (orientations != null) {
        ors = arena<Int32>(n);
        ors.asTypedList(n).setAll(0, orientations);
      }
      final int rc = _lib.detectYuvPlanes(_h, desc, ors, n, mode.index, kFdtMemHost, out.faces, out.counts, out.mesh, out.iris);
      if (rc != FdtStatus.ok) {
        _lib.throwFor(rc, _h); // ArgumentError naming the first bad frame and plane
      }
      return <List<Face>>[
        for (int b = 0; b < n; b++)
          (orientations != null && orientations[b] >= 5)
              ? _facesOf(out, b, frames[b].height, frames[b].width)
              : _facesOf(out, b, frames[b].width, frames[b].height),
      ];
    } finally {
      arena.releaseAll();
    }
  }

  /// detectFacesFromBytes over a list of encoded images (JPEG) in one `fdt_detect_jpeg_batch` call.  An image that cannot
  /// be decoded gives `null` in its place instead of throwing, so one bad photo does not discard the batch.
  Future<List<List<Face>?>> detectFacesFromBytesBatch(
    List<Uint8List> images, {
    FaceDetectionMode mode = FaceDetectionMode.full,
  }) async {
    _check();
    final int n = images.length;
    if (n == 0) return <List<Face>?>[];
    final arena = Arena();
    try {
      final Pointer<Pointer<Uint8>> ptrs = arena<Pointer<Uint8>>(n);
      final Pointer<Size> sizes = arena<Size>(n);
      for (int i = 0; i < n; i++) {
        final Pointer<Uint8> src = arena<Uint8>(images[i].length + 1);
        src.asTypedList(images[i].length).setAll(0, images[i]);
        ptrs[i] = src;
        sizes[i] = images[i].length;
      }
      final Pointer<Int32> wh = arena<Int32>(2 * n);
      final Pointer<Int32> status = arena<Int32>(n);
      final out = _outputs(arena, n, mode);
      final int rc = _lib.detectJpegBatch(_h, ptrs, sizes, n, mode.index, out.faces, out.counts, out.mesh, out.iris, wh, status);
      if (rc != FdtStatus.ok) {
        _lib.throwFor(rc, _h);
      }
      return <List<Face>?>[
        for (int b = 0; b < n; b++) status[b] == FdtStatus.ok ? _facesOf(out, b, wh[2 * b], wh[2 * b + 1]) : null,
      ];
    } finally {
      arena.releaseAll();
    }
  }

  ({Pointer<FdtFace> faces, Pointer<Int32> counts, Pointer<Float> mesh, Pointer<Float> iris}) _outputs(
      Arena arena, int n, FaceDetectionMode mode) {
    final bool wantMesh = mode != FaceDetectionMode.fast;
    final bool wantIris = mode == FaceDetectionMode.full;
    return (
      faces: arena<FdtFace>(n * _maxFaces),
      counts: arena<Int32>(n),
      mesh: wantMesh ? arena<Float>(n * _maxFaces * kFdtMeshFloats) : nullptr,
      iris: wantIris ? arena<Float>(n * _maxFaces * kFdtIrisFloats) : nullptr,
    );
  }

  List<Face> _facesOf(({Pointer<FdtFace> faces, Pointer<Int32> counts, Pointer<Float> mesh, Pointer<Float> iris}) out, int b,
      int width, int height) {
    return <Face>[
      for (int j = 0; j < out.counts[b]; j++)
        _toFace(out.faces[b * _maxFaces + j], out.mesh, out.iris, b * _maxFaces + j, width, height),
    ];
  }

  /// The aligned crop getFaceEmbeddingFromEyesDirect feeds the embedding model (face_detector_core.dart:419-452):
  /// computeEmbeddingAlignment on the (iris-refined) eye landmarks, then extractAlignedSquare(..., -theta, outSize).
  /// Returns `outSize * outSize * 3` BGR bytes.
  Future<Uint8List> embeddingCrop(Face face, Uint8List bytes,
      {required int width, required int height, int matType = 16, int outSize = 112}) async {
    _check();
    final Point? l = face.landmarks.leftEye;
    final Point? r = face.landmarks.rightEye;
    if (l == null || r == null) {
      throw StateError('Face must have left and right eye landmarks');
    }
    final arena = Arena();
    try {
      final Pointer<Double> le = arena<Double>(2), re = arena<Double>(2), roi = arena<Double>(4);
      le[0] = l.x;
      le[1] = l.y;
      re[0] = r.x;
      re[1] = r.y;
      _lib.hostEmbeddingRoi(le, re, roi); // theta, cx, cy, size
      final Pointer<Double> rois = arena<Double>(4);
      rois[0] = roi[1];
      rois[1] = roi[2];
      rois[2] = roi[3];
      rois[3] = -roi[0];
      final Pointer<Uint8> src = arena<Uint8>(bytes.length);
      src.asTypedList(bytes.length).setAll(0, bytes);
      final int channels = matType == 0 ? 1 : (matType == 24 ? 4 : 3);
      final Pointer<Uint8> crop = arena<Uint8>(outSize * outSize * 3);
      final Pointer<Int32> ok = arena<Int32>();
      final int rc =
          _lib.extractAlignedSquares(_h, src, width, height, width * channels, matType, rois, 1, outSize, crop, ok);
      if (rc != FdtStatus.ok) {
        _lib.throwFor(rc, _h);
      }
      if (ok.value == 0) {
        throw StateError('Failed to extract aligned face crop for embedding');
      }
      return Uint8List.fromList(crop.asTypedList(outSize * outSize * 3));
    } finally {
      arena.releaseAll();
    }
  }

  /// FaceDetector.dispose (face_detector.dart:1061-1081).
  Future<void> dispose() async {
    if (_h != nullptr) {
      _lib.destroy(_h);
      _h = nullptr;
    }
  }

  static Face _toFace(FdtFace f, Pointer<Float> mesh, Pointer<Float> iris, int slot, int w, int h) {
    final Size size = Size(w.toDouble(), h.toDouble());
    FaceMesh? fm;
    if (mesh != nullptr && f.hasMesh != 0) {
      final Float32List packed =
          Float32List.fromList((mesh + slot * kFdtMeshFloats).asTypedList(kFdtMeshFloats));
      fm = FaceMesh.packed(packed, score: f.meshScore); // face_types.dart:773-809
    }
    List<Point> irises = const <Point>[];
    if (iris != nullptr && f.hasIris != 0) {
      final Float32List buf = (iris + slot * kFdtIrisFloats).asTypedList(kFdtIrisFloats);
      irises = <Point>[for (int i = 0; i < kFdtIrisFloats ~/ 3; i++) Point(buf[3 * i], buf[3 * i + 1], buf[3 * i + 2])];
    }
    return Face(
      detection: Detection(
        boundingBox: RectF(f.xmin, f.ymin, f.xmax, f.ymax),
        score: f.score,
        keypointsXY: <double>[for (int k = 0; k < 12; k++) f.keypoints[k]],
        imageSize: size,
      ),
      mesh: fm,
      irises: irises,
      originalSize: size,
    );
  }
}

/// Frames in pinned host memory (fdt_alloc_pinned): write decoded camera frames here and pass the buffer to
/// [FdtFaceDetector.detectFacesPinned].  Portable across the devices of a multi-device handle.
class FdtPinnedFrames {
  FdtPinnedFrames._(this.pointer, this.lengthInBytes);

  final Pointer<Uint8> pointer;
  final int lengthInBytes;

  static FdtPinnedFrames allocate(int lengthInBytes) {
    final Pointer<Pointer<Void>> out = calloc<Pointer<Void>>();
    try {
      final int rc = FdtLibrary.instance.allocPinned(lengthInBytes, out);
      if (rc != FdtStatus.ok) {
        throw Exception('fdt_alloc_pinned failed ($rc)');
      }
      return FdtPinnedFrames._(out.value.cast<Uint8>(), lengthInBytes);
    } finally {
      calloc.free(out);
    }
  }

  Uint8List get bytes => pointer.asTypedList(lengthInBytes);

  void free() => FdtLibrary.instance.freePinned(pointer.cast<Void>());
}
