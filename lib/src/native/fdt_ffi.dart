/// dart:ffi binding of libfdt_cuda.so (C ABI: include/fdt_api.h), the B200 implementation of the detection hot path.
///
/// Drop-in location: `lib/src/native/fdt_ffi.dart` of the face_detection_tflite package.  It replaces, for this path,
/// the FFI calls the package makes into flutter_litert (`Interpreter.invoke`, `generateAnchors`, `weightedNms`,
/// `computeLetterboxParams`) and opencv_dart (`cv.resize`, `cv.copyMakeBorder`, `cv.cvtColor`, `convertTo`,
/// `cv.getRotationMatrix2D`, `cv.warpAffine`, `cv.flip`).  No Dart toolchain exists in the build image of this
/// repository: the file is written against the ABI and exercised through the same entry points by tests/ (ctypes).
library;

import 'dart:ffi';
import 'dart:io' show Platform;

import 'package:ffi/ffi.dart';

/// fdt_status (include/fdt_api.h).
abstract final class FdtStatus {
  static const int ok = 0;
  static const int notReady = 1; // StateError
  static const int badArg = 2; // ArgumentError
  static const int sizeMismatch = 3; // ArgumentError (helpers.dart:440-447)
  static const int model = 4;
  static const int cuda = 5;
  static const int unsupported = 6;
  static const int format = 7; // FormatException (undecodable image bytes, face_detector.dart:476)
}

const int kFdtMaxFaces = 100; // weightedNms maxDet (helpers.dart:187)
const int kFdtMeshFloats = 1404;
const int kFdtIrisFloats = 456;
const int kFdtMemHost = 0;
const int kFdtMemDevice = 1;
/// YUV 4:2:0 frame formats (fdt_api.h FDT_FMT_YUV_*), accepted wherever a matType is, except by extractAlignedSquares.
/// A frame is height * rowStride * 3 / 2 bytes: the Y plane, then NV12 / NV21 interleaved chroma (same row stride) or the
/// I420 U and V planes (rowStride / 2 per row).  width and height must be even.
const int kFdtFmtYuvNv12 = 0x1000;
const int kFdtFmtYuvNv21 = 0x1001;
const int kFdtFmtYuvI420 = 0x1002;
/// RGB-ordered frame formats (fdt_api.h FDT_FMT_RGB*), accepted wherever a matType is, except by extractAlignedSquares;
/// results equal those of the BGR image bit for bit.  kFdtFmtRgb: packed R, G, B; kFdtFmtRgba: packed R, G, B, A (alpha
/// ignored) - `ui.Image.toByteData(format: ImageByteFormat.rawRgba)` goes in as it is, width * 4 bytes per row, no conversion;
/// kFdtFmtRgbPlanar: an R, a G and a B plane of height rows of rowStride (>= width) bytes each, back to back.
const int kFdtFmtRgb = 0x1010;
const int kFdtFmtRgba = 0x1011;
const int kFdtFmtRgbPlanar = 0x1012;

/// Frame orientations (fdt_api.h FDT_ORIENT_*): the EXIF Orientation value of a stored frame, as OpenCV's ExifTransform
/// applies it.  Results of the oriented calls refer to the upright image; for 5-8 its width is the stored height.  Camera
/// frames that must be rotated R degrees clockwise to display: 1, 6, 3, 8 for R = 0, 90, 180, 270; rotated R degrees clockwise
/// and then mirrored left-right: 2, 5, 4, 7.
const int kFdtOrientUpright = 1;
const int kFdtOrientMirrorH = 2;
const int kFdtOrientRot180 = 3;
const int kFdtOrientMirrorV = 4;
const int kFdtOrientTranspose = 5;
const int kFdtOrientRot90Cw = 6;
const int kFdtOrientTransverse = 7;
const int kFdtOrientRot90Ccw = 8;

bool fdtIsYuv(int matType) => matType == kFdtFmtYuvNv12 || matType == kFdtFmtYuvNv21 || matType == kFdtFmtYuvI420;

/// Row stride (Y-plane stride for the YUV formats, one plane's for planar RGB) and size in bytes of one tightly packed frame
/// of [matType].
int fdtRowStride(int matType, int width) => fdtIsYuv(matType) || matType == kFdtFmtRgbPlanar
    ? width
    : width * (matType == 0 ? 1 : (matType == 24 || matType == kFdtFmtRgba ? 4 : 3));
int fdtFrameBytes(int matType, int width, int height) => fdtIsYuv(matType)
    ? height * width * 3 ~/ 2
    : (matType == kFdtFmtRgbPlanar ? 3 : 1) * height * fdtRowStride(matType, width);

/// fdt_config: the named arguments of FaceDetector.create that touch the path (48 bytes).
final class FdtConfig extends Struct {
  @Int32()
  external int structSize;
  @Int32()
  external int model; // FaceDetectionModel.index
  @Int32()
  external int device;
  @Int32()
  external int maxBatch;
  @Int32()
  external int maxFaces;
  @Int32()
  external int fuseLevel;
  @Double()
  external double minScore;
  @Double()
  external double minFaceSize;
  @Double()
  external double minFacePresence;
}

/// fdt_face: one face in the wire layout of _faceToFastMap (face_detector.dart:1160-1181); 160 bytes.
final class FdtFace extends Struct {
  @Double()
  external double xmin;
  @Double()
  external double ymin;
  @Double()
  external double xmax;
  @Double()
  external double ymax;
  @Double()
  external double score;
  @Array(12)
  external Array<Double> keypoints;
  @Double()
  external double meshScore;
  @Int32()
  external int hasMesh;
  @Int32()
  external int anchorIndex;
  @Int32()
  external int hasIris;
  @Int32()
  external int reserved;
}

/// fdt_frame: one frame of a mixed batch (fdt_detect_frames); 24 bytes.
final class FdtFrame extends Struct {
  external Pointer<Uint8> data;
  @Int32()
  external int width;
  @Int32()
  external int height;
  @Int32()
  external int rowStride;
  @Int32()
  external int matType;
}

/// fdt_yuv_planes: one YUV 4:2:0 frame as a Y, a U and a V plane with their own base and row stride, U and V sharing a pixel
/// stride of 1 or 2 (fdt_detect_yuv_planes; an Android `YUV_420_888` CameraImage's three planes); 56 bytes.
final class FdtYuvPlanes extends Struct {
  @Array(3)
  external Array<Pointer<Uint8>> plane;
  @Array(3)
  external Array<Int32> rowStride;
  @Int32()
  external int width;
  @Int32()
  external int height;
  @Int32()
  external int pixelStride;
  @Int32()
  external int reserved;
}

typedef _DefaultConfigC = Void Function(Pointer<FdtConfig>);
typedef _DefaultConfigD = void Function(Pointer<FdtConfig>);
typedef _CreateExC = Int32 Function(Pointer<FdtConfig>, Pointer<Uint8>, Size, Pointer<Uint8>, Size, Pointer<Uint8>, Size,
    Pointer<Int32>, Int32, Pointer<Pointer<Void>>);
typedef _CreateExD = int Function(Pointer<FdtConfig>, Pointer<Uint8>, int, Pointer<Uint8>, int, Pointer<Uint8>, int,
    Pointer<Int32>, int, Pointer<Pointer<Void>>);
typedef _DestroyC = Int32 Function(Pointer<Void>);
typedef _DestroyD = int Function(Pointer<Void>);
typedef _DetectOneC = Int32 Function(Pointer<Void>, Pointer<Uint8>, Size, Int32, Int32, Int32, Int32, Pointer<FdtFace>,
    Pointer<Int32>, Pointer<Float>, Pointer<Float>);
typedef _DetectOneD = int Function(Pointer<Void>, Pointer<Uint8>, int, int, int, int, int, Pointer<FdtFace>,
    Pointer<Int32>, Pointer<Float>, Pointer<Float>);
typedef _DetectBatchC = Int32 Function(Pointer<Void>, Pointer<Uint8>, Int32, Int32, Int32, Int32, Int32, Int32, Int32,
    Pointer<FdtFace>, Pointer<Int32>, Pointer<Float>, Pointer<Float>);
typedef _DetectBatchD = int Function(Pointer<Void>, Pointer<Uint8>, int, int, int, int, int, int, int,
    Pointer<FdtFace>, Pointer<Int32>, Pointer<Float>, Pointer<Float>);
typedef _LastErrorC = Pointer<Utf8> Function(Pointer<Void>);
typedef _AllocPinnedC = Int32 Function(Size, Pointer<Pointer<Void>>);
typedef _AllocPinnedD = int Function(int, Pointer<Pointer<Void>>);
typedef _FreePinnedC = Int32 Function(Pointer<Void>);
typedef _FreePinnedD = int Function(Pointer<Void>);
typedef _GetInfoC = Int32 Function(Pointer<Void>, Pointer<Int32>, Pointer<Int32>, Pointer<Int32>, Pointer<Int32>, Pointer<Int32>);
typedef _GetInfoD = int Function(Pointer<Void>, Pointer<Int32>, Pointer<Int32>, Pointer<Int32>, Pointer<Int32>, Pointer<Int32>);
typedef _ExtractSquaresC = Int32 Function(Pointer<Void>, Pointer<Uint8>, Int32, Int32, Int32, Int32, Pointer<Double>, Int32,
    Int32, Pointer<Uint8>, Pointer<Int32>);
typedef _ExtractSquaresD = int Function(Pointer<Void>, Pointer<Uint8>, int, int, int, int, Pointer<Double>, int, int,
    Pointer<Uint8>, Pointer<Int32>);
typedef _EmbeddingRoiC = Int32 Function(Pointer<Double>, Pointer<Double>, Pointer<Double>);
typedef _EmbeddingRoiD = int Function(Pointer<Double>, Pointer<Double>, Pointer<Double>);
typedef _DetectJpegC = Int32 Function(Pointer<Void>, Pointer<Uint8>, Size, Int32, Pointer<FdtFace>, Pointer<Int32>,
    Pointer<Float>, Pointer<Float>, Pointer<Int32>);
typedef _DetectJpegD = int Function(Pointer<Void>, Pointer<Uint8>, int, int, Pointer<FdtFace>, Pointer<Int32>,
    Pointer<Float>, Pointer<Float>, Pointer<Int32>);
typedef _DetectFramesC = Int32 Function(Pointer<Void>, Pointer<FdtFrame>, Int32, Int32, Int32, Pointer<FdtFace>, Pointer<Int32>,
    Pointer<Float>, Pointer<Float>);
typedef _DetectFramesD = int Function(Pointer<Void>, Pointer<FdtFrame>, int, int, int, Pointer<FdtFace>, Pointer<Int32>,
    Pointer<Float>, Pointer<Float>);
typedef _DetectBatchOrientedC = Int32 Function(Pointer<Void>, Pointer<Uint8>, Int32, Int32, Int32, Int32, Int32, Int32, Int32,
    Int32, Pointer<FdtFace>, Pointer<Int32>, Pointer<Float>, Pointer<Float>);
typedef _DetectBatchOrientedD = int Function(Pointer<Void>, Pointer<Uint8>, int, int, int, int, int, int, int, int,
    Pointer<FdtFace>, Pointer<Int32>, Pointer<Float>, Pointer<Float>);
typedef _DetectFramesOrientedC = Int32 Function(Pointer<Void>, Pointer<FdtFrame>, Pointer<Int32>, Int32, Int32, Int32,
    Pointer<FdtFace>, Pointer<Int32>, Pointer<Float>, Pointer<Float>);
typedef _DetectFramesOrientedD = int Function(Pointer<Void>, Pointer<FdtFrame>, Pointer<Int32>, int, int, int, Pointer<FdtFace>,
    Pointer<Int32>, Pointer<Float>, Pointer<Float>);
typedef _DetectJpegBatchC = Int32 Function(Pointer<Void>, Pointer<Pointer<Uint8>>, Pointer<Size>, Int32, Int32, Pointer<FdtFace>,
    Pointer<Int32>, Pointer<Float>, Pointer<Float>, Pointer<Int32>, Pointer<Int32>);
typedef _DetectJpegBatchD = int Function(Pointer<Void>, Pointer<Pointer<Uint8>>, Pointer<Size>, int, int, Pointer<FdtFace>,
    Pointer<Int32>, Pointer<Float>, Pointer<Float>, Pointer<Int32>, Pointer<Int32>);
typedef _DetectYuvPlanesC = Int32 Function(Pointer<Void>, Pointer<FdtYuvPlanes>, Pointer<Int32>, Int32, Int32, Int32,
    Pointer<FdtFace>, Pointer<Int32>, Pointer<Float>, Pointer<Float>);
typedef _DetectYuvPlanesD = int Function(Pointer<Void>, Pointer<FdtYuvPlanes>, Pointer<Int32>, int, int, int, Pointer<FdtFace>,
    Pointer<Int32>, Pointer<Float>, Pointer<Float>);
typedef _NumDevicesC = Int32 Function(Pointer<Void>);
typedef _NumDevicesD = int Function(Pointer<Void>);

/// The loaded library and its entry points.  One instance per process (DynamicLibrary.open caches the handle).
class FdtLibrary {
  FdtLibrary._(this._lib)
      : defaultConfig = _lib.lookupFunction<_DefaultConfigC, _DefaultConfigD>('fdt_default_config'),
        createEx = _lib.lookupFunction<_CreateExC, _CreateExD>('fdt_create_ex'),
        destroy = _lib.lookupFunction<_DestroyC, _DestroyD>('fdt_destroy'),
        detectOne = _lib.lookupFunction<_DetectOneC, _DetectOneD>('fdt_detect_one'),
        detectBatch = _lib.lookupFunction<_DetectBatchC, _DetectBatchD>('fdt_detect_batch'),
        lastError = _lib.lookupFunction<_LastErrorC, _LastErrorC>('fdt_last_error'),
        allocPinned = _lib.lookupFunction<_AllocPinnedC, _AllocPinnedD>('fdt_alloc_pinned'),
        freePinned = _lib.lookupFunction<_FreePinnedC, _FreePinnedD>('fdt_free_pinned'),
        getInfo = _lib.lookupFunction<_GetInfoC, _GetInfoD>('fdt_get_info'),
        extractAlignedSquares = _lib.lookupFunction<_ExtractSquaresC, _ExtractSquaresD>('fdt_extract_aligned_squares'),
        hostEmbeddingRoi = _lib.lookupFunction<_EmbeddingRoiC, _EmbeddingRoiD>('fdt_host_embedding_roi'),
        detectJpeg = _lib.lookupFunction<_DetectJpegC, _DetectJpegD>('fdt_detect_jpeg'),
        detectFrames = _lib.lookupFunction<_DetectFramesC, _DetectFramesD>('fdt_detect_frames'),
        detectBatchOriented = _lib.lookupFunction<_DetectBatchOrientedC, _DetectBatchOrientedD>('fdt_detect_batch_oriented'),
        detectFramesOriented = _lib.lookupFunction<_DetectFramesOrientedC, _DetectFramesOrientedD>('fdt_detect_frames_oriented'),
        detectJpegBatch = _lib.lookupFunction<_DetectJpegBatchC, _DetectJpegBatchD>('fdt_detect_jpeg_batch'),
        detectYuvPlanes = _lib.lookupFunction<_DetectYuvPlanesC, _DetectYuvPlanesD>('fdt_detect_yuv_planes'),
        numDevices = _lib.lookupFunction<_NumDevicesC, _NumDevicesD>('fdt_num_devices');

  final DynamicLibrary _lib;
  final _DefaultConfigD defaultConfig;
  final _CreateExD createEx;
  final _DestroyD destroy;
  final _DetectOneD detectOne;
  final _DetectBatchD detectBatch;
  final _LastErrorC lastError;
  final _AllocPinnedD allocPinned;
  final _FreePinnedD freePinned;
  final _GetInfoD getInfo;
  final _ExtractSquaresD extractAlignedSquares;
  final _EmbeddingRoiD hostEmbeddingRoi;
  final _DetectJpegD detectJpeg;
  final _DetectFramesD detectFrames;
  final _DetectBatchOrientedD detectBatchOriented;
  final _DetectFramesOrientedD detectFramesOriented;
  final _DetectJpegBatchD detectJpegBatch;
  final _DetectYuvPlanesD detectYuvPlanes;
  final _NumDevicesD numDevices;

  static FdtLibrary? _instance;

  /// Opens libfdt_cuda.so from the plugin bundle (linux/CMakeLists.txt bundles it next to the executable's lib/).
  static FdtLibrary get instance {
    if (!Platform.isLinux) {
      throw UnsupportedError('libfdt_cuda.so is a Linux / CUDA (sm_100a) library; there is no CPU fallback');
    }
    return _instance ??= FdtLibrary._(DynamicLibrary.open('libfdt_cuda.so'));
  }

  /// Maps an fdt_status to the exception the reference throws at the same place.
  Never throwFor(int rc, Pointer<Void> handle) {
    final Pointer<Utf8> p = lastError(handle);
    final String msg = p == nullptr ? 'fdt error $rc' : p.toDartString();
    switch (rc) {
      case FdtStatus.notReady:
        throw StateError(msg); // face_detector.dart:1083-1089
      case FdtStatus.badArg:
      case FdtStatus.sizeMismatch:
        throw ArgumentError(msg); // face_gates.dart:31-59, helpers.dart:440-447
      case FdtStatus.format:
        throw FormatException(msg); // undecodable image bytes, face_detector.dart:476
      case FdtStatus.unsupported:
        throw UnsupportedError(msg);
      default:
        throw Exception(msg);
    }
  }
}
