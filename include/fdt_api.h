/*
 * fdt_api.h — C ABI of libfdt_cuda.so, the B200 (sm_100a) implementation of the
 * face_detection_tflite detection hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference has no native compute
 * of its own: its Dart code reaches TFLite/XNNPACK and OpenCV through dart:ffi inside the
 * un-vendored packages flutter_litert 3.8.0 and opencv_dart 2.2.1+4.  The entry points below
 * are what a dart:ffi binding for this path binds instead; each one cites the reference
 * interface it replaces (paths relative to the reference repository root).
 *
 * Conventions: every function returns an fdt_status (0 = ok) and never aborts; the caller owns
 * all input and output buffers; the handle owns weights, workspaces, streams.  A handle
 * serialises its own calls internally (reference: one _detectorLock per detector,
 * lib/src/isolate/face_detector_core.dart:105,:465); different handles are independent.
 * There is no CPU fallback: without a CUDA device fdt_create fails with FDT_ERR_CUDA.
 */
#ifndef FDT_API_H_
#define FDT_API_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define FDT_EXPORT __declspec(dllexport)
#else
#define FDT_EXPORT __attribute__((visibility("default")))
#endif

typedef struct fdt_handle fdt_handle;

/* Status codes.  Mapping to the reference's exceptions (SURVEY.md 8b "Errors"):
 *   FDT_ERR_NOT_READY     <- StateError (not initialised / disposed, lib/src/face_detector.dart:1083-1089)
 *   FDT_ERR_BAD_ARG       <- ArgumentError (gates outside [0,1], lib/src/shared/face_gates.dart:31-59)
 *   FDT_ERR_SIZE_MISMATCH <- ArgumentError (byte length mismatch, lib/src/util/helpers.dart:440-447)
 *   FDT_ERR_MODEL         <- model buffer rejected (Interpreter.fromBuffer failure)
 *   FDT_ERR_CUDA          <- device / driver failure (no reference equivalent)
 *   FDT_ERR_FORMAT        <- FormatException (undecodable image bytes, lib/src/face_detector.dart:476)     */
typedef enum fdt_status {
  FDT_OK = 0,
  FDT_ERR_NOT_READY = 1,
  FDT_ERR_BAD_ARG = 2,
  FDT_ERR_SIZE_MISMATCH = 3,
  FDT_ERR_MODEL = 4,
  FDT_ERR_CUDA = 5,
  FDT_ERR_UNSUPPORTED = 6,
  FDT_ERR_FORMAT = 7
} fdt_status;

/* FaceDetectionModel (lib/src/shared/face_types.dart:100-115) -> SSD anchor option set
 * (ssdOptionsFor, lib/src/shared/face_model_config.dart:128-134). */
typedef enum fdt_model {
  FDT_MODEL_FRONT_CAMERA = 0, /* 128x128, strides 8,16,16,16 -> 896 anchors  */
  FDT_MODEL_BACK_CAMERA = 1,  /* 256x256, strides 16,32,32,32 -> 896 anchors */
  FDT_MODEL_SHORT_RANGE = 2,  /* = front                                      */
  FDT_MODEL_FULL = 3,         /* 192x192, stride 4 -> 2304 anchors            */
  FDT_MODEL_FULL_SPARSE = 4   /* rejected: FDT_ERR_UNSUPPORTED                */
} fdt_model;

/* FaceDetectionMode (lib/src/shared/face_types.dart:118-127). */
typedef enum fdt_mode {
  FDT_MODE_FAST = 0,     /* detector + 6 keypoints                            */
  FDT_MODE_STANDARD = 1, /* + aligned crop + 468-point mesh                   */
  FDT_MODE_FULL = 2      /* + two eye crops + iris_landmark: 152 iris/eye-contour points, iris-refined eye keypoints
                            (the reference's default mode; its blendshape classifier is outside this path)      */
} fdt_mode;

/* cv MatType values accepted by detectFacesFromMatBytes (lib/src/face_detector.dart:588-594;
 * colour conversion rule lib/src/util/helpers.dart:386-392). */
enum { FDT_MAT_8UC1 = 0, FDT_MAT_8UC3 = 16, FDT_MAT_8UC4 = 24 };

/* YUV 4:2:0 frames (camera frames, hardware video decoders), accepted wherever mat_type is, except by
 * fdt_extract_aligned_squares.  The result equals cv::cvtColor(frame, COLOR_YUV2BGR_NV12 / _NV21 / _I420) followed
 * by the BGR path; the conversion is fused into the letterbox and crop kernels (no host pass).
 * width and height are the image size and must both be even (else FDT_ERR_BAD_ARG); row_stride is the Y-plane
 * stride in bytes, >= width (else FDT_ERR_SIZE_MISMATCH).  One frame is height * row_stride * 3 / 2 bytes:
 *   NV12 / NV21: Y plane, then the interleaved chroma plane (U,V / V,U) at height * row_stride, same row stride;
 *   I420: Y plane, then the U plane at height * row_stride with row stride row_stride / 2 (row_stride must be even,
 *         else FDT_ERR_BAD_ARG), then the V plane.
 * With row_stride == width this is cv2's (3H/2) x W single-channel Mat.  The values cannot collide with a cv
 * MatType (at most 4095). */
enum { FDT_FMT_YUV_NV12 = 0x1000, FDT_FMT_YUV_NV21 = 0x1001, FDT_FMT_YUV_I420 = 0x1002 };

/* RGB-ordered frames (PIL, PyAV rgb24, imageio, Flutter rawRgba, browser ImageData, and torchvision / torchcodec GPU decoding,
 * which hands over uint8 [3, H, W] tensors), accepted wherever mat_type is, except by fdt_extract_aligned_squares
 * (FDT_ERR_BAD_ARG).  Every result equals the same call on the BGR image - cv::cvtColor(frame, COLOR_RGB2BGR) / COLOR_RGBA2BGR,
 * or for planar frames the planes in reverse order interleaved (numpy: chw[::-1].transpose(1, 2, 0)) - bit for bit; the channel
 * order and plane layout are read by the letterbox and crop kernels (no converted copy).
 *   FDT_FMT_RGB        packed R, G, B; row_stride >= 3 * width; a frame is height * row_stride bytes.
 *   FDT_FMT_RGBA       packed R, G, B, A (alpha ignored, as for 8UC4); row_stride >= 4 * width; height * row_stride bytes.
 *   FDT_FMT_RGB_PLANAR an R plane, then a G plane, then a B plane, back to back, each height rows of row_stride >= width bytes;
 *                      a frame is 3 * height * row_stride bytes (a contiguous [3, H, W] tensor has row_stride = W).  Any size.
 * A row_stride below the minimum returns FDT_ERR_SIZE_MISMATCH. */
enum { FDT_FMT_RGB = 0x1010, FDT_FMT_RGBA = 0x1011, FDT_FMT_RGB_PLANAR = 0x1012 };

/* Packed YUV 4:2:2 frames (USB / UVC webcams through V4L2: YUYV; SDI / HDMI capture cards, DeckLink 2vuy: UYVY; GStreamer
 * YUY2 / UYVY / YVYU caps), accepted wherever mat_type is, except by fdt_extract_aligned_squares (FDT_ERR_BAD_ARG).  Every
 * result equals the same call on cv::cvtColor(frame, COLOR_YUV2BGR_YUYV / _UYVY / _YVYU) as a BGR frame, bit for bit (BT.601
 * limited range, as the YUV 4:2:0 formats); the conversion is fused into the letterbox and crop kernels (no converted copy).
 * Pixel (x, y) lies in row frame + y * row_stride, in the 4-byte macropixel at byte 4 * (x / 2), which two pixels share:
 *   FDT_FMT_YUYV (= YUY2)  Y0 U Y1 V   Y of pixel x at byte 2x,     U at 4 * (x / 2) + 1, V at 4 * (x / 2) + 3
 *   FDT_FMT_UYVY           U Y0 V Y1   Y of pixel x at byte 2x + 1, U at 4 * (x / 2),     V at 4 * (x / 2) + 2
 *   FDT_FMT_YVYU           Y0 V Y1 U   Y of pixel x at byte 2x,     U at 4 * (x / 2) + 3, V at 4 * (x / 2) + 1
 * width must be even (else FDT_ERR_BAD_ARG; for orientations 5-8 the stored width); height may be any positive value.
 * row_stride >= 2 * width (else FDT_ERR_SIZE_MISMATCH), odd strides included; a frame is height * row_stride bytes (cv2's
 * H x W CV_8UC2 Mat when row_stride = 2 * width). */
enum { FDT_FMT_YUYV = 0x1020, FDT_FMT_UYVY = 0x1021, FDT_FMT_YVYU = 0x1022 };

/* High-bit-depth YUV 4:2:0 (HEVC Main10, AV1 / VP9 profile 2 and 10-bit capture: NVDEC P016 surfaces, Windows DXGI / Media
 * Foundation P010, FFmpeg hwdownload).  Semi-planar 4:2:0 of little-endian 16-bit words with the value in the high bits; the one
 * constant serves P010, P012 and P016.  Accepted wherever mat_type is, except by fdt_extract_aligned_squares (FDT_ERR_BAD_ARG).
 *   Y plane: height rows of row_stride bytes, the Y word of pixel (x, y) at byte y * row_stride + 2x.
 *   UV plane at height * row_stride: height / 2 rows of row_stride bytes; U of pixel (x, y) is the word at byte
 *   (y / 2) * row_stride + 4 * (x / 2) of that plane, V the word 2 bytes behind it.
 *   A frame is height * row_stride * 3 / 2 bytes (with row_stride = 2 * width, cv2's (3H/2) x W CV_16UC1 Mat).
 * width, height and row_stride must be even (else FDT_ERR_BAD_ARG; for orientations 5-8, the stored size); row_stride >=
 * 2 * width (else FDT_ERR_SIZE_MISMATCH).
 * The sample rule, here and in fdt_detect_yuv_planes16: a 16-bit sample s with `bits` significant bits stored from bit 0 becomes
 * the 8-bit sample (s >> (bits - 8)) & 0xFF; high-bit-aligned data (P010 / P012 / P016) is bits = 16, its high byte.  It
 * truncates (what a caller's `>> 8` to uint8 computes, and P010 and P016 of one picture give one answer); the bits below the 8
 * it keeps never affect a result, and bits above `bits` are ignored.  Every result (records, mesh, iris, the letterbox tap, the
 * mesh / iris stage crops, face crops) equals, bit for bit, the same call on the 8-bit FDT_FMT_YUV_NV12 frame made by that rule,
 * in every orientation, memory kind and mode.  Colour is then the NV12 path's BT.601 limited-range conversion: a detector input,
 * not an HDR-correct one; BT.2020 primaries and PQ / HLG transfer functions are not applied. */
enum { FDT_FMT_P010 = 0x1003 };

enum { FDT_MEM_HOST = 0, FDT_MEM_DEVICE = 1 };

/* Frame orientation (fdt_detect_batch_oriented, fdt_detect_frames_oriented): the EXIF Orientation value of the STORED frame,
 * meaning what OpenCV's ExifTransform and fdt_detect_jpeg apply.  The upright image U is the stored frame transformed:
 *   1 as stored              2 mirrored left-right      3 rotated 180 degrees              4 mirrored top-bottom
 *   5 transposed (U[r][c] = stored[c][r])              6 rotated 90 degrees clockwise
 *   7 transverse (U[r][c] = stored[H-1-c][W-1-r])      8 rotated 90 degrees counter-clockwise
 * For orientations 5-8 U's width is the stored height.
 * Camera callers: a frame that must be rotated R degrees clockwise to display upright (Android's rotationDegrees, a video
 * stream's display rotation) has orientation 1, 6, 3, 8 for R = 0, 90, 180, 270.  A frame that must be rotated R degrees
 * clockwise and THEN mirrored left-right (a front camera preview) has 2, 5, 4, 7 for R = 0, 90, 180, 270. */
enum {
  FDT_ORIENT_UPRIGHT = 1, FDT_ORIENT_MIRROR_H = 2, FDT_ORIENT_ROT180 = 3, FDT_ORIENT_MIRROR_V = 4,
  FDT_ORIENT_TRANSPOSE = 5, FDT_ORIENT_ROT90_CW = 6, FDT_ORIENT_TRANSVERSE = 7, FDT_ORIENT_ROT90_CCW = 8
};

enum { FDT_MAX_FACES = 100 };      /* weightedNms maxDet, lib/src/util/helpers.dart:187 */
enum { FDT_MESH_POINTS = 468, FDT_MESH_FLOATS = 1404 };
enum { FDT_IRIS_POINTS = 152, FDT_IRIS_FLOATS = 456 }; /* 76 per eye: 71 contour + 5 iris (face_detector.dart:1888-1893) */

/* Named arguments of FaceDetector.create (lib/src/face_detector.dart:84-101) that touch the path. */
typedef struct fdt_config {
  int32_t struct_size;       /* sizeof(fdt_config), for forward compatibility               */
  int32_t model;             /* fdt_model                                                    */
  int32_t device;            /* CUDA device ordinal                                          */
  int32_t max_batch;         /* frames per internal chunk (0 = default 256)                  */
  int32_t max_faces;         /* result slots per frame (0 = FDT_MAX_FACES)                   */
  int32_t fuse_level;        /* 0 = one kernel per TFLite op (debug / parity taps),
                                1 = fused BlazeBlock kernels (default when < 0)              */
  double min_score;          /* gates, lib/src/shared/face_gates.dart:130-146; default 0     */
  double min_face_size;      /* default 0                                                    */
  double min_face_presence;  /* mesh face-flag gate, default 0.5 (face_model_config.dart:62) */
} fdt_config;

/* One detected face in the wire layout of _faceToFastMap (lib/src/face_detector.dart:1160-1181):
 * RectF + score + 6 keypoints, all normalised to the ORIGINAL frame (after letterbox removal,
 * lib/src/util/helpers.dart:101-136), float64 like Dart doubles. */
typedef struct fdt_face {
  double xmin, ymin, xmax, ymax;
  double score;
  double keypoints[12];      /* leftEye, rightEye, noseTip, mouth, leftTragion, rightTragion (x,y) */
  double mesh_score;         /* sigmoid(face flag); NaN when no mesh was computed            */
  int32_t has_mesh;
  int32_t anchor_index;      /* anchor of the top detection of the NMS cluster (parity aid)  */
  int32_t has_iris;          /* 1: iris points were computed and the eye keypoints are iris-refined
                                (face_detector_core.dart:356-373)                             */
  int32_t reserved;
} fdt_face;

FDT_EXPORT void fdt_default_config(fdt_config* cfg);

/* FaceDetector.create / initialize (lib/src/face_detector.dart:84-119, :297-415) and
 * _FaceDetectorCore.initializeFromBuffers (lib/src/isolate/face_detector_core.dart:118-212):
 * parses the detector (and optional face_landmark) .tflite flatbuffers, uploads weights,
 * generates the SSD anchors.  mesh_tflite may be NULL (fast mode only). */
FDT_EXPORT int32_t fdt_create(const fdt_config* cfg, const uint8_t* det_tflite, size_t det_len,
                              const uint8_t* mesh_tflite, size_t mesh_len, fdt_handle** out);

/* As fdt_create, plus the iris model (iris_landmark.tflite; IrisLandmark.createFromBuffer x2,
 * lib/src/isolate/face_detector_core.dart:172-190; NULL = no FDT_MODE_FULL) and an optional device list:
 * with num_devices > 1 the handle owns one replica per listed CUDA device and every detect call splits its
 * batch contiguously across them (one host thread, streams and staging per device, results in frame order;
 * no collective: frames are independent).  The reference's closest analogue is the interpreter pool inside
 * one detector object (RoundRobinPool, face_detector_core.dart:151-166).  devices == NULL: cfg->device only. */
FDT_EXPORT int32_t fdt_create_ex(const fdt_config* cfg, const uint8_t* det_tflite, size_t det_len,
                                 const uint8_t* mesh_tflite, size_t mesh_len, const uint8_t* iris_tflite,
                                 size_t iris_len, const int32_t* devices, int32_t num_devices, fdt_handle** out);

/* FaceDetector.dispose (lib/src/face_detector.dart:1061-1081). */
FDT_EXPORT int32_t fdt_destroy(fdt_handle* h);

/* New batched entry point (Dart: detectFacesBatch).  `frames` is `batch` tightly laid out images
 * of height x row_stride bytes (row_stride >= width * channels(mat_type); YUV formats: height * row_stride * 3 / 2
 * bytes, see FDT_FMT_YUV_NV12; planar RGB: 3 * height * row_stride, see FDT_FMT_RGB; packed YUV 4:2:2: row_stride >= 2 * width,
 * see FDT_FMT_YUYV), in host (pinned or
 * pageable) or device memory.  Replaces the per-frame sequence
 * _detectDetections -> applyDetectionGates -> computeFaceAlignment [-> extractAlignedSquare ->
 * FaceLandmark.callWithScore -> transformMeshToAbsolute]
 * (lib/src/isolate/face_detector_core.dart:215-394, :461-524).
 *   out_faces : [batch * max_faces] fdt_face      (host)
 *   out_counts: [batch] int32                     (host)
 *   out_mesh  : [batch * max_faces * 1404] float  (host; absolute pixels x,y,z) or NULL
 *   out_iris  : [batch * max_faces * 456] float   (host; FDT_MODE_FULL; absolute pixels x,y + raw z) or NULL
 * Only the first out_counts[b] slots of frame b are written. */
FDT_EXPORT int32_t fdt_detect_batch(fdt_handle* h, const uint8_t* frames, int32_t batch, int32_t width,
                                    int32_t height, int32_t row_stride, int32_t mat_type, int32_t mode,
                                    int32_t mem_kind, fdt_face* out_faces, int32_t* out_counts,
                                    float* out_mesh, float* out_iris);

/* One frame of a mixed batch (fdt_detect_frames): its own size and format. */
typedef struct fdt_frame {
  const uint8_t* data;       /* host or device memory, per the call's mem_kind                                   */
  int32_t width, height;     /* image size                                                                        */
  int32_t row_stride;        /* as fdt_detect_batch: >= width * channels; YUV: the Y-plane stride                 */
  int32_t mat_type;          /* FDT_MAT_8UC1 / _8UC3 / _8UC4, FDT_FMT_YUV_NV12 / _NV21 / _I420, FDT_FMT_RGB / _RGBA /
                                _RGB_PLANAR, FDT_FMT_YUYV / _UYVY / _YVYU, FDT_FMT_P010                           */
} fdt_frame;                 /* 24 bytes */

/* detectFacesFromMat over a list of frames of different sizes and formats (photos, mixed camera feeds), batched like
 * fdt_detect_batch: the frames run in chunks of up to max_batch through the same kernels, launches and two-slot pipeline.
 * Host frames also close a chunk when its staged bytes would pass max_batch * 8 MiB (a larger frame is a chunk of its own);
 * they go up whole (no sparse row upload), so fdt_last_h2d_bytes is the sum of the frames' sizes.  Device frames must be in
 * the handle's device memory; a multi-device handle takes host frames only and splits the list contiguously.
 * Outputs as fdt_detect_batch: faces [n][max_faces], counts [n], mesh [n][max_faces][1404], iris [n][max_faces][456]; each
 * frame's faces are normalised to its own size, mesh and iris points are in its own pixels.  Results are bitwise those of
 * fdt_detect_batch on each frame alone.  Every descriptor is checked before any work: the first bad one returns the code
 * fdt_detect_batch would return for it, and fdt_last_error names its index.  n == 0 returns FDT_OK. */
FDT_EXPORT int32_t fdt_detect_frames(fdt_handle* h, const fdt_frame* frames, int32_t n, int32_t mode, int32_t mem_kind,
                                     fdt_face* out_faces, int32_t* out_counts, float* out_mesh, float* out_iris);

/* Rotated and mirrored frames (video coded sideways, sensor-orientation camera frames, decoded photos with an EXIF tag) without a
 * rotation pass: fdt_detect_batch / fdt_detect_frames on frames stored in one of the eight FDT_ORIENT_* orientations.  width,
 * height, row_stride and mat_type (and every fdt_frame field) describe the STORED frame and are checked as before; YUV frames need
 * an even stored size.  Every result refers to the upright image U: faces are normalised to U's width and height, mesh and iris
 * points are in U's pixels, and the letterbox tap shows U letterboxed.  Results are bitwise those of the same call on U itself.
 * The letterbox and crop kernels read each stored pixel where U's tap falls; no rotated copy is made, and the kernel launch count
 * is that of orientation 1.  An orientation outside 1..8 returns FDT_ERR_BAD_ARG before any work (fdt_detect_frames_oriented:
 * fdt_last_error names the first bad index).  orientations: int32 [n], or NULL for all FDT_ORIENT_UPRIGHT.  fdt_detect_batch
 * is fdt_detect_batch_oriented with FDT_ORIENT_UPRIGHT, fdt_detect_frames is fdt_detect_frames_oriented with NULL.
 * Multi-device handles split the frames (and the orientations with them) contiguously, as the plain calls do. */
FDT_EXPORT int32_t fdt_detect_batch_oriented(fdt_handle* h, const uint8_t* frames, int32_t batch, int32_t width,
                                             int32_t height, int32_t row_stride, int32_t mat_type, int32_t orientation,
                                             int32_t mode, int32_t mem_kind, fdt_face* out_faces, int32_t* out_counts,
                                             float* out_mesh, float* out_iris);
FDT_EXPORT int32_t fdt_detect_frames_oriented(fdt_handle* h, const fdt_frame* frames, const int32_t* orientations, int32_t n,
                                              int32_t mode, int32_t mem_kind, fdt_face* out_faces, int32_t* out_counts,
                                              float* out_mesh, float* out_iris);

/* One YUV 4:2:0 frame given as three planes, each with its own base pointer and row stride (fdt_detect_yuv_planes): hardware
 * decoder surfaces (NVDEC / PyNvVideoCodec / FFmpeg cuda frames: pitched NV12 with the chroma at pitch * surface height), FFmpeg
 * and PyAV AVFrames (data[] and linesize[] of yuv420p / nv12) and Android YUV_420_888 images (three plane buffers, rowStride,
 * and a chroma pixelStride of 1 or 2).  The samples of pixel (x, y), x < width, y < height:
 *   Y  plane[0][y * row_stride[0] + x]
 *   U  plane[1][(y / 2) * row_stride[1] + (x / 2) * pixel_stride]
 *   V  plane[2][(y / 2) * row_stride[2] + (x / 2) * pixel_stride]
 * NV12 is U = chroma, V = chroma + 1, pixel_stride 2 (NV21 the other way round); I420 / YV12 are three planes with
 * pixel_stride 1.  width and height must be even and positive, every plane non-NULL, pixel_stride 1 or 2 and every row_stride
 * positive (else FDT_ERR_BAD_ARG; bottom-up frames with negative strides are not taken); row_stride[0] >= width and
 * row_stride[1], row_stride[2] >= (width / 2 - 1) * pixel_stride + 1 (else FDT_ERR_SIZE_MISMATCH).
 * The library reads only the sampled extent of each plane, (rows - 1) * row_stride + (cols - 1) * step + 1 bytes from its base
 * (Y: rows = height, cols = width, step 1; U and V: rows = height / 2, cols = width / 2, step = pixel_stride), so a buffer that
 * ends at its last sample (Android's truncated last chroma row) is complete. */
typedef struct fdt_yuv_planes {
  const uint8_t* plane[3];   /* Y, U, V; host or device memory, per the call's mem_kind                              */
  int32_t row_stride[3];     /* bytes between rows of each plane                                                       */
  int32_t width, height;     /* image size (even)                                                                      */
  int32_t pixel_stride;      /* bytes between neighbouring chroma samples of U and V: 1 (planar) or 2 (interleaved)    */
  int32_t reserved;          /* 0                                                                                      */
} fdt_yuv_planes;            /* 56 bytes */

/* fdt_detect_frames_oriented over separate-plane YUV 4:2:0 frames (fdt_yuv_planes): outputs, chunking, the two-slot pipeline,
 * orientations (int32 [n], or NULL for all upright), modes and multi-device splitting (host frames only) as there.  Every result
 * equals, bit for bit, fdt_detect_frames_oriented on the same samples packed into a contiguous FDT_FMT_YUV_I420 frame.  Every
 * descriptor is checked before any work; the first bad one returns its code and fdt_last_error names its index and plane.
 * n == 0 returns FDT_OK.
 * Host frames: each plane's sampled columns of every row go up (width bytes of each Y row, (width / 2 - 1) * pixel_stride + 1
 * bytes of each U and V row; no stride padding, nothing past a plane's extent).  Interleaved chroma - pixel_stride 2, U and V one
 * byte apart with one row stride >= width (NV12, NV21, Android views of one buffer) - goes up as one area of width bytes per row,
 * the two extents' bytes.  So fdt_last_h2d_bytes is the sum over the frames of width * height + (height / 2) * width for
 * interleaved chroma (what fdt_detect_frames uploads for an NV12 frame), else width * height + 2 * (height / 2) *
 * ((width / 2 - 1) * pixel_stride + 1).  No sparse row upload in fast mode.
 * Device frames must be in the handle's device memory; each plane pointer is checked, each allocation queried once per call.
 * A chunk whose frames all have U and V with one row stride and less than
 * 2^31 bytes apart (NVDEC NV12 surfaces, contiguous I420) runs the fdt_detect_frames kernels; any other chunk runs their
 * variants that read each frame's U and V planes through a per-frame plane table. */
FDT_EXPORT int32_t fdt_detect_yuv_planes(fdt_handle* h, const fdt_yuv_planes* frames, const int32_t* orientations, int32_t n,
                                         int32_t mode, int32_t mem_kind, fdt_face* out_faces, int32_t* out_counts,
                                         float* out_mesh, float* out_iris);

/* fdt_detect_yuv_planes over planes of little-endian 16-bit words: NVDEC / PyNvVideoCodec P016 surfaces (pitched, the chroma
 * at pitch * surface height: U = chroma, V = chroma + 2 bytes, pixel_stride 2) and FFmpeg / PyAV yuv420p10le / yuv420p12le
 * frames (three planes, data[] and linesize[], pixel_stride 1).  The same fdt_yuv_planes descriptors: row_stride[] counts bytes,
 * pixel_stride counts SAMPLES, so the words of pixel (x, y) are at
 *   Y  plane[0] + y * row_stride[0] + 2x
 *   U  plane[1] + (y / 2) * row_stride[1] + 2 * (x / 2) * pixel_stride,   V likewise from plane[2].
 * sample_bits (10, 12 or 16 for the whole call, else FDT_ERR_BAD_ARG before any work) is the number of significant bits stored
 * from bit 0: 10 / 12 for yuv420p10le / p12le, 16 for P010 / P016 surfaces; each sample becomes (s >> (sample_bits - 8)) & 0xFF,
 * the rule of FDT_FMT_P010.  Every result equals, bit for bit, fdt_detect_yuv_planes on the 8-bit planes made by that rule.
 * Checks as fdt_detect_yuv_planes, with the extents in samples x 2 bytes: row_stride[0] >= 2 * width and row_stride[1],
 * row_stride[2] >= 2 * ((width / 2 - 1) * pixel_stride + 1) (else FDT_ERR_SIZE_MISMATCH); every plane pointer and row stride must
 * be even (else FDT_ERR_BAD_ARG naming the frame and the plane).  Orientations, chunking, modes, face crops and multi-device
 * splitting of host frames are as there.
 * Host frames: each plane's sampled columns go up, twice the bytes of fdt_detect_yuv_planes' rule; interleaved chroma
 * (pixel_stride 2, U and V 2 bytes apart with one row stride >= 2 * width) as one area of 2 * width bytes per row.  So
 * fdt_last_h2d_bytes is the sum over the frames of 2 * width * height + (height / 2) * 2 * width for interleaved chroma, else
 * 2 * width * height + 4 * (height / 2) * ((width / 2 - 1) * pixel_stride + 1).  Every chunk runs the plane-table variants of
 * the letterbox and crop kernels. */
FDT_EXPORT int32_t fdt_detect_yuv_planes16(fdt_handle* h, const fdt_yuv_planes* frames, const int32_t* orientations, int32_t n,
                                           int32_t sample_bits, int32_t mode, int32_t mem_kind, fdt_face* out_faces,
                                           int32_t* out_counts, float* out_mesh, float* out_iris);

/* fdt_detect_jpeg over n encoded images in one call.  The host parses and Huffman-decodes them on a pool of
 * min(n, hardware threads) threads; the device decodes them into a handle-owned frame arena and detects them as one mixed
 * batch (chunks of up to max_batch images and max_batch * 8 MiB of decoded BGR).  out_status[i] is FDT_OK, FDT_ERR_FORMAT
 * (not a decodable JPEG; also NULL or empty buffers) or FDT_ERR_UNSUPPORTED; a failed image gets count 0 and out_wh 0, 0
 * and does not stop the others.  The call returns FDT_OK unless an argument or CUDA error stops the whole batch.
 * out_wh: [n][2] decoded width, height, or NULL.  Outputs otherwise as fdt_detect_frames; a multi-device handle splits the
 * list contiguously over its replicas. */
FDT_EXPORT int32_t fdt_detect_jpeg_batch(fdt_handle* h, const uint8_t* const* images, const size_t* sizes, int32_t n,
                                         int32_t mode, fdt_face* out_faces, int32_t* out_counts, float* out_mesh,
                                         float* out_iris, int32_t* out_wh, int32_t* out_status);

/* ---- Aligned face crops of the detect calls (the input of a second model: recognition, attributes, liveness) ----
 * With crops on (fdt_set_face_crops), every detect call - fdt_detect_batch[_oriented], fdt_detect_one, fdt_detect_frames[_oriented],
 * fdt_detect_yuv_planes, fdt_detect_jpeg, fdt_detect_jpeg_batch - also warps one square crop per returned face on the device,
 * straight from the frame it already holds there, in every format, orientation and memory kind.
 *   Which faces: every face the call returns (the out_counts[b] records of each frame, after the gates; in standard and full mode
 *     after the presence gate), packed in output order, frame by frame and then slot by slot: crop k is the k-th face of the
 *     flattened result.  No max_faces padding.
 *   ROI: built on the host from the RETURNED record's keypoints in pixels of the upright image (kp[2i] * width, kp[2i+1] * height,
 *     f64; in full mode the eyes are iris-refined):
 *       FDT_CROP_EMBEDDING  computeEmbeddingAlignment on the two eye keypoints (fdt_host_embedding_roi), then
 *                           extractAlignedSquare(cx, cy, size, -theta, out_size): the crop getFaceEmbedding feeds MobileFaceNet
 *                           (face_detector_core.dart:419-452; with layout 0 and out_size 112 it equals FaceDetector.embeddingCrop);
 *       FDT_CROP_FACE       computeFaceAlignment on the keypoints (fdt_host_face_roi), then extractAlignedSquare(cx, cy, size,
 *                           -theta, out_size): the face-mesh ROI (at out_size 192 the standard-mode mesh crop).
 *   Pixels: each crop equals extractAlignedSquare on the upright BGR image bit for bit.  layout 0 is u8 HWC BGR; the flags only
 *     reorder and convert: FDT_CROP_RGB reverses the channel order, FDT_CROP_CHW stores three S x S planes, FDT_CROP_F32 stores
 *     float (float)u8 * scale[c] + bias[c], a rounded multiply then a rounded add (no fused multiply-add), c in OUTPUT order.
 *     A crop of out_size S takes 3 * S * S bytes, times 4 with FDT_CROP_F32.
 *   Degenerate ROI (round(size) <= 0, where the reference returns null): the crop is all zero bytes and its ok flag 0.  The
 *     detector drops faces whose face ROI is degenerate, so detector output should not reach this.
 *   Lifetime: the crops of the last detect call (any of the entry points above); each such call and fdt_set_face_crops replace
 *     them.  With crops off the count is 0.
 *   Fast mode with crops on runs the standard-mode pipeline shape (faces to the host after the detector, then a host stage per
 *     chunk that writes the records and launches the crop warp), so host frames go up whole: fdt_last_h2d_bytes is the frames'
 *     full size.  fdt_detect_batch_device returns FDT_ERR_UNSUPPORTED while crops are on (its results never reach the host).
 *   Nothing else changes: with crops on, records, mesh, iris, counts and every debug tap are bitwise those of crops off.  The crop
 *     warps count in fdt_last_launch_count and are stage 9 of fdt_get_stage_ms. */
enum { FDT_CROP_EMBEDDING = 0, FDT_CROP_FACE = 1 };                 /* fdt_crop_spec.kind                                    */
enum { FDT_CROP_RGB = 1, FDT_CROP_CHW = 2, FDT_CROP_F32 = 4 };      /* fdt_crop_spec.layout flags; 0 = u8 HWC BGR            */
typedef struct fdt_crop_spec {
  int32_t struct_size;       /* sizeof(fdt_crop_spec)                                                                    */
  int32_t kind;              /* FDT_CROP_EMBEDDING / FDT_CROP_FACE                                                       */
  int32_t out_size;          /* S, 1..4096 (as fdt_extract_aligned_squares)                                              */
  int32_t layout;            /* FDT_CROP_* flags                                                                         */
  float scale[3], bias[3];   /* FDT_CROP_F32: out = (float)u8 * scale[c] + bias[c], c in output order; finite            */
} fdt_crop_spec;             /* 40 bytes */
/* spec NULL: crops off (the default).  A bad struct_size, kind, layout bit or out_size, or a non-finite scale or bias, returns
 * FDT_ERR_BAD_ARG and leaves the setting as it was.  A multi-device handle applies the spec to every replica. */
FDT_EXPORT int32_t fdt_set_face_crops(fdt_handle* h, const fdt_crop_spec* spec);
/* *out_n (optional): the crops of the last detect call.  *out_dev (optional): their packed array in a handle-owned device arena,
 * valid until the next detect call or fdt_set_face_crops; single-device handles only (a non-NULL out_dev returns
 * FDT_ERR_UNSUPPORTED on a multi-device handle). */
FDT_EXPORT int32_t fdt_get_face_crops(fdt_handle* h, int64_t* out_n, const void** out_dev);
/* Copies all crops to dst: host memory (mem_kind FDT_MEM_HOST) or the handle's device memory (FDT_MEM_DEVICE, single-device
 * handles only, else FDT_ERR_UNSUPPORTED).  capacity (bytes) below n * crop bytes returns FDT_ERR_SIZE_MISMATCH.  A multi-device
 * handle concatenates its replicas' crops in frame order.  out_ok (optional): int32 [n], 1 per crop, 0 where the ROI was
 * degenerate. */
FDT_EXPORT int32_t fdt_copy_face_crops(fdt_handle* h, void* dst, size_t capacity, int32_t mem_kind, int32_t* out_ok);

/* detectFacesFromMatBytes (lib/src/face_detector.dart:588-609): one packed frame of
 * `nbytes` bytes; FDT_ERR_SIZE_MISMATCH when nbytes != width*height*channels
 * (matFromPackedBytes, lib/src/util/helpers.dart:432-450), or != width*height*3/2 for the YUV formats
 * (FDT_FMT_RGB: width*height*3, FDT_FMT_RGBA: width*height*4, FDT_FMT_RGB_PLANAR: 3*width*height,
 * FDT_FMT_YUYV / _UYVY / _YVYU: 2*width*height, FDT_FMT_P010: 3*width*height, row_stride 2 * width). */
FDT_EXPORT int32_t fdt_detect_one(fdt_handle* h, const uint8_t* bytes, size_t nbytes, int32_t width,
                                  int32_t height, int32_t mat_type, int32_t mode, fdt_face* out_faces,
                                  int32_t* out_count, float* out_mesh, float* out_iris);

/* Throughput variant used by the benchmark: frames already resident in device memory, results
 * left in device memory (no host transfer, no sync); `*d_faces` / `*d_counts` receive internal
 * device pointers valid until the next call.  Same computation as fdt_detect_batch(fast).
 * FDT_ERR_UNSUPPORTED while face crops are on (fdt_set_face_crops). */
FDT_EXPORT int32_t fdt_detect_batch_device(fdt_handle* h, const uint8_t* d_frames, int32_t batch,
                                           int32_t width, int32_t height, int32_t row_stride,
                                           int32_t mat_type, int32_t mode, const fdt_face** d_faces,
                                           const int32_t** d_counts);
FDT_EXPORT int32_t fdt_synchronize(fdt_handle* h);

/* Model facts (FaceDetection.inputWidth/inputHeight, anchors; lib/src/models/face_detection_model.dart:138,:178). */
FDT_EXPORT int32_t fdt_get_info(fdt_handle* h, int32_t* input_w, int32_t* input_h, int32_t* num_anchors,
                                int32_t* max_faces, int32_t* max_batch);
FDT_EXPORT int32_t fdt_get_anchors(fdt_handle* h, double* out_xy /* [num_anchors*2] */);

/* computeLetterboxParams (flutter_litert; call site lib/src/util/helpers.dart:312-317):
 * out[6] = newW,newH,padTop,padBottom,padLeft,padRight. Pure host function. */
FDT_EXPORT int32_t fdt_letterbox_params(int32_t src_w, int32_t src_h, int32_t dst_w, int32_t dst_h,
                                        int32_t* out6);

/* Pinned host memory for frame / result buffers (dart:ffi callers allocate frames here so the
 * H2D copy runs at PCIe speed). */
FDT_EXPORT int32_t fdt_alloc_pinned(size_t nbytes, void** out);
FDT_EXPORT int32_t fdt_free_pinned(void* p);
/* Device memory helpers for callers that keep frames resident on the GPU (FDT_MEM_DEVICE). */
FDT_EXPORT int32_t fdt_alloc_device(fdt_handle* h, size_t nbytes, void** out);
FDT_EXPORT int32_t fdt_free_device(fdt_handle* h, void* p);
FDT_EXPORT int32_t fdt_copy_to_device(fdt_handle* h, void* dst, const void* src, size_t nbytes);
FDT_EXPORT int32_t fdt_copy_to_host(fdt_handle* h, void* dst, const void* src, size_t nbytes);

/* ---- parity taps (test / debug only; valid for the frames of the LAST detect call, first chunk) ----
 * n (or image) may not exceed the first chunk's frames (min(batch, max_batch)).  Chunks alternate over two
 * pipeline slots, so a call of more than two chunks (batch > 2 * max_batch) overwrites the first chunk's
 * buffers: after such a call the letterbox, input-tensor, raw-head and detector-tensor (which=0) taps
 * return FDT_ERR_BAD_ARG.  The candidate tap keeps the first chunk's index sets for any batch.
 * fdt_debug_get_letterboxed : u8 [n, S, S, 3] BGR after resize + copyMakeBorder
 *                             (convertImageToTensor u8 stage, lib/src/util/helpers.dart:303-347)
 * fdt_debug_get_input_tensor: f32 [n, S, S, 3] RGB in [-1,1] (bgrMatToSignedFloat32, :377-421)
 * fdt_debug_get_raw_heads   : f32 boxes [n, A, 16], scores [n, A] (Interpreter outputs 0 / 1,
 *                             lib/src/models/face_detection_model.dart:19)
 * fdt_debug_get_candidates  : ascending anchor indices with raw score >= logit(minScore)
 *                             (_collectCandidateScores, face_detection_model.dart:477-492)
 * fdt_debug_get_tensor      : any materialised activation of the detector (which=0), mesh (which=1)
 *                             or iris (which=2) graph by TFLite tensor index, as dense NHWC f32.
 *                             The mesh and iris tensors hold the last call's last mesh / iris pass. */
FDT_EXPORT int32_t fdt_debug_get_letterboxed(fdt_handle* h, int32_t n, uint8_t* out);
FDT_EXPORT int32_t fdt_debug_get_input_tensor(fdt_handle* h, int32_t n, float* out);
FDT_EXPORT int32_t fdt_debug_get_raw_heads(fdt_handle* h, int32_t n, float* out_boxes, float* out_scores);
FDT_EXPORT int32_t fdt_debug_get_candidates(fdt_handle* h, int32_t image, int32_t* out_indices,
                                            int32_t capacity, int32_t* out_n);
FDT_EXPORT int32_t fdt_debug_get_tensor(fdt_handle* h, int32_t which, int32_t tflite_tensor, int32_t n,
                                        float* out, size_t out_capacity_floats, int32_t* out_dims4);
/* Mesh stage taps: u8 [n,192,192,3] BGR crops (extractAlignedSquare, helpers.dart:583-625), raw
 * mesh outputs f32 [n,1404] + face-flag logits [n], for the first n faces of the LAST mesh pass of the
 * last call (a pass holds up to 2 * max_batch faces of one chunk, in frame then detection order).
 * out_n receives the size of that pass. */
FDT_EXPORT int32_t fdt_debug_get_mesh_stage(fdt_handle* h, int32_t n, uint8_t* out_crops,
                                            float* out_raw1404, float* out_flag, int32_t* out_n);
/* Iris stage taps for the first n faces of the LAST iris pass of the last call (the faces of the last mesh
 * pass that passed the presence gate and have two valid eye ROIs); out_n receives the faces of that pass:
 * u8 [2n,64,64,3] BGR eye crops (left, right-mirrored), the eye ROIs [2n,4] = cx, cy, size, theta
 * (eyeRoisFromMesh, face_geometry.dart:155-168), raw outputs f32 [2n,213] contours + [2n,15] iris. */
FDT_EXPORT int32_t fdt_debug_get_iris_stage(fdt_handle* h, int32_t n, uint8_t* out_crops, double* out_rois,
                                            float* out_contours, float* out_iris, int32_t* out_n);
/* Detector post-processing on caller-supplied tensors (host pointers), through the same k_decode_nms the
 * pipeline runs: crafted inputs and the reference's own unit-test vectors reach the device this way.
 *  fdt_debug_decode: raw heads boxes [n_images, N, 16] + scores [n_images, N] (Interpreter outputs 0 / 1),
 *    anchors_xy [N, 2] (NULL: the handle's), scale = model input height, pad4 = top, bottom, left, right
 *    (normalised; NULL = none).  Outputs faces [n_images, FDT_MAX_FACES] + counts, and optionally the decoded
 *    candidates before NMS: out_dec [n_images, N, 18] rows (box4, score, kp12, kept) in ascending anchor order
 *    + out_ndec [n_images] (_collectCandidateScores + _decodeBoxesForIndices + _toDetectionsFiltered,
 *    face_detection_model.dart:431-516; lib/src/web/detection_decode.dart:44-88).
 *  fdt_debug_nms: detections [n, 17] rows (xmin, ymin, xmax, ymax, score, kp12) -> weightedNms +
 *    letterbox removal (testNms / testDetectionLetterboxRemoval, helpers.dart:101-136, :183-221). */
FDT_EXPORT int32_t fdt_debug_decode(fdt_handle* h, const float* raw_boxes, const float* raw_scores,
                                    const double* anchors_xy, int32_t n_images, int32_t num_anchors, double scale,
                                    double score_thresh, double iou_thresh, const double* pad4,
                                    fdt_face* out_faces, int32_t* out_counts, double* out_dec, int32_t* out_ndec);
FDT_EXPORT int32_t fdt_debug_nms(fdt_handle* h, const double* dets17, int32_t n, double score_thresh,
                                 double iou_thresh, const double* pad4, fdt_face* out_faces, int32_t* out_count);
/* Number of kernel launches issued by the last detect call (bench.py "gpu_launches"). */
FDT_EXPORT int64_t fdt_last_launch_count(fdt_handle* h);
/* Bytes copied host->device by the last detect call.  In fast mode only the source rows the
 * INTER_LINEAR taps read are uploaded when they form a periodic pattern (e.g. 2 of every 10 rows
 * for 720 -> 72), so this can be far below batch * frame size.  YUV frames: the same rule applies to the Y plane
 * and to the chroma plane(s) independently (720 -> 72: Y rows 10k+4, 10k+5 and chroma rows 5k+2).
 * Oriented frames (fdt_detect_batch_oriented): the rule is "the stored rows the upright image's taps read" - U's y taps for
 * orientations 1-4, U's x taps for 5-8 (a 1280x720 frame stored sideways still uploads 2 rows in 10), after the flips.  The two
 * axes clamp differently at the borders, so at some sizes that set differs from orientation 1's.  RGB and RGBA frames upload as
 * BGR and BGRA do.  Planar RGB frames are read as 3 * height stacked rows: when height is a multiple of the period the same
 * pattern runs through all three planes (1280x720: 552,960 bytes per frame, as BGR), otherwise whole frames go up.  Packed YUV
 * 4:2:2 frames upload as a packed format of 2 bytes per pixel (1280x720: rows 10k+4, 10k+5, 368,640 bytes per frame).  FDT_FMT_P010
 * frames keep the YUV rule on both planes, each row 2 * width bytes (1280x720: Y rows 10k+4, 10k+5 and chroma row 5k+2, 552,960
 * bytes per frame, twice NV12's).  Mixed calls upload whole frames; fdt_detect_yuv_planes and fdt_detect_yuv_planes16 upload each
 * plane's sampled columns (see there). */
FDT_EXPORT int64_t fdt_last_h2d_bytes(fdt_handle* h);
/* Device time in ms of the named stage summed over the last call when stage timing was enabled
 * with fdt_set_stage_timing(h,1) (adds cudaEvent records; off by default).
 * stage: 0 letterbox, 1 conv stack, 2 decode+nms, 3 warp, 4 mesh net, 5 mesh post, 6 eye warp, 7 iris net, 8 iris post,
 * 9 face crops (fdt_set_face_crops) */
FDT_EXPORT int32_t fdt_set_stage_timing(fdt_handle* h, int32_t enable);
FDT_EXPORT int32_t fdt_get_stage_ms(fdt_handle* h, int32_t stage, float* ms, int32_t* launches);

/* Device-side timing of a region spanning all internal streams (bench.py): begin/end bracket any
 * number of detect calls; *ms is measured with CUDA events recorded on the library's own streams. */
FDT_EXPORT int32_t fdt_timer_begin(fdt_handle* h);
FDT_EXPORT int32_t fdt_timer_end(fdt_handle* h, float* ms);

/* Per-kernel device timing of the detector plan (bench.py roofline): runs `repeats` passes of one
 * chunk (n <= max_batch frames already in device memory) on one stream with a CUDA event between
 * consecutive kernels; out_ms[i] = mean duration of launch i, i = 0 letterbox, 1..S conv-stack
 * steps, S+1 decode+NMS.  fdt_get_step_info describes launch i: kernel name, tensor name, MACs and
 * algorithmic bytes (activation read + write, fp32) per image. */
FDT_EXPORT int32_t fdt_profile_chunk(fdt_handle* h, const uint8_t* d_frames, int32_t n, int32_t width,
                                     int32_t height, int32_t row_stride, int32_t mat_type, int32_t repeats,
                                     float* out_ms, int32_t capacity, int32_t* out_launches);
FDT_EXPORT int32_t fdt_get_step_info(fdt_handle* h, int32_t launch, char* kernel, char* tensor, int32_t str_cap,
                                     double* macs_per_image, double* bytes_per_image);
/* Same for the mesh (which = 1) and iris (which = 2) nets: `repeats` passes over the first n crops left in the
 * stage buffers by the last standard / full call (n <= 0 or too large: all of them; fdt_debug_get_mesh_stage /
 * fdt_debug_get_iris_stage report how many there are); out_ms[i] = mean duration of plan step i;
 * fdt_get_net_step_info describes step i of that plan. */
FDT_EXPORT int32_t fdt_profile_net(fdt_handle* h, int32_t which, int32_t n, int32_t repeats, float* out_ms,
                                   int32_t capacity, int32_t* out_steps);
FDT_EXPORT int32_t fdt_get_net_step_info(fdt_handle* h, int32_t which, int32_t step, char* kernel, char* tensor,
                                         int32_t str_cap, double* macs_per_image, double* bytes_per_image);
/* extractAlignedSquare on the device (lib/src/util/helpers.dart:583-625) for caller-supplied ROIs of ONE host frame:
 * rois [n, 4] = cx, cy, size, theta_arg (the function's own `theta` argument: the face path passes -theta, the eye
 * path +theta, the embedding path -theta with out_size 112, face_detector_core.dart:433-440).  out_crops u8
 * [n, out_size, out_size, 3] BGR; out_ok[i] = 0 where round(size) <= 0 (the reference returns null there). */
FDT_EXPORT int32_t fdt_extract_aligned_squares(fdt_handle* h, const uint8_t* frame, int32_t width, int32_t height,
                                               int32_t row_stride, int32_t mat_type, const double* rois, int32_t n,
                                               int32_t out_size, uint8_t* out_crops, int32_t* out_ok);
/* ---- JPEG front end: detectFacesFromBytes (lib/src/face_detector.dart:477-485; the reference decodes with cv.imdecode
 * and throws FormatException when the bytes cannot be decoded, :472-476) ------------------------------------------
 * The host parses the markers and runs the Huffman decoder (baseline and progressive, 8-bit, grey or YCbCr with 1x / 2x
 * chroma subsampling, restart intervals); dequantisation, the integer IDCT, fancy chroma upsampling, colour conversion
 * and the EXIF orientation run on the device and equal cv2.imdecode (libjpeg-turbo) byte for byte.
 * FDT_ERR_FORMAT: the bytes are not a decodable JPEG (FormatException); FDT_ERR_UNSUPPORTED: arithmetic coding, 12-bit,
 * CMYK, lossless.
 * fdt_detect_jpeg : decode + detect in `mode`; out_wh[2] (optional) receives the decoded width, height.
 * fdt_decode_jpeg : decode only; out_bgr (optional, host, packed BGR, capacity in bytes) receives the frame.
 * fdt_get_decoded_frame : copies the frame the last fdt_decode_jpeg / fdt_detect_jpeg left on the device (so a caller can
 *                   size its buffer from out_wh first without decoding twice). */
FDT_EXPORT int32_t fdt_detect_jpeg(fdt_handle* h, const uint8_t* bytes, size_t nbytes, int32_t mode, fdt_face* out_faces,
                                   int32_t* out_count, float* out_mesh, float* out_iris, int32_t* out_wh);
FDT_EXPORT int32_t fdt_decode_jpeg(fdt_handle* h, const uint8_t* bytes, size_t nbytes, uint8_t* out_bgr, size_t out_capacity,
                                   int32_t* out_wh);
FDT_EXPORT int32_t fdt_get_decoded_frame(fdt_handle* h, uint8_t* out_bgr, size_t out_capacity);

/* Number of CUDA devices the handle spans (1 unless created with a device list). */
FDT_EXPORT int32_t fdt_num_devices(fdt_handle* h);

/* ---- host-only helpers (no CUDA device needed; used by the CPU test-suite and by bindings) ----
 * fdt_host_anchors        : generateAnchors for a FaceDetectionModel; returns the anchor count
 *                           (out_xy may be NULL to query it).
 * fdt_host_plan_describe  : parses a .tflite buffer and lowers it to the kernel plan; writes a
 *                           human-readable listing (one line per kernel launch) into buf.
 * fdt_host_resize_taps    : cv::resize INTER_LINEAR 8U tap tables for one axis.
 * fdt_host_decode_box     : _decodeBoxesForIndices for one anchor (face_detection_model.dart:431-467).
 * fdt_host_face_roi       : computeFaceAlignment + extractAlignedSquare's inverse affine map
 *                           (face_geometry.dart:17-45, helpers.dart:583-625); out10 =
 *                           theta,cx,cy,size, a00,a01,b0,a10,a11,b1; returns 0 when round(size) <= 0.
 * fdt_host_eye_rois       : eyeRoisFromMesh (face_geometry.dart:155-168) from the four eye-corner mesh points
 *                           33, 133, 362, 263 (x,y absolute pixels) -> out8 = (cx, cy, size, theta) x {left, right}.
 * fdt_host_embedding_roi  : computeEmbeddingAlignment (lib/src/models/face_embedding.dart:362-384) from the two
 *                           eye points in pixels -> out4 = theta, cx, cy, size (the 112x112 embedding crop is
 *                           extractAlignedSquare(cx, cy, size, -theta, 112); the MobileFaceNet model itself is
 *                           not shipped by the reference).                                                  */
FDT_EXPORT int32_t fdt_host_anchors(int32_t model, double* out_xy, int32_t capacity_pairs);
FDT_EXPORT int32_t fdt_host_plan_describe(const uint8_t* tflite, size_t len, int32_t fuse_level, char* buf,
                                          size_t buf_len);
FDT_EXPORT int32_t fdt_host_resize_taps(int32_t src, int32_t dst, int32_t is_x_axis, int32_t* i0, int32_t* i1,
                                        int16_t* w0, int16_t* w1);
FDT_EXPORT int32_t fdt_host_decode_box(const float* raw16, double ax, double ay, double scale, double* out_box4,
                                       double* out_kp12);
FDT_EXPORT int32_t fdt_host_face_roi(const double* kp12, double img_w, double img_h, int32_t out_size,
                                     double* out10);
FDT_EXPORT int32_t fdt_host_eye_rois(const double* corners8, double* out8);
FDT_EXPORT int32_t fdt_host_embedding_roi(const double* left_eye_xy, const double* right_eye_xy, double* out4);
/* The incremental tile walk of the persistent kernels (csrc/tile_walk.h), run on the host: tiles first, first + stride, ...
 * (n of them) of a batch tiled tiles_x by tiles_y per image -> out3[3 i] = image, tile row, tile column.  Test hook: the
 * kernels advance (image, row, column) with adds and carries instead of dividing the tile index. */
FDT_EXPORT int32_t fdt_host_tile_walk(int32_t first, int32_t stride, int32_t tiles_x, int32_t tiles_y, int32_t n, int32_t* out3);
/* Host half of the JPEG front end, for tests and bindings: info8 = width, height, components, progressive, EXIF
 * orientation, hmax, vmax, 0.  fdt_host_jpeg_coefficients copies component `comp`'s quantised coefficients
 * ([blocks_h][blocks_w][64] int16, natural order, MCU-padded) and its quantisation table (natural order); dims6 =
 * blocks_w, blocks_h, samples_w, samples_h, h sampling factor, v sampling factor.  `out` may be NULL to query the sizes. */
FDT_EXPORT int32_t fdt_host_jpeg_info(const uint8_t* bytes, size_t nbytes, int32_t* info8);
FDT_EXPORT int32_t fdt_host_jpeg_coefficients(const uint8_t* bytes, size_t nbytes, int32_t comp, int16_t* out,
                                              size_t capacity, int32_t* dims6, uint16_t* qt64);

FDT_EXPORT const char* fdt_last_error(fdt_handle* h); /* NULL handle -> last create error */
FDT_EXPORT const char* fdt_version(void);

#ifdef __cplusplus
}
#endif
#endif /* FDT_API_H_ */
