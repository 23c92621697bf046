// C ABI of libfdt_cuda.so (see include/fdt_api.h).  Host-side orchestration of one detector handle:
// frames are processed in chunks that alternate over two slots (stream + arenas + staging each),
//   [H2D] -> letterbox -> BlazeFace conv stack -> decode + weighted NMS -> [D2H]                          (fast)
//   ... -> host: face ROIs -> warpAffine 192 -> face_landmark -> mesh unpack -> [D2H] -> presence gate     (standard)
//   ... -> host: eye ROIs -> warpAffine 64 x2 (+flip) -> iris_landmark -> iris unpack -> [D2H]             (full)
// mirroring _FaceDetectorCore.detectFacesDirect (lib/src/isolate/face_detector_core.dart:215-394).
// In standard / full mode the host sits between the stages exactly where the reference's Dart code does (ROI
// geometry with the host libm, presence gate); while it handles chunk c the other slot's stream runs chunk c + 1.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <tuple>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/fdt_api.h"
#include "engine.h"
#include "jpeg_host.h"
#include "fdt_math.h"
#include "kernels.h"
#include "tile_walk.h"

using namespace fdt;

static_assert(sizeof(fdt_face) == 160, "fdt_face wire layout (bindings rely on it)");
static_assert(sizeof(fdt_config) == 48, "fdt_config layout");
static_assert(sizeof(fdt_frame) == 24, "fdt_frame layout (bindings rely on it)");
static_assert(sizeof(fdt_crop_spec) == 40, "fdt_crop_spec layout (bindings rely on it)");

namespace {

constexpr int kSlots = 2;                 // chunks alternate over this many slots (stream + arenas each)
constexpr int kMeshInput = 192;           // face_landmark input
constexpr int kIrisInput = 64;            // iris_landmark input
constexpr double kMinScore = 0.5;         // lib/src/shared/face_model_config.dart:53
constexpr double kMinSuppression = 0.3;   // lib/src/shared/face_model_config.dart:77
constexpr int kNumStages = 10;
constexpr int kCropStage = 9;             // fdt_get_stage_ms stage of the face-crop warps
constexpr int kEagerSlots = 4;            // result slots per frame copied to the host with the chunk (more on demand)
// Mixed batches: a chunk of host frames (fdt_detect_frames) or of decoded JPEGs stages at most max_batch * this many bytes,
// e.g. 256 frames of 1920x1080 BGRA; a larger frame runs as a chunk of its own.
constexpr long long kStageBytesPerFrame = 8ll << 20;
constexpr size_t kStageAlign = 256;       // staged frames start at multiples of this

std::string g_create_error;
std::mutex g_create_mu;

struct SsdOptions { int num_layers, input_h, input_w; int strides[4]; double interp; };

// kSsdFront / kSsdBack / kSsdFull (lib/src/shared/face_model_config.dart:80-125)
SsdOptions ssd_options(int model) {
  switch (model) {
    case FDT_MODEL_BACK_CAMERA: return {4, 256, 256, {16, 32, 32, 32}, 1.0};
    case FDT_MODEL_FULL: case FDT_MODEL_FULL_SPARSE: return {1, 192, 192, {4, 0, 0, 0}, 0.0};
    default: return {4, 128, 128, {8, 16, 16, 16}, 1.0};
  }
}

// flutter_litert generateAnchors (call site lib/src/models/face_detection_model.dart:138,:178):
// layers with equal stride are merged; aspectRatios = [1.0] plus one interpolated-scale anchor.
std::vector<double> generate_anchors(const SsdOptions& o) {
  std::vector<double> out;
  int layer = 0;
  while (layer < o.num_layers) {
    int last = layer, repeats = 0;
    while (last < o.num_layers && o.strides[last] == o.strides[layer]) {
      repeats += 1 + (o.interp > 0 ? 1 : 0);
      ++last;
    }
    int stride = o.strides[layer];
    int fh = (o.input_h + stride - 1) / stride, fw = (o.input_w + stride - 1) / stride;
    for (int y = 0; y < fh; ++y) {
      double cy = (y + 0.5) / fh;
      for (int x = 0; x < fw; ++x) {
        double cx = (x + 0.5) / fw;
        for (int r = 0; r < repeats; ++r) { out.push_back(cx); out.push_back(cy); }
      }
    }
    layer = last;
  }
  return out;
}

struct LbTables {
  int w = 0, h = 0, o = 1;   // stored size, EXIF orientation; lp and the taps are those of the upright image (fdt_detect_batch_oriented)
  bool transposed = false;   // orientations 5-8: the x taps name stored rows, the y taps stored columns (k_letterbox_tr)
  LetterboxParams lp;
  int *x0 = nullptr, *x1 = nullptr, *y0 = nullptr, *y1 = nullptr;
  short *ax0 = nullptr, *ax1 = nullptr, *by0 = nullptr, *by1 = nullptr;
  bool identity = false;
  // Sparse upload (host frames, fast mode): INTER_LINEAR only reads the rows y0/y1 name (x0/x1 when transposed).  When those
  // rows form a periodic pattern (`run` consecutive rows every `period`, e.g. rows 10y+4,10y+5 for
  // 720 -> 72) a single strided DMA copies just them; y0c/y1c are those row taps renumbered into the compacted frame.
  bool sparse = false;
  int r0 = 0, run = 0, period = 0, rows_c = 0;
  int *y0c = nullptr, *y1c = nullptr;
  // YUV 4:2:0 frames (even sizes, resizing): chroma rows of the row taps (y0 / y1, or x0 / x1 when transposed, halved), and
  // the same sparse rule applied to the h / 2 rows of one chroma plane (c_rows_c: compacted rows per plane)
  int *cy0 = nullptr, *cy1 = nullptr;
  bool c_sparse = false;
  int c_r0 = 0, c_run = 0, c_period = 0, c_rows_c = 0;
  int *cy0c = nullptr, *cy1c = nullptr;
};

template <typename T> T* dev_upload(const std::vector<T>& v) {
  T* p = nullptr;
  if (cudaMalloc(&p, std::max<size_t>(v.size(), 1) * sizeof(T)) != cudaSuccess) return nullptr;
  cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
  return p;
}

// One pipeline slot: everything a chunk in flight owns.
struct Slot {
  cudaStream_t stream = nullptr;
  cudaEvent_t ev_det = nullptr;
  EngineCtx det_ctx, mesh_ctx, iris_ctx;
  uint8_t* d_frames = nullptr; size_t d_frames_cap = 0;   // host-frame staging (grown on demand)
  uint8_t* d_lb = nullptr;
  int* d_cand_idx = nullptr; int* d_cand_n = nullptr;
  int* h_counts = nullptr; fdt_face* h_faces = nullptr;                       // pinned [chunk], [chunk][max_faces]
  // mesh stage: ROI list (host-built, pinned -> device), crops, outputs
  int *h_crop_img = nullptr, *d_crop_img = nullptr;
  double *h_affine = nullptr, *d_affine = nullptr, *h_roi = nullptr, *d_roi = nullptr;
  uint8_t* d_crops = nullptr;
  float *d_mesh_out = nullptr, *h_mesh_out = nullptr;
  double *d_mesh_score = nullptr, *h_mesh_score = nullptr, *d_eye_corners = nullptr, *h_eye_corners = nullptr;
  // iris stage: two eye crops per face
  int *h_eye_img = nullptr, *d_eye_img = nullptr;
  double *h_eye_affine = nullptr, *d_eye_affine = nullptr, *h_eye_roi = nullptr, *d_eye_roi = nullptr;
  uint8_t* d_eye_crops = nullptr;
  float *d_iris_out = nullptr, *h_iris_out = nullptr;
  double *d_eye_kp = nullptr, *h_eye_kp = nullptr;
  // mixed batches: per chunk one pinned blob (frame descriptors, tap tables, decode geometry) goes up in one copy;
  // ev_blob follows that copy, and the next chunk on this slot waits on it before rewriting h_blob
  uint8_t *h_blob = nullptr, *d_blob = nullptr; size_t blob_cap = 0;
  cudaEvent_t ev_blob = nullptr;
  double *h_eye_wh = nullptr, *d_eye_wh = nullptr;    // frame size per iris face [F][2]
  PixFmt *h_pf = nullptr, *d_pf = nullptr;             // uniform RGB-family calls: the frames' pixel rule for the crop warps
  // face crops (fdt_set_face_crops): one pass's frame indices and inverse maps; ev_fc follows their upload
  int *h_fc_img = nullptr, *d_fc_img = nullptr;
  double *h_fc_aff = nullptr, *d_fc_aff = nullptr;
  cudaEvent_t ev_fc = nullptr;
};

}  // namespace

struct fdt_handle {
  fdt_config cfg;
  int chunk = 256, max_faces = FDT_MAX_FACES;
  Engine det, mesh, iris;
  bool has_mesh = false, has_iris = false;
  Slot slots[kSlots];
  fdt_face* d_faces = nullptr;
  int* d_counts = nullptr;
  int res_cap = 0;
  double* d_anchors = nullptr;
  std::vector<double> anchors;
  int num_anchors = 0, cand_cap = 0;
  std::vector<LbTables> tables;
  int mesh_cap = 0;                          // faces per mesh pass (iris: 2 * mesh_cap eye crops)
  std::vector<void*> dev_allocs, pin_allocs; // everything the slots own
  // multi-device parent: one replica per device, no device state of its own
  std::vector<fdt_handle*> shards;
  // bookkeeping
  std::mutex mu;
  std::string err;
  long long launches = 0;
  long long h2d_bytes = 0;
  long long jpeg_launches = 0;
  int last_first_chunk = 0;                  // images of the last call's first chunk (debug taps)
  bool slot0_first_chunk = true;             // slot 0 still holds that chunk: false once a third chunk reused the slot
  int last_mesh_faces = 0, last_mesh_slot = 0, last_iris_faces = 0, last_iris_slot = 0;
  bool stage_timing = false;
  float stage_ms[kNumStages] = {};
  int stage_launches[kNumStages] = {};
  cudaEvent_t ev[2] = {};
  cudaEvent_t tev[3] = {};
  // JPEG front end: coefficient / plane / frame buffers, grown on demand
  int16_t* d_jcoef = nullptr; size_t jcoef_cap = 0;
  uint8_t* d_jplanes = nullptr; size_t jplanes_cap = 0;
  uint8_t* d_jframe = nullptr; size_t jframe_cap = 0;
  uint16_t* d_jq = nullptr;
  int jw = 0, jh = 0;                        // size of the frame in d_jframe
  uint8_t* d_jarena = nullptr; size_t jarena_cap = 0;   // fdt_detect_jpeg_batch: one chunk's decoded frames
  // face crops of the detect calls (fdt_set_face_crops): the spec, and the last call's crops packed in a device arena
  bool crops_on = false;
  fdt_crop_spec crop_spec = {};
  int crop_cap = 0;                          // faces per crop pass (the slots' ROI buffers)
  uint8_t* d_crop_arena = nullptr; size_t crop_arena_cap = 0;
  long long crop_n = 0;
  std::vector<int32_t> crop_ok;
  bool ready = false;
};

namespace {

int fail(fdt_handle* h, int code, const std::string& msg) {
  if (h) h->err = msg;
  else { std::lock_guard<std::mutex> g(g_create_mu); g_create_error = msg; }
  return code;
}

bool cuda_ok(fdt_handle* h, cudaError_t e, const char* what) {
  if (e == cudaSuccess) return true;
  h->err = std::string(what) + ": " + cudaGetErrorString(e);
  return false;
}

int channels_of(int mat_type) {
  switch (mat_type) {
    case FDT_MAT_8UC1: return 1;
    case FDT_MAT_8UC3: return 3;
    case FDT_MAT_8UC4: return 4;
    default: return 0;
  }
}

bool is_yuv(int mat_type) { return mat_type == FDT_FMT_YUV_NV12 || mat_type == FDT_FMT_YUV_NV21 || mat_type == FDT_FMT_YUV_I420; }
bool is_rgb(int mat_type) { return mat_type == FDT_FMT_RGB || mat_type == FDT_FMT_RGBA || mat_type == FDT_FMT_RGB_PLANAR; }
bool is_yuv422(int mat_type) { return mat_type == FDT_FMT_YUYV || mat_type == FDT_FMT_UYVY || mat_type == FDT_FMT_YVYU; }

// Bytes of one pixel within a row: the packed formats' channels, 1 for planar RGB and YUV 4:2:0 (a row is one plane's), 2 for
// packed YUV 4:2:2 and P010 (a Y row of 16-bit words); 0: unknown.
int row_step(int mat_type) {
  if (is_yuv(mat_type) || mat_type == FDT_FMT_RGB_PLANAR) return 1;
  if (is_yuv422(mat_type) || mat_type == FDT_FMT_P010) return 2;
  if (mat_type == FDT_FMT_RGB) return 3;
  if (mat_type == FDT_FMT_RGBA) return 4;
  return channels_of(mat_type);
}

// Where the bytes of one input frame are.  Packed formats: height rows of row_stride bytes.  YUV 4:2:0: the Y plane, then the
// chroma area at c_off: c_rows rows of c_row_bytes (NV12 / NV21: h / 2 interleaved rows; I420: the h / 2 rows of U, then those
// of V), the chroma of pixel (x, y) at row y / 2 (+ h / 2 for V of I420), byte (x / 2) * c_step + u_off / v_off.
struct FrameLayout {
  int channels = 0;          // packed formats (RGB family and YUV 4:2:2: the pixel step); 0 for YUV 4:2:0
  bool yuv = false;
  bool rgb = false;          // FDT_FMT_RGB / _RGBA / _RGB_PLANAR and packed YUV 4:2:2: read through px by k_letterbox_rgb and the
                             // format-aware warps
  int planes = 1;            // planar RGB: 3 planes of height rows of row_stride, back to back
  PixFmt px;                 // every non-YUV format: pixel step and B, G, R offsets, P = one plane of the whole frame
  long long frame_bytes = 0;
  long long c_off = 0;
  int c_row_bytes = 0, c_rows = 0, c_step = 0, u_off = 0, v_off = 0;
  bool planar = false;       // I420: V is a plane of its own, h / 2 rows behind U
  bool p010 = false;         // FDT_FMT_P010: laid out as NV12 of 2-byte samples; c_step 4, u_off 1, v_off 3 name the chroma
                             // words' high bytes, and the k16 kernels read the Y word's high byte
};

// The pixel rule of a non-YUV 4:2:0 format (kernels.h, PixFmt); plane = bytes of one plane where the frame lies.
PixFmt pix_fmt(int mat_type, long long plane) {
  PixFmt f;
  f.step = row_step(mat_type);
  f.yuv422 = is_yuv422(mat_type) ? 1 : 0;
  // packed YUV 4:2:2: Y from byte 2x, U and V from the macropixel (kernels.h, load_422)
  if (mat_type == FDT_FMT_YUYV) { f.b = 0; f.g = 1; f.r = 3; }
  else if (mat_type == FDT_FMT_UYVY) { f.b = 1; f.g = 0; f.r = 2; }
  else if (mat_type == FDT_FMT_YVYU) { f.b = 0; f.g = 3; f.r = 1; }
  else if (mat_type == FDT_FMT_RGB_PLANAR) { f.b = 2 * plane; f.g = plane; f.r = 0; }
  else if (mat_type == FDT_FMT_RGB || mat_type == FDT_FMT_RGBA) { f.b = 2; f.g = 1; f.r = 0; }
  else if (f.step > 1) { f.b = 0; f.g = 1; f.r = 2; }
  return f;
}

// Validates the frame arguments (w, hh > 0 checked by the caller); *msg names the failure.
int frame_layout(int mat_type, int w, int hh, int row_stride, FrameLayout* L, const char** msg) {
  *L = FrameLayout();
  if (mat_type == FDT_FMT_P010) {
    if ((w & 1) || (hh & 1)) { *msg = "P010 frames need an even width and height"; return FDT_ERR_BAD_ARG; }
    if (row_stride & 1) { *msg = "P010 frames need an even row_stride"; return FDT_ERR_BAD_ARG; }
    if (row_stride < 2 * w) { *msg = "row_stride smaller than 2 * width"; return FDT_ERR_SIZE_MISMATCH; }
    L->yuv = true; L->p010 = true;
    L->frame_bytes = (long long)hh * row_stride * 3 / 2;
    L->c_off = (long long)hh * row_stride;
    L->c_row_bytes = row_stride; L->c_rows = hh / 2; L->c_step = 4; L->u_off = 1; L->v_off = 3;
    return FDT_OK;
  }
  if (!is_yuv(mat_type)) {
    L->channels = row_step(mat_type);
    if (L->channels == 0) { *msg = "bad frame arguments"; return FDT_ERR_BAD_ARG; }
    if (is_yuv422(mat_type) && (w & 1)) { *msg = "YUV 4:2:2 frames need an even width"; return FDT_ERR_BAD_ARG; }
    if (row_stride < w * L->channels) {
      *msg = L->channels == 1 && is_rgb(mat_type) ? "row_stride smaller than width"
             : is_yuv422(mat_type)                ? "row_stride smaller than 2 * width"
                                                  : "row_stride smaller than width * channels";
      return FDT_ERR_SIZE_MISMATCH;
    }
    L->rgb = is_rgb(mat_type) || is_yuv422(mat_type);
    L->planes = mat_type == FDT_FMT_RGB_PLANAR ? 3 : 1;
    L->frame_bytes = (long long)L->planes * hh * row_stride;
    L->px = pix_fmt(mat_type, (long long)hh * row_stride);
    return FDT_OK;
  }
  if ((w & 1) || (hh & 1)) { *msg = "YUV 4:2:0 frames need an even width and height"; return FDT_ERR_BAD_ARG; }
  if (row_stride < w) { *msg = "row_stride smaller than width"; return FDT_ERR_SIZE_MISMATCH; }
  L->yuv = true;
  L->frame_bytes = (long long)hh * row_stride * 3 / 2;
  L->c_off = (long long)hh * row_stride;
  if (mat_type == FDT_FMT_YUV_I420) {
    if (row_stride & 1) { *msg = "I420 frames need an even row_stride"; return FDT_ERR_BAD_ARG; }
    L->planar = true;
    L->c_row_bytes = row_stride / 2; L->c_rows = hh; L->c_step = 1; L->u_off = 0; L->v_off = hh / 2 * L->c_row_bytes;
  } else {
    L->c_row_bytes = row_stride; L->c_rows = hh / 2; L->c_step = 2;
    L->u_off = mat_type == FDT_FMT_YUV_NV12 ? 0 : 1; L->v_off = 1 - L->u_off;
  }
  return FDT_OK;
}

// The mode and model-availability checks of every detect entry point.
int check_mode(fdt_handle* h, int mode) {
  if (mode != FDT_MODE_FAST && mode != FDT_MODE_STANDARD && mode != FDT_MODE_FULL) return fail(h, FDT_ERR_BAD_ARG, "unknown mode");
  if (mode != FDT_MODE_FAST && !h->has_mesh) return fail(h, FDT_ERR_NOT_READY, "standard / full mode needs the face_landmark model");
  if (mode == FDT_MODE_FULL && !h->has_iris) return fail(h, FDT_ERR_NOT_READY, "full mode needs the iris_landmark model");
  return FDT_OK;
}

template <typename T> bool dalloc(fdt_handle* h, T** p, size_t n) {
  void* q = nullptr;
  if (cudaMalloc(&q, std::max<size_t>(n, 1) * sizeof(T)) != cudaSuccess) return false;
  h->dev_allocs.push_back(q);
  *p = static_cast<T*>(q);
  return true;
}
template <typename T> bool palloc(fdt_handle* h, T** p, size_t n) {
  void* q = nullptr;
  if (cudaMallocHost(&q, std::max<size_t>(n, 1) * sizeof(T)) != cudaSuccess) return false;
  h->pin_allocs.push_back(q);
  *p = static_cast<T*>(q);
  return true;
}

// The rows `need` marks are `run` consecutive rows every `period` (rows first .. first + run - 1 of each period), all the way
// down, with the plane height a multiple of the period and at most half of each period needed: worth a strided upload.
bool periodic_rows(const std::vector<char>& need, int* first_out, int* run_out, int* period_out) {
  const int hh = (int)need.size();
  int first = 0;
  while (first < hh && !need[first]) ++first;
  int run = 0;
  while (first + run < hh && need[first + run]) ++run;
  int next = first + run;
  while (next < hh && !need[next]) ++next;
  int period = next < hh ? next - first : 0;
  bool ok = period > run && hh % period == 0 && first + run <= period;
  for (int r = 0; ok && r < hh; ++r) {
    int ph = r % period;
    ok = (need[r] != 0) == (ph >= first && ph < first + run);
  }
  if (!ok || run * 2 > period) return false;
  *first_out = first; *run_out = run; *period_out = period;
  return true;
}

// EXIF orientation (fdt_detect_batch_oriented): the upright image U = exif_transform(stored, o) is the stored frame transposed
// for 5-8, then read backwards along U's x axis for 2, 3, 6, 7 and along U's y axis for 3, 4, 7, 8.
bool orient_transposed(int o) { return o >= 5; }
bool orient_flips_x(int o) { return o == 2 || o == 3 || o == 6 || o == 7; }
bool orient_flips_y(int o) { return o == 3 || o == 4 || o == 7 || o == 8; }
void upright_size(int w, int hh, int o, int* uw, int* uh) {
  *uw = orient_transposed(o) ? hh : w;
  *uh = orient_transposed(o) ? w : hh;
}
// Folds a flip into one axis' taps: tap i of an axis of n source pixels reads pixel n - 1 - i instead, weights unchanged.
void fold_flip(int* i0, int* i1, int taps, int n) {
  for (int i = 0; i < taps; ++i) { i0[i] = n - 1 - i0[i]; i1[i] = n - 1 - i1[i]; }
}

const LbTables* get_tables(fdt_handle* h, int w, int hh, int o) {
  for (const LbTables& t : h->tables)
    if (t.w == w && t.h == hh && t.o == o) return &t;
  // the cache is bounded: a stream of distinct resolutions recycles the oldest entry
  if (h->tables.size() >= 16) {
    LbTables& t = h->tables.front();
    for (int i = 0; i < kSlots; ++i) cudaStreamSynchronize(h->slots[i].stream);
    void* tp[] = {t.x0, t.x1, t.y0, t.y1, t.ax0, t.ax1, t.by0, t.by1, t.y0c, t.y1c, t.cy0, t.cy1, t.cy0c, t.cy1c};
    for (void* p : tp) if (p) cudaFree(p);
    h->tables.erase(h->tables.begin());
  }
  LbTables t;
  t.w = w; t.h = hh; t.o = o; t.transposed = orient_transposed(o);
  // U's letterbox and U's taps: the x axis rule for U's x taps even when they address stored rows (the axes clamp differently
  // at the borders).  Rotated / mirrored frames always take the tap path; at equal sizes it returns the pixels exactly.
  int uw = 0, uh = 0;
  upright_size(w, hh, o, &uw, &uh);
  t.lp = letterbox_params(uw, uh, h->det.in_w(), h->det.in_h());
  t.identity = o == 1 && t.lp.new_w == w && t.lp.new_h == hh;
  std::vector<int> x0(t.lp.new_w), x1(t.lp.new_w), y0(t.lp.new_h), y1(t.lp.new_h);
  std::vector<short> ax0(t.lp.new_w), ax1(t.lp.new_w), by0(t.lp.new_h), by1(t.lp.new_h);
  resize_linear_taps(uw, t.lp.new_w, true, x0.data(), x1.data(), ax0.data(), ax1.data());
  resize_linear_taps(uh, t.lp.new_h, false, y0.data(), y1.data(), by0.data(), by1.data());
  if (orient_flips_x(o)) fold_flip(x0.data(), x1.data(), t.lp.new_w, uw);
  if (orient_flips_y(o)) fold_flip(y0.data(), y1.data(), t.lp.new_h, uh);
  t.x0 = dev_upload(x0); t.x1 = dev_upload(x1); t.ax0 = dev_upload(ax0); t.ax1 = dev_upload(ax1);
  t.y0 = dev_upload(y0); t.y1 = dev_upload(y1); t.by0 = dev_upload(by0); t.by1 = dev_upload(by1);
  if (!t.x0 || !t.x1 || !t.ax0 || !t.ax1 || !t.y0 || !t.y1 || !t.by0 || !t.by1) return nullptr;
  if (!t.identity) {
    // the stored rows the taps read: named by the y taps, or by the x taps of a transposed frame
    const std::vector<int>& r0v = t.transposed ? x0 : y0;
    const std::vector<int>& r1v = t.transposed ? x1 : y1;
    const int nr = (int)r0v.size();
    std::vector<char> need(hh, 0);
    for (int i = 0; i < nr; ++i) { need[r0v[i]] = 1; need[r1v[i]] = 1; }
    int first = 0, run = 0, period = 0;
    if (periodic_rows(need, &first, &run, &period)) {
      std::vector<int> y0c(nr), y1c(nr);
      auto compact = [&](int r) { return (r / period) * run + (r % period - first); };
      for (int i = 0; i < nr; ++i) { y0c[i] = compact(r0v[i]); y1c[i] = compact(r1v[i]); }
      t.y0c = dev_upload(y0c); t.y1c = dev_upload(y1c);
      if (t.y0c && t.y1c) { t.sparse = true; t.r0 = first; t.run = run; t.period = period; t.rows_c = hh / period * run; }
    }
    if (hh % 2 == 0 && w % 2 == 0) {
      // YUV 4:2:0 chroma rows: the rows of one chroma plane (h / 2 of them) the taps read, same sparse rule
      const int ch = hh / 2;
      std::vector<int> cy0(nr), cy1(nr);
      std::vector<char> cneed(ch, 0);
      for (int i = 0; i < nr; ++i) { cy0[i] = r0v[i] >> 1; cy1[i] = r1v[i] >> 1; cneed[cy0[i]] = 1; cneed[cy1[i]] = 1; }
      t.cy0 = dev_upload(cy0); t.cy1 = dev_upload(cy1);
      if (!t.cy0 || !t.cy1) return nullptr;
      if (periodic_rows(cneed, &first, &run, &period)) {
        auto compact = [&](int r) { return (r / period) * run + (r % period - first); };
        for (int i = 0; i < nr; ++i) { cy0[i] = compact(cy0[i]); cy1[i] = compact(cy1[i]); }
        t.cy0c = dev_upload(cy0); t.cy1c = dev_upload(cy1);
        if (t.cy0c && t.cy1c) { t.c_sparse = true; t.c_r0 = first; t.c_run = run; t.c_period = period; t.c_rows_c = ch / period * run; }
      }
    }
  }
  h->tables.push_back(t);
  return &h->tables.back();
}

bool ensure_results(fdt_handle* h, int batch) {
  if (batch <= h->res_cap) return true;
  for (int i = 0; i < kSlots; ++i) cudaStreamSynchronize(h->slots[i].stream);
  if (h->d_faces) cudaFree(h->d_faces);
  if (h->d_counts) cudaFree(h->d_counts);
  h->d_faces = nullptr; h->d_counts = nullptr; h->res_cap = 0;
  int cap = std::max(batch, h->chunk);
  if (!cuda_ok(h, cudaMalloc(&h->d_faces, (size_t)cap * h->max_faces * sizeof(fdt_face)), "cudaMalloc(faces)")) return false;
  if (!cuda_ok(h, cudaMalloc(&h->d_counts, (size_t)cap * sizeof(int)), "cudaMalloc(counts)")) return false;
  cudaMemset(h->d_faces, 0, (size_t)cap * h->max_faces * sizeof(fdt_face));   // unused slots never expose stale device memory
  cudaMemset(h->d_counts, 0, (size_t)cap * sizeof(int));
  h->res_cap = cap;
  return true;
}

struct StageTimer {
  fdt_handle* h; int stage; cudaStream_t s; int launches;
  StageTimer(fdt_handle* hh, int st, cudaStream_t ss) : h(hh), stage(st), s(ss), launches(0) {
    if (h->stage_timing) cudaEventRecord(h->ev[0], s);
  }
  ~StageTimer() {
    h->launches += launches;
    if (!h->stage_timing) return;
    cudaEventRecord(h->ev[1], s);
    cudaEventSynchronize(h->ev[1]);
    float ms = 0;
    cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]);
    h->stage_ms[stage] += ms;
    h->stage_launches[stage] += launches;
  }
};

void fill_letterbox(LetterboxP& lb, const LbTables* tb, const uint8_t* d_fr, long long frame_stride, int row_stride, int channels,
                    int w, int hh, uint8_t* out, int S_w, int S_h, bool sparse) {
  lb.frames = d_fr; lb.frame_stride = frame_stride; lb.row_stride = row_stride; lb.channels = channels;
  lb.src_w = w; lb.src_h = hh; lb.out = out; lb.dst_w = S_w; lb.dst_h = S_h;
  lb.new_w = tb->lp.new_w; lb.new_h = tb->lp.new_h; lb.pad_top = tb->lp.pad_top; lb.pad_left = tb->lp.pad_left;
  // a compacted upload renumbers the taps that address rows: the y taps, or the x taps of a transposed frame
  const bool xs = sparse && tb->transposed, ys = sparse && !tb->transposed;
  lb.x0 = xs ? tb->y0c : tb->x0; lb.x1 = xs ? tb->y1c : tb->x1; lb.ax0 = tb->ax0; lb.ax1 = tb->ax1;
  lb.y0 = ys ? tb->y0c : tb->y0; lb.y1 = ys ? tb->y1c : tb->y1; lb.by0 = tb->by0; lb.by1 = tb->by1;
  lb.identity = tb->identity ? 1 : 0;
}

// YUV frames: the Y planes at d_y (y_stride bytes apart, compacted when y_sparse), the chroma areas at d_c (c_stride apart,
// compacted when c_sparse); for whole frames d_c = d_y + c_off and both strides are the frame size.
void fill_letterbox_yuv(LetterboxYuvP& p, const LbTables* tb, const FrameLayout& L, const uint8_t* d_y, long long y_stride,
                        bool y_sparse, const uint8_t* d_c, long long c_stride, bool c_sparse, int row_stride, int w, int hh,
                        uint8_t* out, int S_w, int S_h) {
  fill_letterbox(p.lb, tb, d_y, y_stride, row_stride, 0, w, hh, out, S_w, S_h, y_sparse);
  p.chroma = d_c; p.c_frame_stride = c_stride;
  p.c_row_stride = L.c_row_bytes; p.c_step = L.c_step; p.u_off = L.u_off;
  // I420: V follows U, whose rows are compacted like V's
  p.v_off = L.planar ? (c_sparse ? tb->c_rows_c : hh / 2) * L.c_row_bytes : L.v_off;
  p.cy0 = c_sparse ? tb->cy0c : tb->cy0; p.cy1 = c_sparse ? tb->cy1c : tb->cy1;
}

void set_warp_layout(WarpP& wp, const FrameLayout& L) {
  wp.yuv = L.yuv ? 1 : 0; wp.c_off = L.c_off; wp.c_row_stride = L.c_row_bytes; wp.c_step = L.c_step;
  wp.u_off = L.u_off; wp.v_off = L.v_off;
}

// `run` rows of every `period` of one plane (row_bytes per row, `groups` periods) of each of n frames fb bytes apart, src =
// the first needed row of frame 0, into dst as [n][groups * run][row_bytes].  One 3-D copy when the frame size is a whole number
// of periods (the host side is then one pitched volume), else one 2-D copy per frame.
void upload_rows(uint8_t* dst, const uint8_t* src, size_t row_bytes, int run, int period, int groups, size_t fb, int n, cudaStream_t s) {
  const size_t pitch = (size_t)period * row_bytes, width = (size_t)run * row_bytes;
  if (fb % pitch == 0) {
    cudaMemcpy3DParms c = {};
    c.srcPtr = make_cudaPitchedPtr(const_cast<uint8_t*>(src), pitch, width, fb / pitch);
    c.dstPtr = make_cudaPitchedPtr(dst, width, width, (size_t)groups);
    c.extent = make_cudaExtent(width, (size_t)groups, (size_t)n);
    c.kind = cudaMemcpyHostToDevice;
    cudaMemcpy3DAsync(&c, s);
  } else {
    for (int f = 0; f < n; ++f)
      cudaMemcpy2DAsync(dst + (size_t)f * width * groups, width, src + (size_t)f * fb, pitch, width, (size_t)groups,
                        cudaMemcpyHostToDevice, s);
  }
}

void fill_decode(DecodeP& d, fdt_handle* h, const Slot& sl, const LbTables* tb, int w, int hh) {
  const Plan& dp = h->det.plan();
  const int S_w = h->det.in_w(), S_h = h->det.in_h();
  d.boxes = sl.det_ctx.outputs[0]; d.boxes_istride = dp.out_elems[0];   // _boundingBoxIndex = 0
  d.scores = sl.det_ctx.outputs[1]; d.scores_istride = dp.out_elems[1]; // _scoreIndex = 1
  d.anchors = h->d_anchors; d.N = h->num_anchors; d.input_h = S_h;
  d.raw_thresh = std::log(kMinScore / (1.0 - kMinScore));
  d.score_thresh = kMinScore; d.iou_thresh = kMinSuppression;
  d.pad_t = d.pad_b = d.pad_l = d.pad_r = 0.0;    // no tables: mixed chunks pass per-image geometry (DecodeP::geom)
  if (tb) {
    d.pad_t = (double)tb->lp.pad_top / S_h; d.pad_b = (double)tb->lp.pad_bottom / S_h;
    d.pad_l = (double)tb->lp.pad_left / S_w; d.pad_r = (double)tb->lp.pad_right / S_w;
  }
  d.min_score = h->cfg.min_score; d.min_face_size = h->cfg.min_face_size;
  d.img_w = w; d.img_h = hh; d.max_faces = h->max_faces;
  d.cand_idx = nullptr; d.cand_cap = 0; d.cand_n = nullptr;
  d.pre = nullptr; d.dbg_dec = nullptr; d.skip_roi = 0;
}

// Letterbox geometry and INTER_LINEAR taps of one frame size and orientation, as k_letterbox_multi reads them: x0, x1, ax0, ax1
// (new_w each), then y0, y1, by0, by1, cy0, cy1 (new_h each).  Built on the host with resize_linear_taps for the upright size,
// flips folded in, like LbTables.
struct SizeTaps {
  LetterboxParams lp;
  bool identity = false;
  std::vector<int> t;
};

SizeTaps make_taps(int sw, int sh, int o, int S_w, int S_h) {
  SizeTaps st;
  int w = 0, hh = 0;
  upright_size(sw, sh, o, &w, &hh);
  st.lp = letterbox_params(w, hh, S_w, S_h);
  st.identity = o == 1 && st.lp.new_w == w && st.lp.new_h == hh;
  const int nw = st.lp.new_w, nh = st.lp.new_h;
  st.t.resize((size_t)4 * nw + 6 * nh);
  int* x = st.t.data();
  int* y = x + 4 * nw;
  std::vector<short> a0(std::max(nw, nh)), a1(std::max(nw, nh));
  resize_linear_taps(w, nw, true, x, x + nw, a0.data(), a1.data());
  for (int i = 0; i < nw; ++i) { x[2 * nw + i] = a0[i]; x[3 * nw + i] = a1[i]; }
  if (orient_flips_x(o)) fold_flip(x, x + nw, nw, w);
  resize_linear_taps(hh, nh, false, y, y + nh, a0.data(), a1.data());
  if (orient_flips_y(o)) fold_flip(y, y + nh, nh, hh);
  for (int i = 0; i < nh; ++i) { y[2 * nh + i] = a0[i]; y[3 * nh + i] = a1[i]; y[4 * nh + i] = y[i] >> 1; y[5 * nh + i] = y[nh + i] >> 1; }
  return st;
}

// One mixed call (fdt_detect_frames): the frames, their layouts and the taps of each distinct size.  The taps are computed once
// per size within the call instead of going through the handle's table cache: a stream of distinct sizes would evict that
// cache on every frame, and each eviction synchronises both slots.
struct Ragged {
  const fdt_frame* frames = nullptr;
  const int32_t* orientations = nullptr;   // [n] EXIF 1..8, or null: all upright
  std::vector<FrameLayout> lay;
  // fdt_detect_yuv_planes: the descriptors, and `frames` points at pframes, one fdt_frame per descriptor that gives the size and
  // the Y plane as the kernels read it (staged host frames: row stride = width); lay[i] is the staged layout (plane_layout)
  const fdt_yuv_planes* planes = nullptr;
  std::vector<fdt_frame> pframes;
  int bits = 0;                                         // fdt_detect_yuv_planes16: the call's sample_bits; 0: 8-bit planes
  std::map<std::tuple<int, int, int>, SizeTaps> taps;   // (stored width, height, orientation)
  int orientation(int i) const { return orientations ? orientations[i] : 1; }
};

struct CallArgs {
  const uint8_t* frames; int batch, w, hh, row_stride, channels, mode, mem_kind;
  FrameLayout lay;
  fdt_face* out_faces; int32_t* out_counts; float* out_mesh; float* out_iris;
  bool keep_on_device;
  const LbTables* tb;
  long long frame_stride;
  Ragged* rg = nullptr;                   // mixed call: per-frame sizes and layouts (the uniform fields above are unused)
  int orientation = 1;                    // EXIF orientation of every frame; w, hh are the stored size, uw, uh the upright one
  int uw = 0, uh = 0;
  bool crops = false;                     // face crops on (fdt_set_face_crops): fast mode runs a host stage per chunk too
};

// Upright size of frame i of the call: faces are normalised to it, the mesh and iris stages map their points into it.
void frame_size(const CallArgs& a, int i, double* w, double* hh) {
  if (a.rg) {
    int uw = 0, uh = 0;
    upright_size(a.rg->frames[i].width, a.rg->frames[i].height, a.rg->orientation(i), &uw, &uh);
    *w = uw; *hh = uh;
  } else {
    *w = a.uw; *hh = a.uh;
  }
}

// d_desc: a mixed chunk's frame descriptors on the device (the crop warps read the frames through them); orientation: as
// WarpP::orientation; d_pf: a mixed chunk's PixFmt table when it holds an RGB-family or YUV 4:2:2 frame, else null; d_pl: a
// chunk's YuvPlaneD table when its separate-plane device frames do not fit FrameD, else null; yuv422: the chunk holds a packed
// YUV 4:2:2 frame (the crop warps' launch_warp_affine flag); yuv16: the chunk holds a P010 frame or fdt_detect_yuv_planes16
// frames (the same for the yuv16 flags)
struct ChunkJob {
  int off = 0, n = 0; const uint8_t* d_fr = nullptr; const FrameD* d_desc = nullptr; bool active = false; int orientation = 1;
  const PixFmt* d_pf = nullptr;
  bool yuv422 = false, yuv16 = false;
  const YuvPlaneD* d_pl = nullptr;
};

// Samples of the sampled columns of one chroma row of a separate-plane frame: (width / 2 - 1) * pixel_stride + 1 (bytes for
// 8-bit planes; fdt_detect_yuv_planes16's 16-bit planes take twice as many).
long long chroma_cols(const fdt_yuv_planes& f) { return (long long)(f.width / 2 - 1) * f.pixel_stride + 1; }

// U and V interleaved in one chroma plane (NV12 / NV21, Android pixel stride 2 views of one buffer; P016 surfaces with bps = 2):
// pixel stride 2, one row stride of at least width samples, V one sample behind or before U.  Each chroma row's width samples
// from the lower of the two are then exactly the two sampled extents' bytes in that row.  bps: bytes per sample, 1 or 2.
bool interleaved_chroma(const fdt_yuv_planes& f, int bps) {
  const uintptr_t u = reinterpret_cast<uintptr_t>(f.plane[1]), v = reinterpret_cast<uintptr_t>(f.plane[2]);
  return f.pixel_stride == 2 && f.row_stride[1] == f.row_stride[2] && f.row_stride[1] >= f.width * bps &&
         (v == u + bps || u == v + bps);
}

// A separate-plane frame as it is staged from host memory: the Y plane (width samples per row), then the chroma, which FrameD
// describes as it describes NV12 / NV21 and I420 frames.  Interleaved chroma: one area of height / 2 rows of width samples (the
// bytes fdt_detect_frames uploads for an NV12 frame).  Otherwise the U and then the V area, height / 2 rows of chroma_cols
// samples each, chroma step pixel_stride.  bps: bytes per sample (2: fdt_detect_yuv_planes16, whose staged chroma the kernels
// read through YuvPlaneD with u_off, v_off and c_row_bytes in bytes).
FrameLayout plane_layout(const fdt_yuv_planes& f, int bps) {
  FrameLayout L;
  L.yuv = true;
  L.c_off = (long long)f.width * bps * f.height;
  L.c_step = f.pixel_stride * bps;
  if (interleaved_chroma(f, bps)) {
    L.c_row_bytes = f.width * bps; L.c_rows = f.height / 2;
    L.u_off = f.plane[1] < f.plane[2] ? 0 : bps; L.v_off = bps - L.u_off;
    L.frame_bytes = L.c_off + (long long)(f.height / 2) * L.c_row_bytes;
    return L;
  }
  const long long cc = chroma_cols(f) * bps;
  L.planar = true;
  L.c_row_bytes = (int)cc; L.c_rows = f.height; L.u_off = 0; L.v_off = (int)(f.height / 2 * cc);
  L.frame_bytes = L.c_off + 2 * (f.height / 2) * cc;
  return L;
}

// The sampled columns of every row, one 2-D copy per plane (interleaved chroma: one copy for U and V): nothing past a plane's
// sampled extent is read.  bps: bytes per sample.
void upload_planes(uint8_t* dst, const fdt_yuv_planes& f, const FrameLayout& L, int bps, cudaStream_t s) {
  const size_t y_row = (size_t)f.width * bps;
  cudaMemcpy2DAsync(dst, y_row, f.plane[0], f.row_stride[0], y_row, f.height, cudaMemcpyHostToDevice, s);
  if (!L.planar) {
    cudaMemcpy2DAsync(dst + L.c_off, L.c_row_bytes, std::min(f.plane[1], f.plane[2]), f.row_stride[1], L.c_row_bytes, f.height / 2,
                      cudaMemcpyHostToDevice, s);
    return;
  }
  for (int k = 1; k < 3; ++k)
    cudaMemcpy2DAsync(dst + L.c_off + (k == 2 ? L.v_off : 0), L.c_row_bytes, f.plane[k], f.row_stride[k], L.c_row_bytes,
                      f.height / 2, cudaMemcpyHostToDevice, s);
}

// Separate-plane device frames whose U and V share a row stride and lie less than 2^31 bytes apart (NVDEC NV12 surfaces,
// contiguous I420 / NV21) are FrameD frames with the chroma base at the lower of the two; others need the YuvPlaneD table.
bool fits_frame_desc(const fdt_yuv_planes& f) {
  const long long d = (long long)(reinterpret_cast<uintptr_t>(f.plane[2]) - reinterpret_cast<uintptr_t>(f.plane[1]));
  return f.row_stride[1] == f.row_stride[2] && d < INT32_MAX && d > -INT32_MAX;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// A mixed chunk on its slot's stream: host frames go up whole, one copy each at kStageAlign-aligned offsets; then the chunk's
// blob (frame descriptors, concatenated tap tables, decode geometry and, for a chunk with an RGB-family frame, every frame's
// PixFmt) in one copy; then k_letterbox_multi.
int stage_ragged(fdt_handle* h, Slot& sl, const CallArgs& a, int off, int n, const FrameD** d_desc, const double** d_geom,
                 int* orientation, const PixFmt** d_pf, const YuvPlaneD** d_pl, bool* yuv422, bool* yuv16) {
  cudaStream_t s = sl.stream;
  Ragged& rg = *a.rg;
  const fdt_frame* fr = rg.frames + off;
  const int S_w = h->det.in_w(), S_h = h->det.in_h();
  std::vector<const uint8_t*> base(n);
  if (a.mem_kind == FDT_MEM_HOST) {
    std::vector<size_t> at(n);
    size_t need = 0;
    for (int i = 0; i < n; ++i) { at[i] = need; need += align_up((size_t)rg.lay[off + i].frame_bytes, kStageAlign); }
    if (sl.d_frames_cap < need) {
      cudaStreamSynchronize(s);
      if (sl.d_frames) cudaFree(sl.d_frames);
      sl.d_frames = nullptr; sl.d_frames_cap = 0;
      if (!cuda_ok(h, cudaMalloc(&sl.d_frames, need), "cudaMalloc(frame staging)")) return FDT_ERR_CUDA;
      sl.d_frames_cap = need;
    }
    for (int i = 0; i < n; ++i) {
      const size_t fb = (size_t)rg.lay[off + i].frame_bytes;
      if (rg.planes) upload_planes(sl.d_frames + at[i], rg.planes[off + i], rg.lay[off + i], rg.bits ? 2 : 1, s);
      else cudaMemcpyAsync(sl.d_frames + at[i], fr[i].data, fb, cudaMemcpyHostToDevice, s);
      h->h2d_bytes += (long long)fb;
      base[i] = sl.d_frames + at[i];
    }
  } else {
    for (int i = 0; i < n; ++i) base[i] = fr[i].data;
  }
  // the chunk's distinct sizes and orientations, each with its taps at an offset of the concatenated table
  std::map<std::tuple<int, int, int>, int> tap_at;
  std::vector<const SizeTaps*> st(n);
  size_t ntaps = 0;
  bool upright = true, transposed = false, rgb = false;
  *yuv422 = false;
  *yuv16 = rg.bits != 0;
  for (int i = 0; i < n; ++i) {
    rgb = rgb || rg.lay[off + i].rgb;
    *yuv422 = *yuv422 || rg.lay[off + i].px.yuv422;
    *yuv16 = *yuv16 || rg.lay[off + i].p010;
    const int o = rg.orientation(off + i);
    upright = upright && o == 1;
    transposed = transposed || orient_transposed(o);
    const std::tuple<int, int, int> key(fr[i].width, fr[i].height, o);
    auto it = rg.taps.find(key);
    if (it == rg.taps.end()) it = rg.taps.emplace(key, make_taps(fr[i].width, fr[i].height, o, S_w, S_h)).first;
    st[i] = &it->second;
    if (tap_at.emplace(key, (int)ntaps).second) ntaps += it->second.t.size();
  }
  *orientation = upright ? 1 : 0;
  const fdt_yuv_planes* pl = rg.planes ? rg.planes + off : nullptr;
  // fdt_detect_yuv_planes16 frames, host or device, always go through the table (it carries their shift)
  bool table = rg.bits != 0;
  for (int i = 0; pl && a.mem_kind == FDT_MEM_DEVICE && i < n; ++i) table = table || !fits_frame_desc(pl[i]);
  const size_t taps_at = align_up((size_t)n * sizeof(FrameD), 16), geom_at = align_up(taps_at + ntaps * sizeof(int), 16);
  // a chunk with an RGB-family or YUV 4:2:2 frame also carries every frame's PixFmt (k_letterbox_multi<true, true>,
  // k_warp_affine<., ., true>; with a YUV 4:2:2 frame, k_letterbox_multi<true, true, false, true> and yuv422::k_warp_affine);
  // a chunk of separate-plane device frames that FrameD cannot describe, every frame's YuvPlaneD (the <., ., ., true> variants)
  const size_t pf_at = align_up(geom_at + (size_t)n * 6 * sizeof(double), 16);
  const size_t bytes = rgb ? pf_at + (size_t)n * sizeof(PixFmt)
                           : table ? pf_at + (size_t)n * sizeof(YuvPlaneD) : geom_at + (size_t)n * 6 * sizeof(double);
  if (sl.blob_cap < bytes) {
    cudaStreamSynchronize(s);
    if (sl.h_blob) cudaFreeHost(sl.h_blob);
    if (sl.d_blob) cudaFree(sl.d_blob);
    sl.h_blob = nullptr; sl.d_blob = nullptr; sl.blob_cap = 0;
    const size_t cap = bytes + bytes / 4;
    if (!cuda_ok(h, cudaMallocHost(&sl.h_blob, cap), "cudaMallocHost(chunk blob)") ||
        !cuda_ok(h, cudaMalloc(&sl.d_blob, cap), "cudaMalloc(chunk blob)")) return FDT_ERR_CUDA;
    sl.blob_cap = cap;
  } else if (!cuda_ok(h, cudaEventSynchronize(sl.ev_blob), "chunk blob")) {
    return FDT_ERR_CUDA;       // the blob of two chunks back may still be on its way up
  }
  FrameD* desc = reinterpret_cast<FrameD*>(sl.h_blob);
  int* taps = reinterpret_cast<int*>(sl.h_blob + taps_at);
  double* geom = reinterpret_cast<double*>(sl.h_blob + geom_at);
  for (const auto& kv : tap_at) {
    const std::vector<int>& t = rg.taps.at(kv.first).t;
    std::memcpy(taps + kv.second, t.data(), t.size() * sizeof(int));
  }
  for (int i = 0; i < n; ++i) {
    const FrameLayout& L = rg.lay[off + i];
    const LetterboxParams& lp = st[i]->lp;
    FrameD& d = desc[i];
    d.y = base[i]; d.c = L.yuv ? base[i] + L.c_off : nullptr;
    d.w = fr[i].width; d.h = fr[i].height; d.row_stride = fr[i].row_stride; d.channels = L.channels;
    d.c_row_stride = L.c_row_bytes; d.c_step = L.c_step; d.u_off = L.u_off; d.v_off = L.v_off;
    d.new_w = lp.new_w; d.new_h = lp.new_h; d.pad_top = lp.pad_top; d.pad_left = lp.pad_left; d.identity = st[i]->identity ? 1 : 0;
    if (pl && table) {
      const fdt_yuv_planes& f = pl[i];
      d.c = nullptr;
      YuvPlaneD q{f.plane[1], f.plane[2], f.row_stride[1], f.row_stride[2], f.pixel_stride, rg.bits ? rg.bits - 8 : 0};
      if (a.mem_kind == FDT_MEM_HOST) {   // fdt_detect_yuv_planes16: the staged chroma (plane_layout)
        q.u = base[i] + L.c_off + L.u_off; q.v = base[i] + L.c_off + L.v_off; q.u_stride = q.v_stride = L.c_row_bytes;
      }
      reinterpret_cast<YuvPlaneD*>(sl.h_blob + pf_at)[i] = q;
    } else if (pl && a.mem_kind == FDT_MEM_DEVICE) {
      const fdt_yuv_planes& f = pl[i];
      d.c = std::min(f.plane[1], f.plane[2]);
      d.c_row_stride = f.row_stride[1]; d.c_step = f.pixel_stride;
      d.u_off = (int)(f.plane[1] - d.c); d.v_off = (int)(f.plane[2] - d.c);
    }
    d.orientation = rg.orientation(off + i);
    d.tx = tap_at[std::make_tuple(d.w, d.h, d.orientation)]; d.ty = d.tx + 4 * lp.new_w;
    // the values fill_decode derives from LbTables, computed the same way
    double* g = geom + 6 * (size_t)i;
    g[0] = (double)lp.pad_top / S_h; g[1] = (double)lp.pad_bottom / S_h;
    g[2] = (double)lp.pad_left / S_w; g[3] = (double)lp.pad_right / S_w;
    int uw = 0, uh = 0;
    upright_size(d.w, d.h, d.orientation, &uw, &uh);
    g[4] = uw; g[5] = uh;
    if (rgb) reinterpret_cast<PixFmt*>(sl.h_blob + pf_at)[i] = L.px;
  }
  cudaMemcpyAsync(sl.d_blob, sl.h_blob, bytes, cudaMemcpyHostToDevice, s);
  cudaEventRecord(sl.ev_blob, s);
  *d_desc = reinterpret_cast<const FrameD*>(sl.d_blob);
  *d_geom = reinterpret_cast<const double*>(sl.d_blob + geom_at);
  *d_pf = rgb ? reinterpret_cast<const PixFmt*>(sl.d_blob + pf_at) : nullptr;
  *d_pl = table ? reinterpret_cast<const YuvPlaneD*>(sl.d_blob + pf_at) : nullptr;
  StageTimer t(h, 0, s);
  LetterboxMultiP lb;
  lb.fr = *d_desc; lb.taps = reinterpret_cast<const int*>(sl.d_blob + taps_at); lb.out = sl.d_lb; lb.dst_w = S_w; lb.dst_h = S_h;
  launch_letterbox_multi(lb, n, transposed, s, *d_pf, *d_pl, *yuv422, *yuv16);
  t.launches = 1;
  return FDT_OK;
}

// Stage 1 of a chunk on its slot's stream: [H2D] -> letterbox -> detector -> decode + NMS -> [D2H of counts and the
// first kEagerSlots result slots per frame].
// Uniform chunk: [H2D] -> k_letterbox / k_letterbox_yuv / k_letterbox_tr / k_letterbox_rgb; *d_fr = the frames on the device.
int stage_uniform(fdt_handle* h, Slot& sl, const CallArgs& a, int off, int n, const uint8_t** d_fr_out) {
  cudaStream_t s = sl.stream;
  const LbTables* tb = a.tb;
  const int S_w = h->det.in_w(), S_h = h->det.in_h();
  const bool fast_host = a.mem_kind == FDT_MEM_HOST && a.mode == FDT_MODE_FAST && !a.crops;   // the crop warps read whole frames
  const bool sparse = fast_host && !a.lay.yuv && tb->sparse;
  // YUV frames: the Y plane and the chroma area go up independently, each compacted when its tap rows are periodic
  const bool y_sparse = fast_host && a.lay.yuv && tb->sparse, c_sparse = fast_host && a.lay.yuv && tb->c_sparse;
  long long dev_frame_stride = a.frame_stride;
  const uint8_t* d_fr;
  const uint8_t* d_c = nullptr;
  long long y_stride = a.frame_stride, c_stride = a.frame_stride;
  if (a.mem_kind == FDT_MEM_HOST) {
    size_t need = (size_t)h->chunk * a.frame_stride;
    if (sl.d_frames_cap < need) {
      cudaStreamSynchronize(s);
      if (sl.d_frames) cudaFree(sl.d_frames);
      sl.d_frames = nullptr; sl.d_frames_cap = 0;
      if (!cuda_ok(h, cudaMalloc(&sl.d_frames, need), "cudaMalloc(frame staging)")) return FDT_ERR_CUDA;
      sl.d_frames_cap = need;
    }
    const uint8_t* src = a.frames + (size_t)off * a.frame_stride;
    if (y_sparse || c_sparse) {
      const FrameLayout& L = a.lay;
      const size_t fb = (size_t)a.frame_stride, y_bytes = (size_t)a.hh * a.row_stride, c_bytes = (size_t)L.c_rows * L.c_row_bytes;
      uint8_t* d_y = sl.d_frames;
      if (y_sparse) {
        upload_rows(d_y, src + (size_t)tb->r0 * a.row_stride, a.row_stride, tb->run, tb->period, a.hh / tb->period, fb, n, s);
        y_stride = (long long)tb->rows_c * a.row_stride;
      } else {
        cudaMemcpy2DAsync(d_y, y_bytes, src, fb, y_bytes, n, cudaMemcpyHostToDevice, s);
        y_stride = (long long)y_bytes;
      }
      uint8_t* dc = d_y + (size_t)n * y_stride;
      if (c_sparse) {
        // I420: U and V stacked are one area of h rows with the same period (h / 2 is a multiple of it)
        upload_rows(dc, src + L.c_off + (size_t)tb->c_r0 * L.c_row_bytes, L.c_row_bytes, tb->c_run, tb->c_period,
                    L.c_rows / tb->c_period, fb, n, s);
        c_stride = (long long)(L.c_rows / tb->c_period * tb->c_run) * L.c_row_bytes;
      } else {
        cudaMemcpy2DAsync(dc, c_bytes, src + L.c_off, fb, c_bytes, n, cudaMemcpyHostToDevice, s);
        c_stride = (long long)c_bytes;
      }
      h->h2d_bytes += (long long)n * (y_stride + c_stride);
      d_c = dc;
    } else if (sparse) {
      // one strided DMA: `run` rows out of every `period`, for all n frames (frames are contiguous).  Planar RGB: the planes are
      // 3 * hh stacked rows, and hh is a multiple of the period, so the pattern runs on through the G and B planes.
      const int planes = a.lay.planes;
      size_t width_b = (size_t)tb->run * a.row_stride;
      cudaMemcpy2DAsync(sl.d_frames, width_b, src + (size_t)tb->r0 * a.row_stride, (size_t)tb->period * a.row_stride,
                        width_b, (size_t)n * planes * (a.hh / tb->period), cudaMemcpyHostToDevice, s);
      dev_frame_stride = (long long)planes * tb->rows_c * a.row_stride;
      h->h2d_bytes += (long long)width_b * n * planes * (a.hh / tb->period);
    } else {
      cudaMemcpyAsync(sl.d_frames, src, (size_t)n * a.frame_stride, cudaMemcpyHostToDevice, s);
      h->h2d_bytes += (long long)n * a.frame_stride;
    }
    d_fr = sl.d_frames;
  } else {
    d_fr = a.frames + (size_t)off * a.frame_stride;
  }
  {
    StageTimer t(h, 0, s);
    if (a.lay.rgb) {
      LetterboxRgbP lb;
      fill_letterbox(lb.lb, tb, d_fr, dev_frame_stride, a.row_stride, a.channels, a.w, a.hh, sl.d_lb, S_w, S_h, sparse);
      lb.pf = a.lay.px;
      if (a.lay.planes > 1) lb.pf = pix_fmt(FDT_FMT_RGB_PLANAR, dev_frame_stride / a.lay.planes);   // the plane as uploaded
      launch_letterbox_rgb(lb, n, tb->transposed, s);
    } else if (tb->transposed) {
      LetterboxTrP lb;
      lb.yuv = a.lay.yuv ? 1 : 0;
      if (a.lay.yuv) {
        if (!d_c) d_c = d_fr + a.lay.c_off;
        fill_letterbox_yuv(lb.yp, tb, a.lay, d_fr, y_stride, y_sparse, d_c, c_stride, c_sparse, a.row_stride, a.w, a.hh, sl.d_lb, S_w, S_h);
      } else {
        lb.yp = LetterboxYuvP();
        fill_letterbox(lb.yp.lb, tb, d_fr, dev_frame_stride, a.row_stride, a.channels, a.w, a.hh, sl.d_lb, S_w, S_h, sparse);
      }
      launch_letterbox_tr(lb, n, s, a.lay.p010);
    } else if (a.lay.yuv) {
      if (!d_c) d_c = d_fr + a.lay.c_off;     // whole frames
      LetterboxYuvP lb;
      fill_letterbox_yuv(lb, tb, a.lay, d_fr, y_stride, y_sparse, d_c, c_stride, c_sparse, a.row_stride, a.w, a.hh, sl.d_lb, S_w, S_h);
      launch_letterbox_yuv(lb, n, s, a.lay.p010);
    } else {
      LetterboxP lb;
      fill_letterbox(lb, tb, d_fr, dev_frame_stride, a.row_stride, a.channels, a.w, a.hh, sl.d_lb, S_w, S_h, sparse);
      launch_letterbox(lb, n, s);
    }
    t.launches = 1;
  }
  *d_fr_out = d_fr;
  return FDT_OK;
}

int enqueue_detect(fdt_handle* h, Slot& sl, const CallArgs& a, int off, int n, bool first_chunk, ChunkJob* job) {
  cudaStream_t s = sl.stream;
  const uint8_t* d_fr = nullptr;
  const FrameD* d_desc = nullptr;
  const double* d_geom = nullptr;
  int orientation = a.orientation;
  const PixFmt* d_pf = nullptr;
  const YuvPlaneD* d_pl = nullptr;
  bool yuv422 = a.lay.px.yuv422 != 0, yuv16 = a.lay.p010;
  const int rc = a.rg ? stage_ragged(h, sl, a, off, n, &d_desc, &d_geom, &orientation, &d_pf, &d_pl, &yuv422, &yuv16)
                      : stage_uniform(h, sl, a, off, n, &d_fr);
  if (rc != FDT_OK) return rc;
  {
    StageTimer t(h, 1, s);
    t.launches = h->det.run(sl.det_ctx, sl.d_lb, n, s);
  }
  {
    StageTimer t(h, 2, s);
    DecodeP d;
    fill_decode(d, h, sl, a.tb, a.uw, a.uh);
    d.geom = d_geom;
    d.faces = h->d_faces + (size_t)off * h->max_faces; d.counts = h->d_counts + off;
    if (first_chunk) { d.cand_idx = sl.d_cand_idx; d.cand_cap = h->cand_cap; d.cand_n = sl.d_cand_n; }
    launch_decode_nms(d, n, s);
    t.launches = 1;
  }
  const size_t pitch = (size_t)h->max_faces * sizeof(fdt_face);
  const size_t eager = (size_t)std::min(kEagerSlots, h->max_faces) * sizeof(fdt_face);
  if (a.mode != FDT_MODE_FAST || a.crops) {
    cudaMemcpyAsync(sl.h_counts, h->d_counts + off, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, s);
    cudaMemcpy2DAsync(sl.h_faces, pitch, h->d_faces + (size_t)off * h->max_faces, pitch, eager, n, cudaMemcpyDeviceToHost, s);
    cudaEventRecord(sl.ev_det, s);
  } else if (!a.keep_on_device) {
    // Results leave compacted: counts + the first kEagerSlots slots of every frame now, the (rare) frames with more
    // faces are completed after the pipeline has drained (finish_fast).
    cudaMemcpyAsync(a.out_counts + off, h->d_counts + off, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, s);
    cudaMemcpy2DAsync(a.out_faces + (size_t)off * h->max_faces, pitch, h->d_faces + (size_t)off * h->max_faces, pitch, eager, n,
                      cudaMemcpyDeviceToHost, s);
  }
  job->off = off; job->n = n; job->d_fr = d_fr; job->d_desc = d_desc; job->active = true; job->orientation = orientation;
  job->d_pf = d_pf; job->d_pl = d_pl; job->yuv422 = yuv422; job->yuv16 = yuv16;
  return FDT_OK;
}

// Frames with more than kEagerSlots faces: fetch the remaining slots (all streams are idle here).
int fetch_overflow_faces(fdt_handle* h, const int32_t* counts, fdt_face* faces, int first, int n) {
  const int eager = std::min(kEagerSlots, h->max_faces);
  for (int b = 0; b < n; ++b) {
    const int c = counts[b];
    if (c <= eager) continue;
    const size_t o = (size_t)(first + b) * h->max_faces + eager;
    if (!cuda_ok(h, cudaMemcpy(faces + (size_t)b * h->max_faces + eager, h->d_faces + o, (size_t)(c - eager) * sizeof(fdt_face),
                               cudaMemcpyDeviceToHost), "result copy")) return FDT_ERR_CUDA;
  }
  return FDT_OK;
}

// eyeRoisFromMesh (lib/src/shared/face_geometry.dart:155-168): corners = mesh points 33, 133 (left) and 362, 263 (right)
void eye_rois_from_corners(const double* c8, double* out8 /* (cx, cy, size, theta) x 2 */) {
  for (int e = 0; e < 2; ++e) {
    const double p0x = c8[4 * e], p0y = c8[4 * e + 1], p1x = c8[4 * e + 2], p1y = c8[4 * e + 3];
    const double dx = p1x - p0x, dy = p1y - p0y;
    out8[4 * e + 0] = (p0x + p1x) * 0.5;
    out8[4 * e + 1] = (p0y + p1y) * 0.5;
    out8[4 * e + 2] = std::sqrt(dx * dx + dy * dy) * 2.3;
    out8[4 * e + 3] = std::atan2(dy, dx);
  }
}

// The crop warps' PixFmt: a mixed chunk's table, or for a uniform RGB-family or YUV 4:2:2 call the frames' own (whole frames).
const PixFmt* warp_pix_fmt(Slot& sl, const CallArgs& a, const ChunkJob& job) {
  if (!a.lay.rgb) return job.d_pf;
  *sl.h_pf = a.lay.px;
  cudaMemcpyAsync(sl.d_pf, sl.h_pf, sizeof(PixFmt), cudaMemcpyHostToDevice, sl.stream);
  return sl.d_pf;
}

// A crop warp over a chunk's frames: where they are on the device and how to read them.  The warps read whole frames: host frames
// go up unsparsified whenever a crop warp follows the detector.
WarpP chunk_warp(const CallArgs& a, const ChunkJob& job, const PixFmt* d_pf) {
  WarpP wp;
  wp.frames = job.d_fr; wp.frame_stride = a.frame_stride; wp.row_stride = a.row_stride; wp.channels = a.channels;
  wp.src_w = a.uw; wp.src_h = a.uh;
  set_warp_layout(wp, a.lay);
  wp.fr = job.d_desc; wp.orientation = job.orientation; wp.pf = d_pf;
  return wp;
}

size_t crop_bytes(const fdt_crop_spec& sp) { return (size_t)3 * sp.out_size * sp.out_size * ((sp.layout & FDT_CROP_F32) ? 4 : 1); }

// computeEmbeddingAlignment (lib/src/models/face_embedding.dart:362-384): out4 = theta, cx, cy, size from the eye points in pixels.
void embedding_alignment(const double* l, const double* r, double* out4) {
  const double dx = r[0] - l[0], dy = r[1] - l[1];
  const double theta = std::atan2(dy, dx);
  const double eye_dist = std::sqrt(dx * dx + dy * dy);
  const double size = eye_dist * 2.5;
  const double ecx = (l[0] + r[0]) * 0.5, ecy = (l[1] + r[1]) * 0.5;
  const double ct = std::cos(theta), st = std::sin(theta);
  const double oy = size * 0.15;
  out4[0] = theta; out4[1] = ecx - oy * st; out4[2] = ecy + oy * ct; out4[3] = size;
}

// Grows the crop arena to `need` bytes, keeping the crops earlier chunks of the call wrote.  Both slots' streams may still be
// writing crops, so they drain first; growth is geometric, so this happens a few times per handle.
bool grow_crop_arena(fdt_handle* h, size_t need) {
  if (need <= h->crop_arena_cap) return true;
  for (int i = 0; i < kSlots; ++i)
    if (!cuda_ok(h, cudaStreamSynchronize(h->slots[i].stream), "face crops")) return false;
  const size_t cap = std::max(need, 2 * h->crop_arena_cap);
  uint8_t* p = nullptr;
  if (!cuda_ok(h, cudaMalloc(&p, cap), "cudaMalloc(face crops)")) return false;
  const size_t used = (size_t)h->crop_n * crop_bytes(h->crop_spec);
  cudaStream_t s = h->slots[0].stream;
  if (used && (!cuda_ok(h, cudaMemcpyAsync(p, h->d_crop_arena, used, cudaMemcpyDeviceToDevice, s), "face crop arena") ||
               !cuda_ok(h, cudaStreamSynchronize(s), "face crop arena"))) {
    cudaFree(p);
    return false;
  }
  if (h->d_crop_arena) cudaFree(h->d_crop_arena);
  h->d_crop_arena = p; h->crop_arena_cap = cap;
  return true;
}

// One returned face of a chunk: its frame within the chunk and its record as the caller receives it.
struct FaceAt { int b; const fdt_face* fc; };

// Face crops of a chunk's returned faces, in output order (fdt_set_face_crops): ROIs on the host with the host libm from the
// returned records' keypoints in upright pixels, then one crop warp per pass of up to crop_cap faces, writing crops
// crop_n .. crop_n + nf - 1 of the arena.  Chunks finish in order, so the running count is the face's index in the flattened result.
int launch_face_crops(fdt_handle* h, Slot& sl, const CallArgs& a, const ChunkJob& job, const PixFmt* d_pf,
                      const std::vector<FaceAt>& faces) {
  cudaStream_t s = sl.stream;
  const fdt_crop_spec& sp = h->crop_spec;
  const size_t cb = crop_bytes(sp);
  for (size_t skip = 0; skip < faces.size(); skip += h->crop_cap) {
    const int nf = (int)std::min<size_t>(h->crop_cap, faces.size() - skip);
    if (!grow_crop_arena(h, (size_t)(h->crop_n + nf) * cb)) return FDT_ERR_CUDA;
    if (!cuda_ok(h, cudaEventSynchronize(sl.ev_fc), "face crop ROIs")) return FDT_ERR_CUDA;   // the last upload from these buffers
    std::vector<int> degenerate;
    for (int f = 0; f < nf; ++f) {
      const FaceAt& r = faces[skip + f];
      const double* kp = r.fc->keypoints;
      double fw, fh, theta, cx, cy, size;
      frame_size(a, job.off + r.b, &fw, &fh);
      if (sp.kind == FDT_CROP_FACE) {
        face_alignment(kp, fw, fh, &theta, &cx, &cy, &size);
      } else {
        // Detection.landmarks: the normalised keypoints times the image size, in f64
        const double le[2] = {kp[0] * fw, kp[1] * fh}, re[2] = {kp[2] * fw, kp[3] * fh};
        double e[4];
        embedding_alignment(le, re, e);
        theta = e[0]; cx = e[1]; cy = e[2]; size = e[3];
      }
      sl.h_fc_img[f] = r.b;
      const bool ok = aligned_square_inverse(cx, cy, size, -theta, sp.out_size, sl.h_fc_aff + 6 * f);
      if (!ok) {
        for (int k = 0; k < 6; ++k) sl.h_fc_aff[6 * f + k] = 0.0;
        degenerate.push_back(f);
      }
      h->crop_ok.push_back(ok ? 1 : 0);
    }
    cudaMemcpyAsync(sl.d_fc_img, sl.h_fc_img, (size_t)nf * sizeof(int), cudaMemcpyHostToDevice, s);
    cudaMemcpyAsync(sl.d_fc_aff, sl.h_fc_aff, (size_t)nf * 6 * sizeof(double), cudaMemcpyHostToDevice, s);
    cudaEventRecord(sl.ev_fc, s);
    {
      StageTimer t(h, kCropStage, s);
      WarpP wp = chunk_warp(a, job, d_pf);
      wp.crop_img = sl.d_fc_img; wp.affine = sl.d_fc_aff; wp.ncrops = nf; wp.out_size = sp.out_size; wp.flip_odd = 0;
      wp.crops = nullptr;
      CropOutP o;
      o.dst = h->d_crop_arena; o.first = h->crop_n; o.layout = sp.layout;
      for (int c = 0; c < 3; ++c) { o.scale[c] = sp.scale[c]; o.bias[c] = sp.bias[c]; }
      launch_warp_affine(wp, s, job.d_pl, &o, job.yuv422, job.yuv16);
      t.launches = 1;
    }
    // the reference returns null for these: the crop is all zero bytes (its ok flag says so)
    for (int f : degenerate) cudaMemsetAsync(h->d_crop_arena + (size_t)(h->crop_n + f) * cb, 0, cb, s);
    h->crop_n += nf;
  }
  return FDT_OK;
}

// The host stage of a fast-mode chunk with face crops on: the records reach the caller here instead of through the detector
// stage's copies (the same bytes: every frame's eager slots, then the faces past them), then the crop warp.
int finish_crops(fdt_handle* h, Slot& sl, const CallArgs& a, const ChunkJob& job) {
  const int n = job.n, off = job.off;
  if (!cuda_ok(h, cudaEventSynchronize(sl.ev_det), "detector stage")) return FDT_ERR_CUDA;
  if (fetch_overflow_faces(h, sl.h_counts, sl.h_faces, off, n) != FDT_OK) return FDT_ERR_CUDA;
  const int eager = std::min(kEagerSlots, h->max_faces);
  std::vector<FaceAt> faces;
  for (int b = 0; b < n; ++b) {
    const int c = sl.h_counts[b];
    fdt_face* dst = a.out_faces + (size_t)(off + b) * h->max_faces;
    std::memcpy(dst, sl.h_faces + (size_t)b * h->max_faces, (size_t)std::max(c, eager) * sizeof(fdt_face));
    a.out_counts[off + b] = c;
    for (int j = 0; j < c; ++j) faces.push_back({b, dst + j});
  }
  return launch_face_crops(h, sl, a, job, warp_pix_fmt(sl, a, job), faces);
}

// Stages 2-3 of a chunk (standard / full): host-built ROI lists between the device stages, presence gate, assembly.
int finish_mesh(fdt_handle* h, Slot& sl, const CallArgs& a, const ChunkJob& job) {
  cudaStream_t s = sl.stream;
  const int n = job.n, off = job.off;
  if (!cuda_ok(h, cudaEventSynchronize(sl.ev_det), "detector stage")) return FDT_ERR_CUDA;
  if (fetch_overflow_faces(h, sl.h_counts, sl.h_faces, off, n) != FDT_OK) return FDT_ERR_CUDA;
  struct Ref { int b, j; };
  std::vector<Ref> list;
  for (int b = 0; b < n; ++b)
    for (int j = 0; j < sl.h_counts[b]; ++j) list.push_back({b, j});
  std::vector<int> kept(n, 0);
  const long long total = (long long)list.size();
  const bool full = a.mode == FDT_MODE_FULL;
  const double gate = h->cfg.min_face_presence;
  const PixFmt* d_pf = warp_pix_fmt(sl, a, job);
  for (long long skip = 0; skip < total; skip += h->mesh_cap) {
    const int nf = (int)std::min<long long>(h->mesh_cap, total - skip);
    // ---- face ROIs on the host: computeFaceAlignment + extractAlignedSquare's matrix (face_detector_core.dart:478-507)
    for (int f = 0; f < nf; ++f) {
      const Ref r = list[(size_t)(skip + f)];
      const fdt_face& fc = sl.h_faces[(size_t)r.b * h->max_faces + r.j];
      double theta, cx, cy, size, fw, fh;
      frame_size(a, off + r.b, &fw, &fh);
      face_alignment(fc.keypoints, fw, fh, &theta, &cx, &cy, &size);
      double* roi = sl.h_roi + 6 * f;
      roi[0] = theta; roi[1] = cx; roi[2] = cy; roi[3] = size; roi[4] = std::cos(theta); roi[5] = std::sin(theta);
      sl.h_crop_img[f] = r.b;
      if (!aligned_square_inverse(cx, cy, size, -theta, kMeshInput, sl.h_affine + 6 * f))
        for (int k = 0; k < 6; ++k) sl.h_affine[6 * f + k] = 0.0;     // cannot happen: such faces were dropped by the decode kernel
    }
    cudaMemcpyAsync(sl.d_crop_img, sl.h_crop_img, (size_t)nf * sizeof(int), cudaMemcpyHostToDevice, s);
    cudaMemcpyAsync(sl.d_affine, sl.h_affine, (size_t)nf * 6 * sizeof(double), cudaMemcpyHostToDevice, s);
    cudaMemcpyAsync(sl.d_roi, sl.h_roi, (size_t)nf * 6 * sizeof(double), cudaMemcpyHostToDevice, s);
    {
      StageTimer t(h, 3, s);
      WarpP wp = chunk_warp(a, job, d_pf);
      wp.crop_img = sl.d_crop_img; wp.affine = sl.d_affine; wp.ncrops = nf; wp.out_size = kMeshInput; wp.flip_odd = 0;
      wp.crops = sl.d_crops;
      launch_warp_affine(wp, s, job.d_pl, nullptr, job.yuv422, job.yuv16);
      t.launches = 1;
    }
    {
      StageTimer t(h, 4, s);
      t.launches = h->mesh.run(sl.mesh_ctx, sl.d_crops, nf, s);
    }
    {
      StageTimer t(h, 5, s);
      // face_landmark.dart:154-166: landmarks = largest output divisible by 3, score = first 1-element output
      const Plan& mp = h->mesh.plan();
      int li = -1, si = -1;
      for (size_t k = 0; k < mp.out_elems.size(); ++k) {
        if (mp.out_elems[k] % 3 == 0 && (li < 0 || mp.out_elems[k] > mp.out_elems[li])) li = (int)k;
        if (mp.out_elems[k] == 1 && si < 0) si = (int)k;
      }
      MeshPostP pp;
      pp.raw = sl.mesh_ctx.outputs[li]; pp.raw_istride = mp.out_elems[li];
      pp.flag = sl.mesh_ctx.outputs[si]; pp.flag_istride = mp.out_elems[si];
      pp.roi = sl.d_roi; pp.nfaces = nf; pp.in_size = kMeshInput;
      pp.mesh_out = sl.d_mesh_out; pp.score_out = sl.d_mesh_score; pp.eye_corners = full ? sl.d_eye_corners : nullptr;
      launch_mesh_post(pp, s);
      t.launches = 1;
    }
    cudaMemcpyAsync(sl.h_mesh_score, sl.d_mesh_score, (size_t)nf * sizeof(double), cudaMemcpyDeviceToHost, s);
    if (a.out_mesh)
      cudaMemcpyAsync(sl.h_mesh_out, sl.d_mesh_out, (size_t)nf * FDT_MESH_FLOATS * sizeof(float), cudaMemcpyDeviceToHost, s);
    if (full) cudaMemcpyAsync(sl.h_eye_corners, sl.d_eye_corners, (size_t)nf * 8 * sizeof(double), cudaMemcpyDeviceToHost, s);
    if (!cuda_ok(h, cudaStreamSynchronize(s), "mesh stage")) return FDT_ERR_CUDA;
    h->last_mesh_faces = nf; h->last_mesh_slot = (int)(&sl - h->slots);
    // ---- presence gate (_passesPresence, face_detector_core.dart:101-103, :353) + slot assignment
    std::vector<int> slot_of(nf, -1);
    std::vector<int> iris_faces;
    for (int f = 0; f < nf; ++f) {
      const Ref r = list[(size_t)(skip + f)];
      const double sc = sl.h_mesh_score[f];
      if (!(gate <= 0.0 || sc >= gate)) continue;
      fdt_face fc = sl.h_faces[(size_t)r.b * h->max_faces + r.j];
      fc.mesh_score = sc;
      fc.has_mesh = 1;
      fc.has_iris = 0;
      const size_t slot = (size_t)(off + r.b) * h->max_faces + kept[r.b]++;
      a.out_faces[slot] = fc;
      if (a.out_mesh) std::memcpy(a.out_mesh + slot * FDT_MESH_FLOATS, sl.h_mesh_out + (size_t)f * FDT_MESH_FLOATS, FDT_MESH_FLOATS * sizeof(float));
      slot_of[f] = (int)(slot - (size_t)off * h->max_faces);
      if (full) iris_faces.push_back(f);
    }
    // ---- iris stage (_irisFromMesh, face_detector_core.dart:532-596)
    if (full && !iris_faces.empty()) {
      std::vector<int> run;              // faces whose two eye ROIs are both valid
      int ne = 0;
      for (int f : iris_faces) {
        double rois[8];
        eye_rois_from_corners(sl.h_eye_corners + 8 * f, rois);
        double aff[12];
        // extractAlignedSquare(image, roi.cx, roi.cy, roi.size, roi.theta, outSize: 64) for both eyes; either null -> no iris
        if (!aligned_square_inverse(rois[0], rois[1], rois[2], rois[3], kIrisInput, aff) ||
            !aligned_square_inverse(rois[4], rois[5], rois[6], rois[7], kIrisInput, aff + 6)) continue;
        for (int e = 0; e < 2; ++e) {
          double* roi = sl.h_eye_roi + 6 * (size_t)(ne + e);
          roi[0] = rois[4 * e + 3]; roi[1] = rois[4 * e]; roi[2] = rois[4 * e + 1]; roi[3] = rois[4 * e + 2];
          roi[4] = std::cos(roi[0]); roi[5] = std::sin(roi[0]);
          std::memcpy(sl.h_eye_affine + 6 * (size_t)(ne + e), aff + 6 * e, 6 * sizeof(double));
          sl.h_eye_img[ne + e] = list[(size_t)(skip + f)].b;
        }
        ne += 2;
        if (a.rg) frame_size(a, off + list[(size_t)(skip + f)].b, sl.h_eye_wh + 2 * run.size(), sl.h_eye_wh + 2 * run.size() + 1);
        run.push_back(f);
      }
      const int nfi = (int)run.size();
      if (nfi > 0) {
        cudaMemcpyAsync(sl.d_eye_img, sl.h_eye_img, (size_t)ne * sizeof(int), cudaMemcpyHostToDevice, s);
        cudaMemcpyAsync(sl.d_eye_affine, sl.h_eye_affine, (size_t)ne * 6 * sizeof(double), cudaMemcpyHostToDevice, s);
        cudaMemcpyAsync(sl.d_eye_roi, sl.h_eye_roi, (size_t)ne * 6 * sizeof(double), cudaMemcpyHostToDevice, s);
        if (a.rg) cudaMemcpyAsync(sl.d_eye_wh, sl.h_eye_wh, (size_t)nfi * 2 * sizeof(double), cudaMemcpyHostToDevice, s);
        {
          StageTimer t(h, 6, s);
          WarpP wp = chunk_warp(a, job, d_pf);
          wp.crop_img = sl.d_eye_img; wp.affine = sl.d_eye_affine; wp.ncrops = ne; wp.out_size = kIrisInput; wp.flip_odd = 1;
          wp.crops = sl.d_eye_crops;
          launch_warp_affine(wp, s, job.d_pl, nullptr, job.yuv422, job.yuv16);
          t.launches = 1;
        }
        {
          StageTimer t(h, 7, s);
          t.launches = h->iris.run(sl.iris_ctx, sl.d_eye_crops, ne, s);
        }
        {
          StageTimer t(h, 8, s);
          const Plan& ip = h->iris.plan();
          int ci = -1, ii = -1;                       // IrisLandmark unpacks every output in order: 71 contour points, 5 iris points
          for (size_t k = 0; k < ip.out_elems.size(); ++k) {
            if (ip.out_elems[k] == 213 && ci < 0) ci = (int)k;
            if (ip.out_elems[k] == 15 && ii < 0) ii = (int)k;
          }
          IrisPostP pp;
          pp.contours = sl.iris_ctx.outputs[ci]; pp.contours_istride = ip.out_elems[ci];
          pp.iris = sl.iris_ctx.outputs[ii]; pp.iris_istride = ip.out_elems[ii];
          pp.roi = sl.d_eye_roi; pp.nfaces = nfi; pp.in_size = kIrisInput; pp.img_w = a.uw; pp.img_h = a.uh;
          if (a.rg) pp.img_wh = sl.d_eye_wh;
          pp.iris_out = sl.d_iris_out; pp.eye_kp = sl.d_eye_kp;
          launch_iris_post(pp, s);
          t.launches = 1;
        }
        cudaMemcpyAsync(sl.h_eye_kp, sl.d_eye_kp, (size_t)nfi * 4 * sizeof(double), cudaMemcpyDeviceToHost, s);
        if (a.out_iris)
          cudaMemcpyAsync(sl.h_iris_out, sl.d_iris_out, (size_t)nfi * FDT_IRIS_FLOATS * sizeof(float), cudaMemcpyDeviceToHost, s);
        if (!cuda_ok(h, cudaStreamSynchronize(s), "iris stage")) return FDT_ERR_CUDA;
        h->last_iris_faces = nfi; h->last_iris_slot = (int)(&sl - h->slots);
        for (int k = 0; k < nfi; ++k) {
          const size_t slot = (size_t)off * h->max_faces + slot_of[run[k]];
          fdt_face& fc = a.out_faces[slot];
          // iris-refined eye keypoints (face_detector_core.dart:356-373): leftEye = index 0, rightEye = index 1
          fc.keypoints[0] = sl.h_eye_kp[4 * k]; fc.keypoints[1] = sl.h_eye_kp[4 * k + 1];
          fc.keypoints[2] = sl.h_eye_kp[4 * k + 2]; fc.keypoints[3] = sl.h_eye_kp[4 * k + 3];
          fc.has_iris = 1;
          if (a.out_iris) std::memcpy(a.out_iris + slot * FDT_IRIS_FLOATS, sl.h_iris_out + (size_t)k * FDT_IRIS_FLOATS, FDT_IRIS_FLOATS * sizeof(float));
        }
      }
    }
    // ---- face crops of the pass's returned faces (after the presence gate; full mode: with the iris-refined eyes)
    if (a.crops) {
      std::vector<FaceAt> kf;
      for (int f = 0; f < nf; ++f)
        if (slot_of[f] >= 0) kf.push_back({list[(size_t)(skip + f)].b, a.out_faces + (size_t)off * h->max_faces + slot_of[f]});
      if (int rc = launch_face_crops(h, sl, a, job, d_pf, kf)) return rc;
    }
  }
  for (int b = 0; b < n; ++b) a.out_counts[off + b] = kept[b];
  return FDT_OK;
}

// The chunks of one call (chunk c = frames bounds[c] .. bounds[c + 1] - 1) through the two-slot software pipeline.
int run_chunks(fdt_handle* h, const CallArgs& a, const std::vector<int>& bounds) {
  const int nchunks = (int)bounds.size() - 1, mode = a.mode;
  h->last_first_chunk = bounds[1] - bounds[0];
  h->slot0_first_chunk = nchunks <= kSlots;             // chunk c runs on slot c % kSlots
  h->last_mesh_faces = 0; h->last_iris_faces = 0;

  // the host stage of a chunk: mesh / iris (standard, full) or, in fast mode with face crops on, the records and the crop warp
  const bool host_stage = mode != FDT_MODE_FAST || a.crops;
  auto finish = [&](int i, const ChunkJob& job) {
    return mode == FDT_MODE_FAST ? finish_crops(h, h->slots[i], a, job) : finish_mesh(h, h->slots[i], a, job);
  };
  ChunkJob jobs[kSlots];
  int rc = FDT_OK;
  for (int c = 0; c < nchunks && rc == FDT_OK; ++c) {
    const int off = bounds[c], n = bounds[c + 1] - off;
    Slot& sl = h->slots[c % kSlots];
    // software pipeline: chunk c is queued on its slot, then the host turns to chunk c - 1 on the other slot
    rc = enqueue_detect(h, sl, a, off, n, c == 0, &jobs[c % kSlots]);
    if (rc == FDT_OK && host_stage && c > 0) {
      ChunkJob& prev = jobs[(c - 1) % kSlots];
      rc = finish((c - 1) % kSlots, prev);
      prev.active = false;
    }
  }
  if (rc == FDT_OK && host_stage) {
    for (int i = 0; i < kSlots && rc == FDT_OK; ++i)
      if (jobs[i].active) { rc = finish(i, jobs[i]); jobs[i].active = false; }
  }
  if (rc != FDT_OK) { for (int i = 0; i < kSlots; ++i) cudaStreamSynchronize(h->slots[i].stream); return rc; }
  if (!a.keep_on_device) {
    for (int i = 0; i < kSlots; ++i)
      if (!cuda_ok(h, cudaStreamSynchronize(h->slots[i].stream), "pipeline")) return FDT_ERR_CUDA;
    if (mode == FDT_MODE_FAST && !a.crops && fetch_overflow_faces(h, a.out_counts, a.out_faces, 0, a.batch) != FDT_OK) return FDT_ERR_CUDA;
  }
  if (!cuda_ok(h, cudaGetLastError(), "kernel launch")) return FDT_ERR_CUDA;
  if (h->det.failed() || h->mesh.failed() || h->iris.failed()) { h->err = "a kernel of the plan could not be launched (tensor map encoding / unsupported shape)"; return FDT_ERR_CUDA; }
  return FDT_OK;
}

int detect_single(fdt_handle* h, const uint8_t* frames, int batch, int w, int hh, int row_stride, int mat_type, int orientation,
                  int mode, int mem_kind, fdt_face* out_faces, int32_t* out_counts, float* out_mesh, float* out_iris,
                  bool keep_on_device) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  if (!frames || batch < 0 || w <= 0 || hh <= 0) return fail(h, FDT_ERR_BAD_ARG, "bad frame arguments");
  FrameLayout lay;
  const char* msg = nullptr;
  if (int rc = frame_layout(mat_type, w, hh, row_stride, &lay, &msg)) return fail(h, rc, msg);
  if (int rc = check_mode(h, mode)) return rc;
  if (mode != FDT_MODE_FAST && keep_on_device) return fail(h, FDT_ERR_UNSUPPORTED, "device-resident results are fast-mode only");
  if (!keep_on_device && (!out_faces || !out_counts)) return fail(h, FDT_ERR_BAD_ARG, "null output buffers");
  cudaSetDevice(h->cfg.device);
  h->launches = 0;
  h->h2d_bytes = 0;
  for (int i = 0; i < kNumStages; ++i) { h->stage_ms[i] = 0; h->stage_launches[i] = 0; }
  if (batch == 0) return FDT_OK;
  if (!ensure_results(h, batch)) return FDT_ERR_CUDA;
  CallArgs a;
  a.frames = frames; a.batch = batch; a.w = w; a.hh = hh; a.row_stride = row_stride; a.channels = lay.channels; a.mode = mode;
  a.lay = lay;
  a.mem_kind = mem_kind; a.out_faces = out_faces; a.out_counts = out_counts; a.out_mesh = out_mesh; a.out_iris = out_iris;
  a.keep_on_device = keep_on_device;
  a.orientation = orientation;
  a.crops = h->crops_on;
  upright_size(w, hh, orientation, &a.uw, &a.uh);
  a.tb = get_tables(h, w, hh, orientation);
  if (!a.tb) return fail(h, FDT_ERR_CUDA, "letterbox table upload failed");
  a.frame_stride = lay.frame_bytes;
  std::vector<int> bounds;
  for (int off = 0; off < batch; off += h->chunk) bounds.push_back(off);
  bounds.push_back(batch);
  return run_chunks(h, a, bounds);
}

// fdt_detect_frames' argument checks, every frame before any work; *lay receives the frames' layouts.
int check_frames(fdt_handle* h, const fdt_frame* frames, const int32_t* orientations, int n, int mode, int mem_kind,
                 const fdt_face* out_faces, const int32_t* out_counts, std::vector<FrameLayout>* lay) {
  if (n < 0 || (n > 0 && !frames)) return fail(h, FDT_ERR_BAD_ARG, "bad frame list");
  if (mem_kind != FDT_MEM_HOST && mem_kind != FDT_MEM_DEVICE) return fail(h, FDT_ERR_BAD_ARG, "unknown mem_kind");
  if (int rc = check_mode(h, mode)) return rc;
  if (n > 0 && (!out_faces || !out_counts)) return fail(h, FDT_ERR_BAD_ARG, "null output buffers");
  lay->assign(n, FrameLayout());
  for (int i = 0; i < n; ++i) {
    const fdt_frame& f = frames[i];
    const char* msg = "bad frame arguments";
    int rc = (!f.data || f.width <= 0 || f.height <= 0) ? FDT_ERR_BAD_ARG : frame_layout(f.mat_type, f.width, f.height, f.row_stride, &(*lay)[i], &msg);
    if (rc == FDT_OK && orientations && (orientations[i] < 1 || orientations[i] > 8)) {
      rc = FDT_ERR_BAD_ARG;
      msg = "orientation must be an EXIF value 1..8";
    }
    if (rc != FDT_OK) return fail(h, rc, "frame " + std::to_string(i) + ": " + msg);
  }
  return FDT_OK;
}

// fdt_detect_yuv_planes' argument checks, every descriptor before any work; *lay receives the frames' staged layouts.
// bits: fdt_detect_yuv_planes16's sample_bits (16-bit words: extents of 2 bytes per sample, even pointers and strides); 0: 8-bit.
int check_planes(fdt_handle* h, const fdt_yuv_planes* frames, const int32_t* orientations, int n, int mode, int mem_kind,
                 const fdt_face* out_faces, const int32_t* out_counts, std::vector<FrameLayout>* lay, int bits = 0) {
  if (n < 0 || (n > 0 && !frames)) return fail(h, FDT_ERR_BAD_ARG, "bad frame list");
  if (mem_kind != FDT_MEM_HOST && mem_kind != FDT_MEM_DEVICE) return fail(h, FDT_ERR_BAD_ARG, "unknown mem_kind");
  if (int rc = check_mode(h, mode)) return rc;
  if (n > 0 && (!out_faces || !out_counts)) return fail(h, FDT_ERR_BAD_ARG, "null output buffers");
  static const char* const kPlane[3] = {"plane Y", "plane U", "plane V"};
  lay->assign(n, FrameLayout());
  for (int i = 0; i < n; ++i) {
    const fdt_yuv_planes& f = frames[i];
    auto at = [i] { return "frame " + std::to_string(i) + ": "; };   // built on failure only: the list can be thousands long
    if (f.width <= 0 || f.height <= 0 || (f.width & 1) || (f.height & 1))
      return fail(h, FDT_ERR_BAD_ARG, at() + "YUV 4:2:0 frames need an even, positive width and height");
    for (int k = 0; k < 3; ++k)
      if (!f.plane[k]) return fail(h, FDT_ERR_BAD_ARG, at() + kPlane[k] + " is NULL");
    if (f.pixel_stride != 1 && f.pixel_stride != 2) return fail(h, FDT_ERR_BAD_ARG, at() + "pixel_stride must be 1 or 2");
    for (int k = 0; k < 3; ++k)
      if (f.row_stride[k] <= 0) return fail(h, FDT_ERR_BAD_ARG, at() + kPlane[k] + ": row_stride must be positive");
    const int bps = bits ? 2 : 1;
    if (bits)
      for (int k = 0; k < 3; ++k)
        if ((reinterpret_cast<uintptr_t>(f.plane[k]) | (uintptr_t)f.row_stride[k]) & 1)
          return fail(h, FDT_ERR_BAD_ARG, at() + kPlane[k] + ": 16-bit planes need an even pointer and row_stride");
    if (f.row_stride[0] < (long long)f.width * bps)
      return fail(h, FDT_ERR_SIZE_MISMATCH, at() + (bits ? "plane Y: row_stride smaller than 2 * width" : "plane Y: row_stride smaller than width"));
    for (int k = 1; k < 3; ++k)
      if (f.row_stride[k] < chroma_cols(f) * bps)
        return fail(h, FDT_ERR_SIZE_MISMATCH, at() + kPlane[k] + (bits ? ": row_stride smaller than 2 * ((width / 2 - 1) * pixel_stride + 1)"
                                                                       : ": row_stride smaller than (width / 2 - 1) * pixel_stride + 1"));
    if (orientations && (orientations[i] < 1 || orientations[i] > 8))
      return fail(h, FDT_ERR_BAD_ARG, at() + "orientation must be an EXIF value 1..8");
    (*lay)[i] = plane_layout(f, bps);
  }
  return FDT_OK;
}

// FDT_MEM_DEVICE pointers of one call: p must be in the handle's device memory.  A pointer inside an allocation this call has
// already checked needs no driver query: fdt_detect_yuv_planes checks three planes per frame, and decoder surfaces, tensors and
// their planes usually share a few allocations.  `ranges` keeps the last few checked allocations (driver cuPointerGetAttributes,
// resolved at run time like the tensor-map encoder; without it every pointer is queried).
bool device_pointer_ok(fdt_handle* h, const void* p, std::vector<std::pair<uintptr_t, uintptr_t>>* ranges) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(p);
  for (const auto& r : *ranges)
    if (a >= r.first && a < r.second) return true;
  cudaPointerAttributes pa;
  const bool ok = cudaPointerGetAttributes(&pa, p) == cudaSuccess &&
                  (pa.type == cudaMemoryTypeDevice || pa.type == cudaMemoryTypeManaged) && pa.device == h->cfg.device;
  cudaGetLastError();
  if (!ok) return false;
  using AttrsFn = CUresult (*)(unsigned, CUpointer_attribute*, void**, CUdeviceptr);
  static const AttrsFn attrs = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuPointerGetAttributes", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) f = nullptr;
    return reinterpret_cast<AttrsFn>(f);
  }();
  CUdeviceptr start = 0;
  size_t size = 0;
  CUpointer_attribute which[2] = {CU_POINTER_ATTRIBUTE_RANGE_START_ADDR, CU_POINTER_ATTRIBUTE_RANGE_SIZE};
  void* out[2] = {&start, &size};
  if (attrs && attrs(2, which, out, (CUdeviceptr)a) == CUDA_SUCCESS && size > 0 && a >= start && a < start + size) {
    if (ranges->size() == 8) ranges->erase(ranges->begin());
    ranges->emplace_back((uintptr_t)start, (uintptr_t)(start + size));
  }
  return true;
}

// What a ragged call was given: fdt_frame descriptors (fdt_detect_frames, the JPEG batch) or fdt_yuv_planes descriptors.
enum class FrameList { kFrames, kYuvPlanes };

// fdt_detect_frames (kFrames: `frames`) and fdt_detect_yuv_planes (kYuvPlanes: `planes`, frames unused) on one device; bits:
// fdt_detect_yuv_planes16's sample_bits, 0 for 8-bit planes.
int detect_frames_single(fdt_handle* h, const fdt_frame* frames, const int32_t* orientations, int n, int mode, int mem_kind,
                         fdt_face* out_faces, int32_t* out_counts, float* out_mesh, float* out_iris,
                         FrameList list = FrameList::kFrames, const fdt_yuv_planes* planes = nullptr, int bits = 0) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  Ragged rg;
  if (list == FrameList::kYuvPlanes) {
    if (int rc = check_planes(h, planes, orientations, n, mode, mem_kind, out_faces, out_counts, &rg.lay, bits)) return rc;
    rg.planes = planes;
    rg.bits = bits;
    rg.pframes.resize(n);
    const int bps = bits ? 2 : 1;
    for (int i = 0; i < n; ++i) {
      const fdt_yuv_planes& f = planes[i];
      rg.pframes[i] = fdt_frame{f.plane[0], f.width, f.height, mem_kind == FDT_MEM_HOST ? f.width * bps : f.row_stride[0], FDT_FMT_YUV_I420};
    }
    frames = rg.pframes.data();
  } else if (int rc = check_frames(h, frames, orientations, n, mode, mem_kind, out_faces, out_counts, &rg.lay)) {
    return rc;
  }
  cudaSetDevice(h->cfg.device);
  if (mem_kind == FDT_MEM_DEVICE && list == FrameList::kFrames)
    for (int i = 0; i < n; ++i) {
      cudaPointerAttributes pa;
      const bool ok = cudaPointerGetAttributes(&pa, frames[i].data) == cudaSuccess &&
                      (pa.type == cudaMemoryTypeDevice || pa.type == cudaMemoryTypeManaged) && pa.device == h->cfg.device;
      cudaGetLastError();
      if (!ok) return fail(h, FDT_ERR_BAD_ARG, "frame " + std::to_string(i) + ": FDT_MEM_DEVICE frames must be in the handle's device memory");
    }
  if (mem_kind == FDT_MEM_DEVICE && list == FrameList::kYuvPlanes) {
    static const char* const kPlane[3] = {"plane Y", "plane U", "plane V"};
    std::vector<std::pair<uintptr_t, uintptr_t>> ranges;
    for (int i = 0; i < n; ++i)
      for (int k = 0; k < 3; ++k)
        if (!device_pointer_ok(h, planes[i].plane[k], &ranges))
          return fail(h, FDT_ERR_BAD_ARG, "frame " + std::to_string(i) + ": " + kPlane[k] + ": FDT_MEM_DEVICE planes must be in the handle's device memory");
  }
  h->launches = 0;
  h->h2d_bytes = 0;
  for (int i = 0; i < kNumStages; ++i) { h->stage_ms[i] = 0; h->stage_launches[i] = 0; }
  if (n == 0) return FDT_OK;
  if (!ensure_results(h, n)) return FDT_ERR_CUDA;
  rg.frames = frames;
  rg.orientations = orientations;
  CallArgs a;
  a.frames = nullptr; a.batch = n; a.w = 0; a.hh = 0; a.row_stride = 0; a.channels = 0; a.mode = mode; a.mem_kind = mem_kind;
  a.out_faces = out_faces; a.out_counts = out_counts; a.out_mesh = out_mesh; a.out_iris = out_iris;
  a.keep_on_device = false; a.tb = nullptr; a.frame_stride = 0; a.rg = &rg; a.crops = h->crops_on;
  // a chunk closes at max_batch frames, or (host frames) before its staged bytes would pass the budget
  const long long budget = (long long)h->chunk * kStageBytesPerFrame;
  std::vector<int> bounds(1, 0);
  long long staged = 0;
  for (int i = 0; i < n; ++i) {
    const long long fb = mem_kind == FDT_MEM_HOST ? (long long)align_up((size_t)rg.lay[i].frame_bytes, kStageAlign) : 0;
    if (i - bounds.back() == h->chunk || (i > bounds.back() && staged + fb > budget)) { bounds.push_back(i); staged = 0; }
    staged += fb;
  }
  bounds.push_back(n);
  return run_chunks(h, a, bounds);
}

// Multi-device handle: items 0 .. n - 1 split contiguously (sharding.shard_range), one host thread per replica running
// fn(replica, lo, hi) under the replica's lock; launches and h2d bytes are summed, the first failing replica's error reported.
template <typename F> int on_shards(fdt_handle* h, int n, F fn) {
  const int g = (int)h->shards.size();
  std::vector<int> rcs(g, FDT_OK);
  std::vector<std::thread> th;
  for (int r = 0; r < g; ++r) {
    const int lo = (int)((long long)n * r / g), hi = (int)((long long)n * (r + 1) / g);
    if (hi <= lo) continue;
    th.emplace_back([=, &rcs, &fn] {
      fdt_handle* sh = h->shards[r];
      std::lock_guard<std::mutex> gl(sh->mu);
      rcs[r] = fn(sh, lo, hi);
    });
  }
  for (auto& t : th) t.join();
  h->launches = 0; h->h2d_bytes = 0;
  for (int r = 0; r < g; ++r) {
    h->launches += h->shards[r]->launches; h->h2d_bytes += h->shards[r]->h2d_bytes;
    if (rcs[r] != FDT_OK) { h->err = "device " + std::to_string(h->shards[r]->cfg.device) + ": " + h->shards[r]->err; return rcs[r]; }
  }
  return FDT_OK;
}

int detect_frames_multi(fdt_handle* h, const fdt_frame* frames, const int32_t* orientations, int n, int mode, int mem_kind,
                        fdt_face* out_faces, int32_t* out_counts, float* out_mesh, float* out_iris) {
  std::vector<FrameLayout> lay;
  if (int rc = check_frames(h, frames, orientations, n, mode, mem_kind, out_faces, out_counts, &lay)) return rc;
  if (mem_kind != FDT_MEM_HOST) return fail(h, FDT_ERR_UNSUPPORTED, "a multi-device handle takes host frames (device memory belongs to one device)");
  return on_shards(h, n, [=](fdt_handle* sh, int lo, int hi) {
    const size_t mf = (size_t)sh->max_faces;
    return detect_frames_single(sh, frames + lo, orientations ? orientations + lo : nullptr, hi - lo, mode, mem_kind,
                                out_faces + lo * mf, out_counts + lo,
                                out_mesh ? out_mesh + lo * mf * FDT_MESH_FLOATS : nullptr,
                                out_iris ? out_iris + lo * mf * FDT_IRIS_FLOATS : nullptr);
  });
}

int detect_planes_multi(fdt_handle* h, const fdt_yuv_planes* planes, const int32_t* orientations, int n, int mode, int mem_kind,
                        fdt_face* out_faces, int32_t* out_counts, float* out_mesh, float* out_iris, int bits = 0) {
  std::vector<FrameLayout> lay;
  if (int rc = check_planes(h, planes, orientations, n, mode, mem_kind, out_faces, out_counts, &lay, bits)) return rc;
  if (mem_kind != FDT_MEM_HOST) return fail(h, FDT_ERR_UNSUPPORTED, "a multi-device handle takes host frames (device memory belongs to one device)");
  return on_shards(h, n, [=](fdt_handle* sh, int lo, int hi) {
    const size_t mf = (size_t)sh->max_faces;
    return detect_frames_single(sh, nullptr, orientations ? orientations + lo : nullptr, hi - lo, mode, mem_kind,
                                out_faces + lo * mf, out_counts + lo,
                                out_mesh ? out_mesh + lo * mf * FDT_MESH_FLOATS : nullptr,
                                out_iris ? out_iris + lo * mf * FDT_IRIS_FLOATS : nullptr, FrameList::kYuvPlanes, planes + lo, bits);
  });
}

// Multi-device handle: contiguous split of the batch, one host thread per replica, results land in frame order.
int detect_multi(fdt_handle* h, const uint8_t* frames, int batch, int w, int hh, int row_stride, int mat_type, int orientation,
                 int mode, int mem_kind, fdt_face* out_faces, int32_t* out_counts, float* out_mesh, float* out_iris) {
  if (mem_kind != FDT_MEM_HOST) return fail(h, FDT_ERR_UNSUPPORTED, "a multi-device handle takes host frames (device memory belongs to one device)");
  if (!out_faces || !out_counts) return fail(h, FDT_ERR_BAD_ARG, "null output buffers");
  const int g = (int)h->shards.size();
  if (batch <= 0 || !frames) return detect_single(h->shards[0], frames, batch, w, hh, row_stride, mat_type, orientation, mode, mem_kind, out_faces, out_counts, out_mesh, out_iris, false);
  std::vector<int> rcs(g, FDT_OK);
  std::vector<std::thread> th;
  FrameLayout lay;
  const char* msg = nullptr;
  if (w <= 0 || hh <= 0) return fail(h, FDT_ERR_BAD_ARG, "bad frame arguments");
  if (int rc = frame_layout(mat_type, w, hh, row_stride, &lay, &msg)) return fail(h, rc, msg);
  const long long frame_stride = lay.frame_bytes;
  for (int r = 0; r < g; ++r) {
    const int lo = (int)((long long)batch * r / g), hi = (int)((long long)batch * (r + 1) / g);   // sharding.shard_range
    if (hi <= lo) continue;
    th.emplace_back([=, &rcs] {
      fdt_handle* sh = h->shards[r];
      std::lock_guard<std::mutex> gl(sh->mu);
      const int mf = sh->max_faces;
      rcs[r] = detect_single(sh, frames + (size_t)lo * frame_stride, hi - lo, w, hh, row_stride, mat_type, orientation, mode, mem_kind,
                             out_faces + (size_t)lo * mf, out_counts + lo, out_mesh ? out_mesh + (size_t)lo * mf * FDT_MESH_FLOATS : nullptr,
                             out_iris ? out_iris + (size_t)lo * mf * FDT_IRIS_FLOATS : nullptr, false);
    });
  }
  for (auto& t : th) t.join();
  h->launches = 0; h->h2d_bytes = 0;
  for (int r = 0; r < g; ++r) {
    h->launches += h->shards[r]->launches; h->h2d_bytes += h->shards[r]->h2d_bytes;
    if (rcs[r] != FDT_OK) { h->err = "device " + std::to_string(h->shards[r]->cfg.device) + ": " + h->shards[r]->err; return rcs[r]; }
  }
  return FDT_OK;
}

int detect_impl(fdt_handle* h, const uint8_t* frames, int batch, int w, int hh, int row_stride, int mat_type, int mode,
                int mem_kind, fdt_face* out_faces, int32_t* out_counts, float* out_mesh, float* out_iris, bool keep_on_device,
                int orientation = 1) {
  if (h && !h->shards.empty()) {
    if (keep_on_device) return fail(h, FDT_ERR_UNSUPPORTED, "device-resident results need a single-device handle");
    return detect_multi(h, frames, batch, w, hh, row_stride, mat_type, orientation, mode, mem_kind, out_faces, out_counts, out_mesh, out_iris);
  }
  return detect_single(h, frames, batch, w, hh, row_stride, mat_type, orientation, mode, mem_kind, out_faces, out_counts, out_mesh, out_iris, keep_on_device);
}

// the replica debug taps and profiling entries address (replica 0 of a multi-device handle)
fdt_handle* primary(fdt_handle* h) { return (h && !h->shards.empty()) ? h->shards[0] : h; }

// Every detect entry point replaces the face crops of the previous call (on every replica), whatever it returns.
void reset_crops(fdt_handle* h) {
  h->crop_n = 0;
  h->crop_ok.clear();
  for (fdt_handle* sh : h->shards) reset_crops(sh);
}

// The replicas whose crops a handle holds, in frame order.
std::vector<fdt_handle*> replicas(fdt_handle* h) { return h->shards.empty() ? std::vector<fdt_handle*>{h} : h->shards; }

int create_single(const fdt_config& cfg, const uint8_t* det_tflite, size_t det_len, const uint8_t* mesh_tflite, size_t mesh_len,
                  const uint8_t* iris_tflite, size_t iris_len, fdt_handle** out);

}  // namespace

// ------------------------------------------------------------------------------------------------
// ---- JPEG front end -----------------------------------------------------------------------------------------------
namespace {
template <typename T> bool grow(fdt_handle* h, T** p, size_t* cap, size_t need) {
  if (need <= *cap) return true;
  if (*p) cudaFree(*p);
  *p = nullptr; *cap = 0;
  const size_t want = need + need / 4 + 256;
  if (!cuda_ok(h, cudaMalloc(reinterpret_cast<void**>(p), want * sizeof(T)), "cudaMalloc(jpeg)")) return false;
  *cap = want;
  return true;
}

// size of the decoded frame: EXIF orientations 5-8 swap width and height
void jpeg_oriented_size(const JpegImage& img, int* w, int* hh) {
  const bool swap = img.orientation >= 5;
  *w = swap ? img.height : img.width; *hh = swap ? img.width : img.height;
}

// Device half of one decode, queued on s: coefficients up, IDCT per component, colour conversion + orientation into `out`
// (packed BGR).  Returns the kernel launches, or -1 (h->err set).
int jpeg_decode_device(fdt_handle* h, const JpegImage& img, uint8_t* out, cudaStream_t s) {
  size_t ncoef = 0, nplane = 0, coff[3] = {0, 0, 0}, poff[3] = {0, 0, 0};
  for (int c = 0; c < img.ncomp; ++c) {
    coff[c] = ncoef; poff[c] = nplane;
    ncoef += img.comp[c].coef.size();
    nplane += (size_t)img.comp[c].bw * 8 * img.comp[c].bh * 8;
  }
  int ow = 0, oh = 0;
  jpeg_oriented_size(img, &ow, &oh);
  if (!grow(h, &h->d_jcoef, &h->jcoef_cap, ncoef) || !grow(h, &h->d_jplanes, &h->jplanes_cap, nplane)) return -1;
  if (!h->d_jq && !cuda_ok(h, cudaMalloc(reinterpret_cast<void**>(&h->d_jq), 3 * 64 * sizeof(uint16_t)), "cudaMalloc(jpeg q)")) return -1;
  uint16_t q[3 * 64];
  for (int c = 0; c < img.ncomp; ++c) std::memcpy(q + 64 * c, img.qt[img.comp[c].tq], 64 * sizeof(uint16_t));
  // pageable sources: the copies are staged by the driver before the call returns, so the local buffers may go out of scope
  if (!cuda_ok(h, cudaMemcpyAsync(h->d_jq, q, (size_t)img.ncomp * 64 * sizeof(uint16_t), cudaMemcpyHostToDevice, s), "jpeg q upload")) return -1;
  for (int c = 0; c < img.ncomp; ++c)
    if (!cuda_ok(h, cudaMemcpyAsync(h->d_jcoef + coff[c], img.comp[c].coef.data(), img.comp[c].coef.size() * sizeof(int16_t), cudaMemcpyHostToDevice, s), "jpeg coefficient upload"))
      return -1;
  h->h2d_bytes += (long long)(ncoef * sizeof(int16_t));
  for (int c = 0; c < img.ncomp; ++c) {
    JpegIdctP p;
    p.coef = h->d_jcoef + coff[c]; p.q = h->d_jq + 64 * c; p.bw = img.comp[c].bw; p.bh = img.comp[c].bh;
    p.plane = h->d_jplanes + poff[c]; p.pitch = img.comp[c].bw * 8;
    launch_jpeg_idct(p, s);
  }
  JpegColorP cp;
  cp.py = h->d_jplanes + poff[0]; cp.pitch_y = img.comp[0].bw * 8;
  cp.pcb = cp.pcr = cp.py; cp.pitch_c = cp.pitch_y; cp.cdw = img.comp[0].dw; cp.cdh = img.comp[0].dh; cp.hs = cp.vs = 1;
  if (img.ncomp == 3) {
    cp.pcb = h->d_jplanes + poff[1]; cp.pcr = h->d_jplanes + poff[2]; cp.pitch_c = img.comp[1].bw * 8;
    cp.cdw = img.comp[1].dw; cp.cdh = img.comp[1].dh; cp.hs = img.hmax / img.comp[1].h; cp.vs = img.vmax / img.comp[1].v;
  }
  cp.W = img.width; cp.H = img.height; cp.ncomp = img.ncomp; cp.orientation = img.orientation;
  cp.out = out; cp.out_w = ow;
  launch_jpeg_color(cp, s);
  return img.ncomp + 1;
}

// decodes into h->d_jframe (packed BGR, EXIF orientation applied); *w / *hh = the oriented size
int jpeg_to_device(fdt_handle* h, const uint8_t* bytes, size_t nbytes, int* w, int* hh) {
  if (!bytes || nbytes == 0) return fail(h, FDT_ERR_FORMAT, "empty image buffer");
  JpegImage img;
  std::string e;
  const JpegStatus st = jpeg_decode_coefficients(bytes, nbytes, &img, &e);
  if (st == kJpegBad) return fail(h, FDT_ERR_FORMAT, e);
  if (st == kJpegUnsupported) return fail(h, FDT_ERR_UNSUPPORTED, e);
  cudaSetDevice(h->cfg.device);
  cudaStream_t s = h->slots[0].stream;
  int ow = 0, oh = 0;
  jpeg_oriented_size(img, &ow, &oh);
  if (!grow(h, &h->d_jframe, &h->jframe_cap, (size_t)ow * oh * 3)) return FDT_ERR_CUDA;
  const int launches = jpeg_decode_device(h, img, h->d_jframe, s);
  if (launches < 0) return FDT_ERR_CUDA;
  h->jpeg_launches = launches;
  if (!cuda_ok(h, cudaStreamSynchronize(s), "jpeg decode")) return FDT_ERR_CUDA;   // the coefficient vectors die with this frame
  *w = ow; *hh = oh;
  h->jw = ow; h->jh = oh;
  return FDT_OK;
}

// fdt_detect_jpeg_batch on one replica.  The host parses and Huffman-decodes the images in waves of one image per thread;
// the device decodes each into h->d_jarena (packed BGR at kStageAlign-aligned offsets); a chunk of arena frames (max_batch
// images, max_batch * kStageBytesPerFrame bytes) then runs through detect_frames_single as device frames.  The host decode of
// the next chunk does not overlap the device work of this one.
int jpeg_batch_single(fdt_handle* h, const uint8_t* const* images, const size_t* sizes, int n, int mode, fdt_face* out_faces,
                      int32_t* out_counts, float* out_mesh, float* out_iris, int32_t* out_wh, int32_t* out_status) {
  cudaSetDevice(h->cfg.device);
  cudaStream_t s = h->slots[0].stream;
  const size_t mf = (size_t)h->max_faces, budget = (size_t)h->chunk * kStageBytesPerFrame;
  long long launches = 0, h2d = 0;
  std::vector<int> idx;                       // the images in the arena, in list order
  std::vector<fdt_frame> fr;                  // their frames (data = arena offset until the chunk runs)
  size_t used = 0;
  std::vector<fdt_face> tf;                   // a chunk with failed images between its own runs into these, then scatters
  std::vector<int32_t> tc;
  std::vector<float> tm, ti;
  auto run_chunk = [&]() -> int {
    const int k = (int)idx.size();
    if (k == 0) return FDT_OK;
    if (!cuda_ok(h, cudaStreamSynchronize(s), "jpeg decode")) return FDT_ERR_CUDA;     // detection reads the arena on both slots
    for (fdt_frame& f : fr) f.data = h->d_jarena + reinterpret_cast<size_t>(f.data);
    const size_t i0 = (size_t)idx[0];
    int rc;
    if (idx.back() - idx[0] + 1 == k) {
      rc = detect_frames_single(h, fr.data(), nullptr, k, mode, FDT_MEM_DEVICE, out_faces + i0 * mf, out_counts + i0,
                                out_mesh ? out_mesh + i0 * mf * FDT_MESH_FLOATS : nullptr, out_iris ? out_iris + i0 * mf * FDT_IRIS_FLOATS : nullptr);
    } else {
      tf.resize(k * mf); tc.resize(k);
      if (out_mesh) tm.resize(k * mf * FDT_MESH_FLOATS);
      if (out_iris) ti.resize(k * mf * FDT_IRIS_FLOATS);
      rc = detect_frames_single(h, fr.data(), nullptr, k, mode, FDT_MEM_DEVICE, tf.data(), tc.data(), out_mesh ? tm.data() : nullptr,
                                out_iris ? ti.data() : nullptr);
      for (int j = 0; j < k && rc == FDT_OK; ++j) {
        const size_t i = (size_t)idx[j], c = (size_t)tc[j];
        out_counts[i] = tc[j];
        std::memcpy(out_faces + i * mf, tf.data() + j * mf, c * sizeof(fdt_face));
        if (out_mesh) std::memcpy(out_mesh + i * mf * FDT_MESH_FLOATS, tm.data() + j * mf * FDT_MESH_FLOATS, c * FDT_MESH_FLOATS * sizeof(float));
        if (out_iris) std::memcpy(out_iris + i * mf * FDT_IRIS_FLOATS, ti.data() + j * mf * FDT_IRIS_FLOATS, c * FDT_IRIS_FLOATS * sizeof(float));
      }
    }
    launches += h->launches; h2d += h->h2d_bytes;
    idx.clear(); fr.clear(); used = 0;
    return rc;
  };
  const int nth = std::max(1, std::min(n, (int)std::thread::hardware_concurrency()));
  std::vector<JpegImage> imgs(nth);
  std::vector<JpegStatus> st(nth);
  for (int w0 = 0; w0 < n; w0 += nth) {
    const int m = std::min(nth, n - w0);
    {
      // jpeg_decode_coefficients keeps no state between calls: one image per thread
      std::vector<std::thread> pool;
      for (int t = 0; t < m; ++t)
        pool.emplace_back([&, t] {
          const int i = w0 + t;
          std::string e;
          imgs[t] = JpegImage();
          st[t] = (!images[i] || sizes[i] == 0) ? kJpegBad : jpeg_decode_coefficients(images[i], sizes[i], &imgs[t], &e);
        });
      for (auto& t : pool) t.join();
    }
    for (int t = 0; t < m; ++t) {
      const int i = w0 + t;
      out_counts[i] = 0;
      if (out_wh) { out_wh[2 * i] = 0; out_wh[2 * i + 1] = 0; }
      if (st[t] != kJpegOk) { out_status[i] = st[t] == kJpegBad ? FDT_ERR_FORMAT : FDT_ERR_UNSUPPORTED; continue; }
      int ow = 0, oh = 0;
      jpeg_oriented_size(imgs[t], &ow, &oh);
      const size_t fb = (size_t)ow * oh * 3;
      if (!idx.empty() && ((int)idx.size() == h->chunk || align_up(used, kStageAlign) + fb > budget))
        if (int rc = run_chunk()) return rc;
      const size_t pos = align_up(used, kStageAlign);
      if (pos + fb > h->jarena_cap) {
        // grow, keeping the frames already decoded into the arena
        const size_t want = std::max(pos + fb, std::min(budget, 2 * h->jarena_cap));
        uint8_t* p = nullptr;
        if (!cuda_ok(h, cudaMalloc(&p, want), "cudaMalloc(jpeg arena)")) return FDT_ERR_CUDA;
        if (used) cudaMemcpyAsync(p, h->d_jarena, used, cudaMemcpyDeviceToDevice, s);
        if (!cuda_ok(h, cudaStreamSynchronize(s), "jpeg arena")) { cudaFree(p); return FDT_ERR_CUDA; }
        if (h->d_jarena) cudaFree(h->d_jarena);
        h->d_jarena = p; h->jarena_cap = want;
      }
      h->h2d_bytes = 0;
      const int l = jpeg_decode_device(h, imgs[t], h->d_jarena + pos, s);
      if (l < 0) return FDT_ERR_CUDA;
      launches += l; h2d += h->h2d_bytes;
      fdt_frame f;
      f.data = reinterpret_cast<const uint8_t*>(pos); f.width = ow; f.height = oh; f.row_stride = ow * 3; f.mat_type = FDT_MAT_8UC3;
      idx.push_back(i); fr.push_back(f);
      used = pos + fb;
      out_status[i] = FDT_OK;
      if (out_wh) { out_wh[2 * i] = ow; out_wh[2 * i + 1] = oh; }
    }
  }
  const int rc = run_chunk();
  h->launches = launches; h->h2d_bytes = h2d;
  return rc;
}
}  // namespace


extern "C" {

void fdt_default_config(fdt_config* cfg) {
  if (!cfg) return;
  std::memset(cfg, 0, sizeof(*cfg));
  cfg->struct_size = (int32_t)sizeof(fdt_config);
  cfg->model = FDT_MODEL_BACK_CAMERA;   // FaceDetector.create default (lib/src/face_detector.dart:85)
  cfg->device = 0;
  cfg->max_batch = 0;
  cfg->max_faces = 0;
  cfg->fuse_level = -1;
  cfg->min_score = 0.0;
  cfg->min_face_size = 0.0;
  cfg->min_face_presence = 0.5;         // kDefaultMinFacePresenceConfidence
}

int32_t fdt_destroy(fdt_handle* h);

int32_t fdt_create_ex(const fdt_config* cfg_in, const uint8_t* det_tflite, size_t det_len, const uint8_t* mesh_tflite,
                      size_t mesh_len, const uint8_t* iris_tflite, size_t iris_len, const int32_t* devices, int32_t num_devices,
                      fdt_handle** out) {
  if (!out) return fail(nullptr, FDT_ERR_BAD_ARG, "null out pointer");
  *out = nullptr;
  fdt_config cfg;
  fdt_default_config(&cfg);
  if (cfg_in) {
    if (cfg_in->struct_size != (int32_t)sizeof(fdt_config)) return fail(nullptr, FDT_ERR_BAD_ARG, "fdt_config.struct_size mismatch");
    cfg = *cfg_in;
  }
  // validateFaceGates (lib/src/shared/face_gates.dart:31-59)
  auto bad = [](double v) { return std::isnan(v) || v < 0.0 || v > 1.0; };
  if (bad(cfg.min_score)) return fail(nullptr, FDT_ERR_BAD_ARG, "minScore must be in the inclusive range [0.0, 1.0]");
  if (bad(cfg.min_face_size)) return fail(nullptr, FDT_ERR_BAD_ARG, "minFaceSize must be in the inclusive range [0.0, 1.0]");
  if (bad(cfg.min_face_presence)) return fail(nullptr, FDT_ERR_BAD_ARG, "minFacePresenceConfidence must be in the inclusive range [0.0, 1.0]");
  if (cfg.model < FDT_MODEL_FRONT_CAMERA || cfg.model > FDT_MODEL_FULL_SPARSE) return fail(nullptr, FDT_ERR_BAD_ARG, "unknown model");
  if (cfg.model == FDT_MODEL_FULL_SPARSE) return fail(nullptr, FDT_ERR_UNSUPPORTED, "fullSparse (DENSIFY) is outside this path");
  if (!det_tflite || det_len == 0) return fail(nullptr, FDT_ERR_BAD_ARG, "missing detector model bytes");
  if (iris_tflite && iris_len && !(mesh_tflite && mesh_len)) return fail(nullptr, FDT_ERR_BAD_ARG, "the iris model needs the face_landmark model");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
    return fail(nullptr, FDT_ERR_CUDA, "no CUDA device: libfdt_cuda has no CPU fallback");
  if (num_devices < 0 || (num_devices > 0 && !devices)) return fail(nullptr, FDT_ERR_BAD_ARG, "bad device list");
  if (num_devices <= 1) {
    if (num_devices == 1) cfg.device = devices[0];
    if (cfg.device < 0 || cfg.device >= ndev) return fail(nullptr, FDT_ERR_BAD_ARG, "bad device ordinal");
    return create_single(cfg, det_tflite, det_len, mesh_tflite, mesh_len, iris_tflite, iris_len, out);
  }
  for (int i = 0; i < num_devices; ++i) {
    if (devices[i] < 0 || devices[i] >= ndev) return fail(nullptr, FDT_ERR_BAD_ARG, "bad device ordinal in the device list");
    for (int j = 0; j < i; ++j) if (devices[j] == devices[i]) return fail(nullptr, FDT_ERR_BAD_ARG, "duplicate device in the device list");
  }
  fdt_handle* parent = new fdt_handle();
  parent->cfg = cfg;
  for (int i = 0; i < num_devices; ++i) {
    fdt_config c = cfg;
    c.device = devices[i];
    fdt_handle* sh = nullptr;
    int rc = create_single(c, det_tflite, det_len, mesh_tflite, mesh_len, iris_tflite, iris_len, &sh);
    if (rc != FDT_OK) { fdt_destroy(parent); return rc; }
    parent->shards.push_back(sh);
  }
  parent->chunk = parent->shards[0]->chunk; parent->max_faces = parent->shards[0]->max_faces;
  parent->has_mesh = parent->shards[0]->has_mesh; parent->has_iris = parent->shards[0]->has_iris;
  parent->num_anchors = parent->shards[0]->num_anchors;
  parent->ready = true;
  *out = parent;
  return FDT_OK;
}

int32_t fdt_create(const fdt_config* cfg, const uint8_t* det_tflite, size_t det_len, const uint8_t* mesh_tflite, size_t mesh_len,
                   fdt_handle** out) {
  return fdt_create_ex(cfg, det_tflite, det_len, mesh_tflite, mesh_len, nullptr, 0, nullptr, 0, out);
}

}  // extern "C"

namespace {

int create_single(const fdt_config& cfg, const uint8_t* det_tflite, size_t det_len, const uint8_t* mesh_tflite, size_t mesh_len,
                  const uint8_t* iris_tflite, size_t iris_len, fdt_handle** out) {
  if (cudaSetDevice(cfg.device) != cudaSuccess) return fail(nullptr, FDT_ERR_CUDA, "cudaSetDevice failed");
  // The kernels are sm_100a code (tcgen05 / TMEM / TMA): refuse any other GPU here instead of at the first launch.
  int cc_major = 0, smem_optin = 0;
  cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, cfg.device);
  cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, cfg.device);
  if (cc_major != 10 || smem_optin < 227 * 1024)
    return fail(nullptr, FDT_ERR_CUDA, "libfdt_cuda is built for sm_100a (B200): device " + std::to_string(cfg.device) + " has compute capability major " +
                                       std::to_string(cc_major));
  fdt_handle* h = new fdt_handle();
  h->cfg = cfg;
  h->chunk = cfg.max_batch > 0 ? cfg.max_batch : 256;
  h->max_faces = cfg.max_faces > 0 ? std::min(cfg.max_faces, (int)FDT_MAX_FACES) : FDT_MAX_FACES;
  int fuse = cfg.fuse_level < 0 ? 1 : cfg.fuse_level;
  std::string err;
  auto bail = [&](int code, const std::string& m) {
    fail(nullptr, code, m);
    fdt_destroy(h);
    return code;
  };
  if (!h->det.init(det_tflite, det_len, fuse, &err)) return bail(FDT_ERR_MODEL, "detector model: " + err);
  SsdOptions so = ssd_options(cfg.model);
  if (h->det.in_h() != so.input_h || h->det.in_w() != so.input_w)
    return bail(FDT_ERR_MODEL, "detector input size does not match the selected FaceDetectionModel");
  h->anchors = generate_anchors(so);
  h->num_anchors = (int)h->anchors.size() / 2;
  const Plan& dp = h->det.plan();
  if (dp.out_elems.size() < 2 || dp.out_elems[0] != (long long)h->num_anchors * 16 || dp.out_elems[1] != h->num_anchors)
    return bail(FDT_ERR_MODEL, "detector outputs do not match [N,16] boxes / [N] scores for the SSD anchors");
  h->d_anchors = dev_upload(h->anchors);
  if (!h->d_anchors) return bail(FDT_ERR_CUDA, "anchor upload failed");
  h->cand_cap = h->num_anchors;
  const bool with_mesh = mesh_tflite && mesh_len, with_iris = with_mesh && iris_tflite && iris_len;
  if (with_mesh) {
    if (!h->mesh.init(mesh_tflite, mesh_len, fuse, &err)) return bail(FDT_ERR_MODEL, "mesh model: " + err);
    if (h->mesh.in_h() != kMeshInput || h->mesh.in_w() != kMeshInput) return bail(FDT_ERR_MODEL, "mesh model input must be 192x192");
    bool has3 = false, has1 = false;
    for (long long e : h->mesh.plan().out_elems) { has3 |= (e == FDT_MESH_FLOATS); has1 |= (e == 1); }
    if (!has3 || !has1) return bail(FDT_ERR_MODEL, "mesh model must output 1404 landmarks and a face flag");
    h->mesh_cap = std::max(64, h->chunk * 2);
  }
  if (with_iris) {
    if (!h->iris.init(iris_tflite, iris_len, fuse, &err)) return bail(FDT_ERR_MODEL, "iris model: " + err);
    if (h->iris.in_h() != kIrisInput || h->iris.in_w() != kIrisInput) return bail(FDT_ERR_MODEL, "iris model input must be 64x64");
    bool hc = false, hi = false;
    for (long long e : h->iris.plan().out_elems) { hc |= (e == 213); hi |= (e == 15); }
    if (!hc || !hi) return bail(FDT_ERR_MODEL, "iris model must output 71 contour points and 5 iris points");
  }
  for (int i = 0; i < kSlots; ++i) {
    Slot& sl = h->slots[i];
    if (cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking) != cudaSuccess) return bail(FDT_ERR_CUDA, "stream creation failed");
    if (cudaEventCreateWithFlags(&sl.ev_det, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&sl.ev_blob, cudaEventDisableTiming) != cudaSuccess) return bail(FDT_ERR_CUDA, "event creation failed");
    if (!h->det.make_ctx(h->chunk, &sl.det_ctx, &err)) return bail(FDT_ERR_CUDA, err);
    bool ok = dalloc(h, &sl.d_lb, (size_t)h->chunk * h->det.in_h() * h->det.in_w() * 4) &&     // BGRX
              dalloc(h, &sl.d_cand_idx, (size_t)h->chunk * h->cand_cap) && dalloc(h, &sl.d_cand_n, (size_t)h->chunk) &&
              palloc(h, &sl.h_counts, (size_t)h->chunk) && palloc(h, &sl.h_faces, (size_t)h->chunk * h->max_faces) &&
              dalloc(h, &sl.d_pf, 1) && palloc(h, &sl.h_pf, 1);
    if (!ok) return bail(FDT_ERR_CUDA, "detector stage allocation failed");
    cudaMemset(sl.d_cand_n, 0, (size_t)h->chunk * sizeof(int));
    if (with_mesh) {
      const size_t mc = (size_t)h->mesh_cap;
      if (!h->mesh.make_ctx(h->mesh_cap, &sl.mesh_ctx, &err)) return bail(FDT_ERR_CUDA, err);
      ok = dalloc(h, &sl.d_crop_img, mc) && palloc(h, &sl.h_crop_img, mc) && dalloc(h, &sl.d_affine, mc * 6) && palloc(h, &sl.h_affine, mc * 6) &&
           dalloc(h, &sl.d_roi, mc * 6) && palloc(h, &sl.h_roi, mc * 6) && dalloc(h, &sl.d_crops, mc * kMeshInput * kMeshInput * 4) &&
           dalloc(h, &sl.d_mesh_out, mc * FDT_MESH_FLOATS) && palloc(h, &sl.h_mesh_out, mc * FDT_MESH_FLOATS) &&
           dalloc(h, &sl.d_mesh_score, mc) && palloc(h, &sl.h_mesh_score, mc) && dalloc(h, &sl.d_eye_corners, mc * 8) &&
           palloc(h, &sl.h_eye_corners, mc * 8);
      if (!ok) return bail(FDT_ERR_CUDA, "mesh stage allocation failed");
    }
    if (with_iris) {
      const size_t ec = (size_t)h->mesh_cap * 2;
      if (!h->iris.make_ctx((int)ec, &sl.iris_ctx, &err)) return bail(FDT_ERR_CUDA, err);
      ok = dalloc(h, &sl.d_eye_img, ec) && palloc(h, &sl.h_eye_img, ec) && dalloc(h, &sl.d_eye_affine, ec * 6) && palloc(h, &sl.h_eye_affine, ec * 6) &&
           dalloc(h, &sl.d_eye_roi, ec * 6) && palloc(h, &sl.h_eye_roi, ec * 6) && dalloc(h, &sl.d_eye_crops, ec * kIrisInput * kIrisInput * 4) &&
           dalloc(h, &sl.d_iris_out, (ec / 2) * FDT_IRIS_FLOATS) && palloc(h, &sl.h_iris_out, (ec / 2) * FDT_IRIS_FLOATS) &&
           dalloc(h, &sl.d_eye_kp, (ec / 2) * 4) && palloc(h, &sl.h_eye_kp, (ec / 2) * 4) &&
           dalloc(h, &sl.d_eye_wh, ec) && palloc(h, &sl.h_eye_wh, ec);
      if (!ok) return bail(FDT_ERR_CUDA, "iris stage allocation failed");
    }
  }
  h->has_mesh = with_mesh; h->has_iris = with_iris;
  h->crop_cap = std::max(64, h->chunk * 2);
  cudaEventCreate(&h->ev[0]);
  cudaEventCreate(&h->ev[1]);
  for (int i = 0; i < 3; ++i) cudaEventCreate(&h->tev[i]);
  if (cudaDeviceSynchronize() != cudaSuccess) return bail(FDT_ERR_CUDA, "device initialisation failed");
  h->ready = true;
  *out = h;
  return FDT_OK;
}

}  // namespace

extern "C" {

int32_t fdt_destroy(fdt_handle* h) {
  if (!h) return FDT_OK;
  if (!h->shards.empty()) {
    for (fdt_handle* sh : h->shards) fdt_destroy(sh);
    delete h;
    return FDT_OK;
  }
  {
    std::lock_guard<std::mutex> g(h->mu);
    h->ready = false;
    cudaSetDevice(h->cfg.device);
    cudaDeviceSynchronize();
    for (int i = 0; i < kSlots; ++i) {
      Slot& sl = h->slots[i];
      h->det.free_ctx(&sl.det_ctx);
      h->mesh.free_ctx(&sl.mesh_ctx);
      h->iris.free_ctx(&sl.iris_ctx);
      if (sl.d_frames) cudaFree(sl.d_frames);
      if (sl.stream) cudaStreamDestroy(sl.stream);
      if (sl.ev_det) cudaEventDestroy(sl.ev_det);
      if (sl.ev_blob) cudaEventDestroy(sl.ev_blob);
      if (sl.ev_fc) cudaEventDestroy(sl.ev_fc);
      if (sl.h_blob) cudaFreeHost(sl.h_blob);
      if (sl.d_blob) cudaFree(sl.d_blob);
    }
    for (void* p : h->dev_allocs) cudaFree(p);
    if (h->d_jcoef) cudaFree(h->d_jcoef);
    if (h->d_jplanes) cudaFree(h->d_jplanes);
    if (h->d_jframe) cudaFree(h->d_jframe);
    if (h->d_jq) cudaFree(h->d_jq);
    if (h->d_jarena) cudaFree(h->d_jarena);
    if (h->d_crop_arena) cudaFree(h->d_crop_arena);
    for (void* p : h->pin_allocs) cudaFreeHost(p);
    void* dev[] = {h->d_faces, h->d_counts, h->d_anchors};
    for (void* p : dev) if (p) cudaFree(p);
    for (LbTables& t : h->tables) {
      void* tp[] = {t.x0, t.x1, t.y0, t.y1, t.ax0, t.ax1, t.by0, t.by1, t.y0c, t.y1c, t.cy0, t.cy1, t.cy0c, t.cy1c};
      for (void* p : tp) if (p) cudaFree(p);
    }
    if (h->ev[0]) cudaEventDestroy(h->ev[0]);
    if (h->ev[1]) cudaEventDestroy(h->ev[1]);
    for (int i = 0; i < 3; ++i) if (h->tev[i]) cudaEventDestroy(h->tev[i]);
  }
  delete h;
  return FDT_OK;
}

int32_t fdt_detect_batch(fdt_handle* h, const uint8_t* frames, int32_t batch, int32_t width, int32_t height,
                         int32_t row_stride, int32_t mat_type, int32_t mode, int32_t mem_kind, fdt_face* out_faces,
                         int32_t* out_counts, float* out_mesh, float* out_iris) {
  return fdt_detect_batch_oriented(h, frames, batch, width, height, row_stride, mat_type, FDT_ORIENT_UPRIGHT, mode, mem_kind,
                                   out_faces, out_counts, out_mesh, out_iris);
}

int32_t fdt_detect_batch_oriented(fdt_handle* h, const uint8_t* frames, int32_t batch, int32_t width, int32_t height,
                                  int32_t row_stride, int32_t mat_type, int32_t orientation, int32_t mode, int32_t mem_kind,
                                  fdt_face* out_faces, int32_t* out_counts, float* out_mesh, float* out_iris) {
  if (!h) return fail(nullptr, FDT_ERR_NOT_READY, "null handle");
  std::lock_guard<std::mutex> g(h->mu);
  reset_crops(h);
  if (orientation < 1 || orientation > 8) return fail(h, FDT_ERR_BAD_ARG, "orientation must be an EXIF value 1..8");
  return detect_impl(h, frames, batch, width, height, row_stride, mat_type, mode, mem_kind, out_faces, out_counts, out_mesh, out_iris,
                     false, orientation);
}

int32_t fdt_detect_one(fdt_handle* h, const uint8_t* bytes, size_t nbytes, int32_t width, int32_t height, int32_t mat_type,
                       int32_t mode, fdt_face* out_faces, int32_t* out_count, float* out_mesh, float* out_iris) {
  if (!h) return fail(nullptr, FDT_ERR_NOT_READY, "null handle");
  std::lock_guard<std::mutex> g(h->mu);
  reset_crops(h);
  if (width <= 0 || height <= 0) return fail(h, FDT_ERR_BAD_ARG, "bad frame arguments");
  const int row_stride = width * row_step(mat_type);
  FrameLayout lay;
  const char* msg = nullptr;
  if (int rc = frame_layout(mat_type, width, height, row_stride, &lay, &msg)) return fail(h, rc, msg);
  // matFromPackedBytes length check (lib/src/util/helpers.dart:440-447); YUV: width * height * 3 / 2; planar RGB: 3 * width * height
  if (nbytes != (size_t)lay.frame_bytes) return fail(h, FDT_ERR_SIZE_MISMATCH, "bytes length does not equal the frame size (width * height * channels)");
  return detect_impl(h, bytes, 1, width, height, row_stride, mat_type, mode, FDT_MEM_HOST, out_faces, out_count, out_mesh, out_iris, false);
}

int32_t fdt_detect_batch_device(fdt_handle* h, const uint8_t* d_frames, int32_t batch, int32_t width, int32_t height,
                                int32_t row_stride, int32_t mat_type, int32_t mode, const fdt_face** d_faces,
                                const int32_t** d_counts) {
  if (!h) return fail(nullptr, FDT_ERR_NOT_READY, "null handle");
  std::lock_guard<std::mutex> g(h->mu);
  reset_crops(h);
  if (h->crops_on) return fail(h, FDT_ERR_UNSUPPORTED, "face crops need the results on the host: fdt_set_face_crops(h, NULL) first");
  int rc = detect_impl(h, d_frames, batch, width, height, row_stride, mat_type, mode, FDT_MEM_DEVICE, nullptr, nullptr, nullptr, nullptr, true);
  if (rc == FDT_OK) {
    if (d_faces) *d_faces = h->d_faces;
    if (d_counts) *d_counts = h->d_counts;
  }
  return rc;
}

int32_t fdt_decode_jpeg(fdt_handle* h, const uint8_t* bytes, size_t nbytes, uint8_t* out_bgr, size_t out_capacity, int32_t* out_wh) {
  if (!h) return fail(nullptr, FDT_ERR_NOT_READY, "null handle");
  std::lock_guard<std::mutex> g(h->mu);
  fdt_handle* p = primary(h);
  if (!p->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  int w = 0, hh = 0;
  int rc = jpeg_to_device(p, bytes, nbytes, &w, &hh);
  if (rc != FDT_OK) { if (p != h) h->err = p->err; return rc; }
  if (out_wh) { out_wh[0] = w; out_wh[1] = hh; }
  if (out_bgr) {
    if (out_capacity < (size_t)w * hh * 3) return fail(h, FDT_ERR_SIZE_MISMATCH, "output buffer smaller than width * height * 3");
    if (!cuda_ok(h, cudaMemcpy(out_bgr, p->d_jframe, (size_t)w * hh * 3, cudaMemcpyDeviceToHost), "jpeg frame download")) return FDT_ERR_CUDA;
  }
  return FDT_OK;
}

int32_t fdt_get_decoded_frame(fdt_handle* h, uint8_t* out_bgr, size_t out_capacity) {
  if (!h) return fail(nullptr, FDT_ERR_NOT_READY, "null handle");
  std::lock_guard<std::mutex> g(h->mu);
  fdt_handle* p = primary(h);
  if (!p->ready || !p->d_jframe || p->jw <= 0) return fail(h, FDT_ERR_NOT_READY, "no decoded frame");
  if (!out_bgr || out_capacity < (size_t)p->jw * p->jh * 3) return fail(h, FDT_ERR_SIZE_MISMATCH, "output buffer smaller than width * height * 3");
  cudaSetDevice(p->cfg.device);
  if (!cuda_ok(h, cudaMemcpy(out_bgr, p->d_jframe, (size_t)p->jw * p->jh * 3, cudaMemcpyDeviceToHost), "jpeg frame download")) return FDT_ERR_CUDA;
  return FDT_OK;
}

int32_t fdt_detect_jpeg(fdt_handle* h, const uint8_t* bytes, size_t nbytes, int32_t mode, fdt_face* out_faces, int32_t* out_count,
                        float* out_mesh, float* out_iris, int32_t* out_wh) {
  if (!h) return fail(nullptr, FDT_ERR_NOT_READY, "null handle");
  std::lock_guard<std::mutex> g(h->mu);
  reset_crops(h);
  fdt_handle* p = primary(h);
  if (!p->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  int w = 0, hh = 0;
  int rc = jpeg_to_device(p, bytes, nbytes, &w, &hh);
  if (rc == FDT_OK) {
    if (out_wh) { out_wh[0] = w; out_wh[1] = hh; }
    const long long jl = p->jpeg_launches;
    rc = detect_single(p, p->d_jframe, 1, w, hh, w * 3, FDT_MAT_8UC3, 1, mode, FDT_MEM_DEVICE, out_faces, out_count, out_mesh, out_iris, false);
    p->launches += jl;
  }
  if (p != h) { h->err = p->err; h->launches = p->launches; h->h2d_bytes = p->h2d_bytes; }
  return rc;
}

int32_t fdt_detect_frames(fdt_handle* h, const fdt_frame* frames, int32_t n, int32_t mode, int32_t mem_kind, fdt_face* out_faces,
                          int32_t* out_counts, float* out_mesh, float* out_iris) {
  return fdt_detect_frames_oriented(h, frames, nullptr, n, mode, mem_kind, out_faces, out_counts, out_mesh, out_iris);
}

int32_t fdt_detect_frames_oriented(fdt_handle* h, const fdt_frame* frames, const int32_t* orientations, int32_t n, int32_t mode,
                                   int32_t mem_kind, fdt_face* out_faces, int32_t* out_counts, float* out_mesh, float* out_iris) {
  if (!h) return fail(nullptr, FDT_ERR_NOT_READY, "null handle");
  std::lock_guard<std::mutex> g(h->mu);
  reset_crops(h);
  if (!h->shards.empty()) return detect_frames_multi(h, frames, orientations, n, mode, mem_kind, out_faces, out_counts, out_mesh, out_iris);
  return detect_frames_single(h, frames, orientations, n, mode, mem_kind, out_faces, out_counts, out_mesh, out_iris);
}

int32_t fdt_detect_yuv_planes(fdt_handle* h, const fdt_yuv_planes* frames, const int32_t* orientations, int32_t n, int32_t mode,
                              int32_t mem_kind, fdt_face* out_faces, int32_t* out_counts, float* out_mesh, float* out_iris) {
  if (!h) return fail(nullptr, FDT_ERR_NOT_READY, "null handle");
  std::lock_guard<std::mutex> g(h->mu);
  reset_crops(h);
  if (!h->shards.empty()) return detect_planes_multi(h, frames, orientations, n, mode, mem_kind, out_faces, out_counts, out_mesh, out_iris);
  return detect_frames_single(h, nullptr, orientations, n, mode, mem_kind, out_faces, out_counts, out_mesh, out_iris,
                              FrameList::kYuvPlanes, frames);
}

int32_t fdt_detect_yuv_planes16(fdt_handle* h, const fdt_yuv_planes* frames, const int32_t* orientations, int32_t n,
                                int32_t sample_bits, int32_t mode, int32_t mem_kind, fdt_face* out_faces, int32_t* out_counts,
                                float* out_mesh, float* out_iris) {
  if (!h) return fail(nullptr, FDT_ERR_NOT_READY, "null handle");
  std::lock_guard<std::mutex> g(h->mu);
  reset_crops(h);
  if (sample_bits != 10 && sample_bits != 12 && sample_bits != 16) return fail(h, FDT_ERR_BAD_ARG, "sample_bits must be 10, 12 or 16");
  if (!h->shards.empty())
    return detect_planes_multi(h, frames, orientations, n, mode, mem_kind, out_faces, out_counts, out_mesh, out_iris, sample_bits);
  return detect_frames_single(h, nullptr, orientations, n, mode, mem_kind, out_faces, out_counts, out_mesh, out_iris,
                              FrameList::kYuvPlanes, frames, sample_bits);
}

int32_t fdt_detect_jpeg_batch(fdt_handle* h, const uint8_t* const* images, const size_t* sizes, int32_t n, int32_t mode,
                              fdt_face* out_faces, int32_t* out_counts, float* out_mesh, float* out_iris, int32_t* out_wh,
                              int32_t* out_status) {
  if (!h) return fail(nullptr, FDT_ERR_NOT_READY, "null handle");
  std::lock_guard<std::mutex> g(h->mu);
  reset_crops(h);
  if (!h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  if (n < 0 || (n > 0 && (!images || !sizes || !out_faces || !out_counts || !out_status))) return fail(h, FDT_ERR_BAD_ARG, "bad image list");
  if (int rc = check_mode(h, mode)) return rc;
  h->launches = 0; h->h2d_bytes = 0;
  if (n == 0) return FDT_OK;
  if (h->shards.empty()) return jpeg_batch_single(h, images, sizes, n, mode, out_faces, out_counts, out_mesh, out_iris, out_wh, out_status);
  return on_shards(h, n, [=](fdt_handle* sh, int lo, int hi) {
    const size_t mf = (size_t)sh->max_faces;
    return jpeg_batch_single(sh, images + lo, sizes + lo, hi - lo, mode, out_faces + lo * mf, out_counts + lo,
                             out_mesh ? out_mesh + lo * mf * FDT_MESH_FLOATS : nullptr,
                             out_iris ? out_iris + lo * mf * FDT_IRIS_FLOATS : nullptr, out_wh ? out_wh + 2 * lo : nullptr, out_status + lo);
  });
}

int32_t fdt_host_jpeg_info(const uint8_t* bytes, size_t nbytes, int32_t* info8) {
  JpegImage img;
  std::string e;
  const JpegStatus st = jpeg_decode_coefficients(bytes, nbytes, &img, &e);
  if (st != kJpegOk) { std::lock_guard<std::mutex> g(g_create_mu); g_create_error = e; return st == kJpegBad ? FDT_ERR_FORMAT : FDT_ERR_UNSUPPORTED; }
  if (info8) {
    info8[0] = img.width; info8[1] = img.height; info8[2] = img.ncomp; info8[3] = img.progressive ? 1 : 0;
    info8[4] = img.orientation; info8[5] = img.hmax; info8[6] = img.vmax; info8[7] = 0;
  }
  return FDT_OK;
}

int32_t fdt_host_jpeg_coefficients(const uint8_t* bytes, size_t nbytes, int32_t comp, int16_t* out, size_t capacity, int32_t* dims6, uint16_t* qt64) {
  JpegImage img;
  std::string e;
  const JpegStatus st = jpeg_decode_coefficients(bytes, nbytes, &img, &e);
  if (st != kJpegOk) { std::lock_guard<std::mutex> g(g_create_mu); g_create_error = e; return st == kJpegBad ? FDT_ERR_FORMAT : FDT_ERR_UNSUPPORTED; }
  if (comp < 0 || comp >= img.ncomp) return FDT_ERR_BAD_ARG;
  const JpegComp& c = img.comp[comp];
  if (dims6) { dims6[0] = c.bw; dims6[1] = c.bh; dims6[2] = c.dw; dims6[3] = c.dh; dims6[4] = c.h; dims6[5] = c.v; }
  if (qt64) std::memcpy(qt64, img.qt[c.tq], 64 * sizeof(uint16_t));
  if (out) {
    if (capacity < c.coef.size()) return FDT_ERR_SIZE_MISMATCH;
    std::memcpy(out, c.coef.data(), c.coef.size() * sizeof(int16_t));
  }
  return FDT_OK;
}

int32_t fdt_synchronize(fdt_handle* h) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  std::lock_guard<std::mutex> g(h->mu);
  if (!h->shards.empty()) {
    for (fdt_handle* sh : h->shards) { int rc = fdt_synchronize(sh); if (rc != FDT_OK) return rc; }
    return FDT_OK;
  }
  cudaSetDevice(h->cfg.device);
  for (int i = 0; i < kSlots; ++i)
    if (!cuda_ok(h, cudaStreamSynchronize(h->slots[i].stream), "synchronize")) return FDT_ERR_CUDA;
  return FDT_OK;
}

int32_t fdt_num_devices(fdt_handle* h) { return !h ? 0 : (h->shards.empty() ? 1 : (int32_t)h->shards.size()); }

int32_t fdt_get_info(fdt_handle* h, int32_t* input_w, int32_t* input_h, int32_t* num_anchors, int32_t* max_faces, int32_t* max_batch) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  fdt_handle* p = primary(h);
  if (input_w) *input_w = p->det.in_w();
  if (input_h) *input_h = p->det.in_h();
  if (num_anchors) *num_anchors = p->num_anchors;
  if (max_faces) *max_faces = p->max_faces;
  if (max_batch) *max_batch = p->chunk;
  return FDT_OK;
}

int32_t fdt_get_anchors(fdt_handle* h, double* out_xy) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  if (!out_xy) return fail(h, FDT_ERR_BAD_ARG, "null output");
  fdt_handle* p = primary(h);
  std::memcpy(out_xy, p->anchors.data(), p->anchors.size() * sizeof(double));
  return FDT_OK;
}

int32_t fdt_letterbox_params(int32_t src_w, int32_t src_h, int32_t dst_w, int32_t dst_h, int32_t* out6) {
  if (!out6 || src_w <= 0 || src_h <= 0 || dst_w <= 0 || dst_h <= 0) return FDT_ERR_BAD_ARG;
  LetterboxParams p = letterbox_params(src_w, src_h, dst_w, dst_h);
  out6[0] = p.new_w; out6[1] = p.new_h; out6[2] = p.pad_top; out6[3] = p.pad_bottom; out6[4] = p.pad_left; out6[5] = p.pad_right;
  return FDT_OK;
}

int32_t fdt_alloc_pinned(size_t nbytes, void** out) {
  if (!out) return FDT_ERR_BAD_ARG;
  // portable: usable by every device of a multi-device handle
  return cudaHostAlloc(out, nbytes, cudaHostAllocPortable) == cudaSuccess ? FDT_OK : FDT_ERR_CUDA;
}
int32_t fdt_free_pinned(void* p) { return cudaFreeHost(p) == cudaSuccess ? FDT_OK : FDT_ERR_CUDA; }

int32_t fdt_alloc_device(fdt_handle* h, size_t nbytes, void** out) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  if (!out) return fail(h, FDT_ERR_BAD_ARG, "null out pointer");
  cudaSetDevice(primary(h)->cfg.device);
  return cuda_ok(h, cudaMalloc(out, nbytes), "cudaMalloc") ? FDT_OK : FDT_ERR_CUDA;
}
int32_t fdt_free_device(fdt_handle* h, void* p) {
  if (!h) return FDT_ERR_NOT_READY;
  cudaSetDevice(primary(h)->cfg.device);
  return cudaFree(p) == cudaSuccess ? FDT_OK : FDT_ERR_CUDA;
}
int32_t fdt_copy_to_device(fdt_handle* h, void* dst, const void* src, size_t nbytes) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  cudaSetDevice(primary(h)->cfg.device);
  return cuda_ok(h, cudaMemcpy(dst, src, nbytes, cudaMemcpyHostToDevice), "cudaMemcpy") ? FDT_OK : FDT_ERR_CUDA;
}

int32_t fdt_copy_to_host(fdt_handle* h, void* dst, const void* src, size_t nbytes) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  fdt_handle* p = primary(h);
  cudaSetDevice(p->cfg.device);
  for (int i = 0; i < kSlots; ++i) cudaStreamSynchronize(p->slots[i].stream);
  return cuda_ok(h, cudaMemcpy(dst, src, nbytes, cudaMemcpyDeviceToHost), "cudaMemcpy") ? FDT_OK : FDT_ERR_CUDA;
}

// ---- parity taps ------------------------------------------------------------------------------
static void unpack_bgrx(const std::vector<uint8_t>& tmp, size_t px, uint8_t* out) {
  for (size_t i = 0; i < px; ++i) { out[3 * i] = tmp[4 * i]; out[3 * i + 1] = tmp[4 * i + 1]; out[3 * i + 2] = tmp[4 * i + 2]; }
}

// The letterbox, input-tensor, raw-head and detector-tensor taps read slot 0's buffers.  A call of three or more chunks
// ran its third chunk there, so those buffers no longer describe its first chunk (the candidate tap has buffers of its own).
static int32_t check_first_chunk_tap(fdt_handle* h, int32_t n) {
  if (!h->slot0_first_chunk)
    return fail(h, FDT_ERR_BAD_ARG, "the last call ran more than two chunks, so a later chunk overwrote its first chunk's buffers");
  if (n < 0 || n > h->last_first_chunk) return fail(h, FDT_ERR_BAD_ARG, "n exceeds the last call's first chunk");
  return FDT_OK;
}

int32_t fdt_debug_get_letterboxed(fdt_handle* h, int32_t n, uint8_t* out) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  h = primary(h);
  std::lock_guard<std::mutex> g(h->mu);
  if (!out) return fail(h, FDT_ERR_BAD_ARG, "null output buffer");
  if (int32_t rc = check_first_chunk_tap(h, n)) return rc;
  cudaSetDevice(h->cfg.device);
  size_t px = (size_t)n * h->det.in_h() * h->det.in_w();
  std::vector<uint8_t> tmp(px * 4);
  if (!cuda_ok(h, cudaMemcpy(tmp.data(), h->slots[0].d_lb, px * 4, cudaMemcpyDeviceToHost), "tap")) return FDT_ERR_CUDA;
  unpack_bgrx(tmp, px, out);
  return FDT_OK;
}

int32_t fdt_debug_get_input_tensor(fdt_handle* h, int32_t n, float* out) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  h = primary(h);
  std::lock_guard<std::mutex> g(h->mu);
  if (!out) return fail(h, FDT_ERR_BAD_ARG, "null output buffer");
  if (int32_t rc = check_first_chunk_tap(h, n)) return rc;
  cudaSetDevice(h->cfg.device);
  float* tmp = nullptr;
  size_t elems = (size_t)n * h->det.in_h() * h->det.in_w() * 3;
  if (!cuda_ok(h, cudaMalloc(&tmp, std::max<size_t>(elems, 1) * sizeof(float)), "tap alloc")) return FDT_ERR_CUDA;
  TV v;
  v.p = tmp; v.H = h->det.in_h(); v.W = h->det.in_w(); v.C = 3; v.Cs = 3; v.istride = (long long)v.H * v.W * 3;
  launch_normalize(h->slots[0].d_lb, v, n, h->slots[0].stream);
  cudaStreamSynchronize(h->slots[0].stream);
  bool ok = cuda_ok(h, cudaMemcpy(out, tmp, elems * sizeof(float), cudaMemcpyDeviceToHost), "tap");
  cudaFree(tmp);
  return ok ? FDT_OK : FDT_ERR_CUDA;
}

int32_t fdt_debug_get_raw_heads(fdt_handle* h, int32_t n, float* out_boxes, float* out_scores) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  h = primary(h);
  std::lock_guard<std::mutex> g(h->mu);
  if (int32_t rc = check_first_chunk_tap(h, n)) return rc;
  cudaSetDevice(h->cfg.device);
  const Plan& dp = h->det.plan();
  const EngineCtx& ctx = h->slots[0].det_ctx;
  bool ok = true;
  if (out_boxes) ok &= cuda_ok(h, cudaMemcpy(out_boxes, ctx.outputs[0], (size_t)n * dp.out_elems[0] * sizeof(float), cudaMemcpyDeviceToHost), "tap");
  if (out_scores) ok &= cuda_ok(h, cudaMemcpy(out_scores, ctx.outputs[1], (size_t)n * dp.out_elems[1] * sizeof(float), cudaMemcpyDeviceToHost), "tap");
  return ok ? FDT_OK : FDT_ERR_CUDA;
}

int32_t fdt_debug_get_candidates(fdt_handle* h, int32_t image, int32_t* out_indices, int32_t capacity, int32_t* out_n) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  h = primary(h);
  std::lock_guard<std::mutex> g(h->mu);
  if (image < 0 || image >= h->last_first_chunk || !out_n) return fail(h, FDT_ERR_BAD_ARG, "image exceeds the last call's first chunk");
  cudaSetDevice(h->cfg.device);
  int n = 0;
  if (!cuda_ok(h, cudaMemcpy(&n, h->slots[0].d_cand_n + image, sizeof(int), cudaMemcpyDeviceToHost), "tap")) return FDT_ERR_CUDA;
  *out_n = n;
  int m = std::min(std::min(n, capacity), h->cand_cap);
  if (out_indices && m > 0 &&
      !cuda_ok(h, cudaMemcpy(out_indices, h->slots[0].d_cand_idx + (size_t)image * h->cand_cap, (size_t)m * sizeof(int), cudaMemcpyDeviceToHost), "tap"))
    return FDT_ERR_CUDA;
  return FDT_OK;
}

int32_t fdt_debug_get_tensor(fdt_handle* h, int32_t which, int32_t tflite_tensor, int32_t n, float* out,
                             size_t out_capacity_floats, int32_t* out_dims4) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  h = primary(h);
  std::lock_guard<std::mutex> g(h->mu);
  if (which < 0 || which > 2) return fail(h, FDT_ERR_BAD_ARG, "which: 0 detector, 1 mesh, 2 iris");
  if (which == 1 && !h->has_mesh) return fail(h, FDT_ERR_NOT_READY, "no mesh model");
  if (which == 2 && !h->has_iris) return fail(h, FDT_ERR_NOT_READY, "no iris model");
  const Engine& e = which == 0 ? h->det : (which == 1 ? h->mesh : h->iris);
  const EngineCtx& ctx = which == 0 ? h->slots[0].det_ctx : (which == 1 ? h->slots[h->last_mesh_slot].mesh_ctx : h->slots[h->last_iris_slot].iris_ctx);
  const Plan& p = e.plan();
  auto it = p.tf2pt.find(tflite_tensor);
  if (it == p.tf2pt.end() || !p.tensors[it->second].materialized) return fail(h, FDT_ERR_BAD_ARG, "tensor is not materialised in this plan");
  if (p.fuse_level == 1 && p.tensors[it->second].root < 0) return fail(h, FDT_ERR_UNSUPPORTED, "activation buffers are reused at fuse_level 1; use 0 or 2");
  if (which == 0) {
    if (int32_t rc = check_first_chunk_tap(h, n)) return rc;
  } else {
    const int cap = which == 1 ? h->last_mesh_faces : 2 * h->last_iris_faces;
    if (n < 0 || n > cap) return fail(h, FDT_ERR_BAD_ARG, "n exceeds the crops of the last call's last pass");
  }
  cudaSetDevice(h->cfg.device);
  TV v = e.view(ctx, it->second);
  if (out_dims4) { out_dims4[0] = n; out_dims4[1] = v.H; out_dims4[2] = v.W; out_dims4[3] = v.C; }
  size_t need = (size_t)n * v.H * v.W * v.C;
  if (!out) return FDT_OK;
  if (out_capacity_floats < need) return fail(h, FDT_ERR_SIZE_MISMATCH, "output buffer too small");
  // strided device layout -> dense NHWC on the host
  cudaError_t ce = cudaSuccess;
  if (v.Cs == v.C) {
    ce = cudaMemcpy2D(out, (size_t)v.H * v.W * v.C * sizeof(float), v.p, (size_t)v.istride * sizeof(float),
                      (size_t)v.H * v.W * v.C * sizeof(float), n, cudaMemcpyDeviceToHost);
  } else {
    for (int b = 0; b < n && ce == cudaSuccess; ++b)
      ce = cudaMemcpy2D(out + (size_t)b * v.H * v.W * v.C, (size_t)v.C * sizeof(float), v.p + (size_t)b * v.istride,
                        (size_t)v.Cs * sizeof(float), (size_t)v.C * sizeof(float), (size_t)v.H * v.W, cudaMemcpyDeviceToHost);
  }
  return cuda_ok(h, ce, "tap") ? FDT_OK : FDT_ERR_CUDA;
}

int32_t fdt_debug_get_mesh_stage(fdt_handle* h, int32_t n, uint8_t* out_crops, float* out_raw1404, float* out_flag, int32_t* out_n) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  h = primary(h);
  std::lock_guard<std::mutex> g(h->mu);
  if (!h->has_mesh) return fail(h, FDT_ERR_NOT_READY, "no mesh model");
  if (out_n) *out_n = h->last_mesh_faces;
  n = std::min(n, h->last_mesh_faces);
  if (n <= 0) return FDT_OK;
  cudaSetDevice(h->cfg.device);
  const Slot& sl = h->slots[h->last_mesh_slot];
  const Plan& mp = h->mesh.plan();
  bool ok = true;
  if (out_crops) {
    size_t px = (size_t)n * kMeshInput * kMeshInput;
    std::vector<uint8_t> tmp(px * 4);
    ok &= cuda_ok(h, cudaMemcpy(tmp.data(), sl.d_crops, px * 4, cudaMemcpyDeviceToHost), "tap");
    unpack_bgrx(tmp, px, out_crops);
  }
  for (size_t k = 0; k < mp.out_elems.size(); ++k) {
    if (mp.out_elems[k] == FDT_MESH_FLOATS && out_raw1404)
      ok &= cuda_ok(h, cudaMemcpy(out_raw1404, sl.mesh_ctx.outputs[k], (size_t)n * FDT_MESH_FLOATS * sizeof(float), cudaMemcpyDeviceToHost), "tap");
    if (mp.out_elems[k] == 1 && out_flag)
      ok &= cuda_ok(h, cudaMemcpy(out_flag, sl.mesh_ctx.outputs[k], (size_t)n * sizeof(float), cudaMemcpyDeviceToHost), "tap");
  }
  return ok ? FDT_OK : FDT_ERR_CUDA;
}

int32_t fdt_debug_get_iris_stage(fdt_handle* h, int32_t n, uint8_t* out_crops, double* out_rois, float* out_contours, float* out_iris,
                                 int32_t* out_n) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  h = primary(h);
  std::lock_guard<std::mutex> g(h->mu);
  if (!h->has_iris) return fail(h, FDT_ERR_NOT_READY, "no iris model");
  if (out_n) *out_n = h->last_iris_faces;
  n = std::min(n, h->last_iris_faces);
  if (n <= 0) return FDT_OK;
  cudaSetDevice(h->cfg.device);
  const Slot& sl = h->slots[h->last_iris_slot];
  const Plan& ip = h->iris.plan();
  bool ok = true;
  if (out_crops) {
    size_t px = (size_t)2 * n * kIrisInput * kIrisInput;
    std::vector<uint8_t> tmp(px * 4);
    ok &= cuda_ok(h, cudaMemcpy(tmp.data(), sl.d_eye_crops, px * 4, cudaMemcpyDeviceToHost), "tap");
    unpack_bgrx(tmp, px, out_crops);
  }
  if (out_rois)
    for (int e = 0; e < 2 * n; ++e) {
      const double* r = sl.h_eye_roi + 6 * e;
      out_rois[4 * e] = r[1]; out_rois[4 * e + 1] = r[2]; out_rois[4 * e + 2] = r[3]; out_rois[4 * e + 3] = r[0];
    }
  for (size_t k = 0; k < ip.out_elems.size(); ++k) {
    if (ip.out_elems[k] == 213 && out_contours)
      ok &= cuda_ok(h, cudaMemcpy(out_contours, sl.iris_ctx.outputs[k], (size_t)2 * n * 213 * sizeof(float), cudaMemcpyDeviceToHost), "tap");
    if (ip.out_elems[k] == 15 && out_iris)
      ok &= cuda_ok(h, cudaMemcpy(out_iris, sl.iris_ctx.outputs[k], (size_t)2 * n * 15 * sizeof(float), cudaMemcpyDeviceToHost), "tap");
  }
  return ok ? FDT_OK : FDT_ERR_CUDA;
}

// ---- post-processing on caller-supplied tensors (tests) ---------------------------------------------
static int run_debug_decode(fdt_handle* h, const float* raw_boxes, const float* raw_scores, const double* anchors_xy, const double* pre,
                            int n_images, int N, double scale, double score_thresh, double iou_thresh, const double* pad4,
                            fdt_face* out_faces, int32_t* out_counts, double* out_dec, int32_t* out_ndec) {
  if (n_images <= 0 || N <= 0 || !out_faces || !out_counts) return fail(h, FDT_ERR_BAD_ARG, "bad debug decode arguments");
  if (!(score_thresh > 0.0 && score_thresh < 1.0) && !pre) return fail(h, FDT_ERR_BAD_ARG, "score_thresh must lie in (0, 1)");
  if (decode_smem_bytes(N) > 200 * 1024) return fail(h, FDT_ERR_BAD_ARG, "too many anchors for one block");
  cudaSetDevice(h->cfg.device);
  cudaStream_t s = h->slots[0].stream;
  float *d_boxes = nullptr, *d_scores = nullptr;
  double *d_anch = nullptr, *d_pre = nullptr, *d_dec = nullptr;
  fdt_face* d_faces = nullptr;
  int *d_counts = nullptr, *d_cn = nullptr, *d_ci = nullptr;
  const size_t B = (size_t)n_images;
  bool ok = true;
  auto up = [&](void** d, const void* src, size_t bytes) {
    ok = ok && cudaMalloc(d, std::max<size_t>(bytes, 16)) == cudaSuccess;
    if (ok && src) ok = cudaMemcpy(*d, src, bytes, cudaMemcpyHostToDevice) == cudaSuccess;
  };
  if (pre) {
    up((void**)&d_pre, pre, B * N * 17 * sizeof(double));
  } else {
    up((void**)&d_boxes, raw_boxes, B * N * 16 * sizeof(float));
    up((void**)&d_scores, raw_scores, B * N * sizeof(float));
    if (anchors_xy) up((void**)&d_anch, anchors_xy, (size_t)N * 2 * sizeof(double));
  }
  ok = ok && cudaMalloc(&d_faces, B * FDT_MAX_FACES * sizeof(fdt_face)) == cudaSuccess && cudaMalloc(&d_counts, B * sizeof(int)) == cudaSuccess &&
       cudaMalloc(&d_cn, B * sizeof(int)) == cudaSuccess && cudaMalloc(&d_ci, B * N * sizeof(int)) == cudaSuccess;
  if (out_dec) ok = ok && cudaMalloc(&d_dec, B * N * 18 * sizeof(double)) == cudaSuccess;
  int rc = FDT_OK;
  if (!ok) rc = fail(h, FDT_ERR_CUDA, "debug decode allocation failed");
  if (rc == FDT_OK && !pre && !anchors_xy && N != h->num_anchors) rc = fail(h, FDT_ERR_BAD_ARG, "num_anchors differs from the handle's anchor table");
  if (rc == FDT_OK) {
    DecodeP d;
    d.boxes = d_boxes; d.boxes_istride = (long long)N * 16; d.scores = d_scores; d.scores_istride = N;
    d.anchors = d_anch ? d_anch : h->d_anchors; d.N = N; d.input_h = (int)scale;
    d.raw_thresh = pre ? 0.0 : std::log(score_thresh / (1.0 - score_thresh));
    d.score_thresh = score_thresh; d.iou_thresh = iou_thresh;
    d.pad_t = pad4 ? pad4[0] : 0.0; d.pad_b = pad4 ? pad4[1] : 0.0; d.pad_l = pad4 ? pad4[2] : 0.0; d.pad_r = pad4 ? pad4[3] : 0.0;
    d.min_score = 0.0; d.min_face_size = 0.0; d.img_w = 1.0; d.img_h = 1.0; d.max_faces = FDT_MAX_FACES;
    d.faces = d_faces; d.counts = d_counts; d.cand_idx = d_ci; d.cand_cap = N; d.cand_n = d_cn;
    d.pre = d_pre; d.dbg_dec = d_dec; d.skip_roi = 1;
    launch_decode_nms(d, n_images, s);
    if (!cuda_ok(h, cudaStreamSynchronize(s), "debug decode")) rc = FDT_ERR_CUDA;
  }
  if (rc == FDT_OK) {
    ok = cudaMemcpy(out_counts, d_counts, B * sizeof(int), cudaMemcpyDeviceToHost) == cudaSuccess &&
         cudaMemcpy(out_faces, d_faces, B * FDT_MAX_FACES * sizeof(fdt_face), cudaMemcpyDeviceToHost) == cudaSuccess;
    if (out_dec) ok = ok && cudaMemcpy(out_dec, d_dec, B * N * 18 * sizeof(double), cudaMemcpyDeviceToHost) == cudaSuccess;
    if (out_ndec) ok = ok && cudaMemcpy(out_ndec, d_cn, B * sizeof(int), cudaMemcpyDeviceToHost) == cudaSuccess;
    if (!ok) rc = fail(h, FDT_ERR_CUDA, "debug decode copy failed");
  }
  void* fr[] = {d_boxes, d_scores, d_anch, d_pre, d_dec, d_faces, d_counts, d_cn, d_ci};
  for (void* p : fr) if (p) cudaFree(p);
  return rc;
}

int32_t fdt_debug_decode(fdt_handle* h, const float* raw_boxes, const float* raw_scores, const double* anchors_xy, int32_t n_images,
                         int32_t num_anchors, double scale, double score_thresh, double iou_thresh, const double* pad4,
                         fdt_face* out_faces, int32_t* out_counts, double* out_dec, int32_t* out_ndec) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  h = primary(h);
  std::lock_guard<std::mutex> g(h->mu);
  if (!raw_boxes || !raw_scores || !(scale >= 1.0)) return fail(h, FDT_ERR_BAD_ARG, "bad debug decode arguments");
  return run_debug_decode(h, raw_boxes, raw_scores, anchors_xy, nullptr, n_images, num_anchors, scale, score_thresh, iou_thresh, pad4,
                          out_faces, out_counts, out_dec, out_ndec);
}

int32_t fdt_debug_nms(fdt_handle* h, const double* dets17, int32_t n, double score_thresh, double iou_thresh, const double* pad4,
                      fdt_face* out_faces, int32_t* out_count) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  h = primary(h);
  std::lock_guard<std::mutex> g(h->mu);
  if (n == 0 && out_count) { *out_count = 0; return FDT_OK; }
  if (!dets17) return fail(h, FDT_ERR_BAD_ARG, "bad debug nms arguments");
  return run_debug_decode(h, nullptr, nullptr, nullptr, dets17, 1, n, 1.0, score_thresh, iou_thresh, pad4, out_faces, out_count, nullptr, nullptr);
}

int32_t fdt_extract_aligned_squares(fdt_handle* h, const uint8_t* frame, int32_t width, int32_t height, int32_t row_stride,
                                    int32_t mat_type, const double* rois, int32_t n, int32_t out_size, uint8_t* out_crops, int32_t* out_ok) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  h = primary(h);
  std::lock_guard<std::mutex> g(h->mu);
  const int ch = channels_of(mat_type);
  if (!frame || !rois || !out_crops || n < 0 || width <= 0 || height <= 0 || ch == 0 || out_size <= 0 || out_size > 4096)
    return fail(h, FDT_ERR_BAD_ARG, "bad crop arguments");
  if (row_stride < width * ch) return fail(h, FDT_ERR_SIZE_MISMATCH, "row_stride smaller than width * channels");
  if (n == 0) return FDT_OK;
  cudaSetDevice(h->cfg.device);
  cudaStream_t s = h->slots[0].stream;
  std::vector<double> aff((size_t)n * 6, 0.0);
  std::vector<int> img((size_t)n, 0), okv((size_t)n, 0);
  for (int i = 0; i < n; ++i)
    okv[i] = aligned_square_inverse(rois[4 * i], rois[4 * i + 1], rois[4 * i + 2], rois[4 * i + 3], out_size, &aff[6 * (size_t)i]) ? 1 : 0;
  uint8_t *d_frame = nullptr, *d_crops = nullptr;
  double* d_aff = nullptr;
  int* d_img = nullptr;
  const size_t fb = (size_t)height * row_stride, px = (size_t)n * out_size * out_size;
  bool ok = cudaMalloc(&d_frame, fb) == cudaSuccess && cudaMalloc(&d_crops, px * 4) == cudaSuccess &&
            cudaMalloc(&d_aff, aff.size() * sizeof(double)) == cudaSuccess && cudaMalloc(&d_img, img.size() * sizeof(int)) == cudaSuccess;
  int rc = ok ? FDT_OK : fail(h, FDT_ERR_CUDA, "crop allocation failed");
  if (rc == FDT_OK) {
    cudaMemcpyAsync(d_frame, frame, fb, cudaMemcpyHostToDevice, s);
    cudaMemcpyAsync(d_aff, aff.data(), aff.size() * sizeof(double), cudaMemcpyHostToDevice, s);
    cudaMemcpyAsync(d_img, img.data(), img.size() * sizeof(int), cudaMemcpyHostToDevice, s);
    WarpP wp;
    wp.frames = d_frame; wp.frame_stride = (long long)fb; wp.row_stride = row_stride; wp.channels = ch; wp.src_w = width; wp.src_h = height;
    wp.crop_img = d_img; wp.affine = d_aff; wp.ncrops = n; wp.out_size = out_size; wp.flip_odd = 0; wp.crops = d_crops;
    launch_warp_affine(wp, s);
    std::vector<uint8_t> tmp(px * 4);
    if (!cuda_ok(h, cudaMemcpyAsync(tmp.data(), d_crops, px * 4, cudaMemcpyDeviceToHost, s), "crop copy") ||
        !cuda_ok(h, cudaStreamSynchronize(s), "crop")) rc = FDT_ERR_CUDA;
    else unpack_bgrx(tmp, px, out_crops);
  }
  if (out_ok) for (int i = 0; i < n; ++i) out_ok[i] = okv[i];
  void* fr[] = {d_frame, d_crops, d_aff, d_img};
  for (void* p : fr) if (p) cudaFree(p);
  return rc;
}

// ---- face crops of the detect calls -----------------------------------------------------------------
namespace {
int set_crops_single(fdt_handle* h, const fdt_crop_spec* spec) {
  cudaSetDevice(h->cfg.device);
  for (int i = 0; spec && i < kSlots; ++i) {
    Slot& sl = h->slots[i];
    if (sl.d_fc_img) continue;
    const size_t cc = (size_t)h->crop_cap;
    if (!dalloc(h, &sl.d_fc_img, cc) || !palloc(h, &sl.h_fc_img, cc) || !dalloc(h, &sl.d_fc_aff, cc * 6) ||
        !palloc(h, &sl.h_fc_aff, cc * 6) || cudaEventCreateWithFlags(&sl.ev_fc, cudaEventDisableTiming) != cudaSuccess) {
      sl.d_fc_img = nullptr;
      return fail(h, FDT_ERR_CUDA, "face crop allocation failed");
    }
  }
  h->crops_on = spec != nullptr;
  if (spec) h->crop_spec = *spec;
  reset_crops(h);
  return FDT_OK;
}
}  // namespace

int32_t fdt_set_face_crops(fdt_handle* h, const fdt_crop_spec* spec) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  std::lock_guard<std::mutex> g(h->mu);
  if (spec) {
    if (spec->struct_size != (int32_t)sizeof(fdt_crop_spec)) return fail(h, FDT_ERR_BAD_ARG, "fdt_crop_spec.struct_size mismatch");
    if (spec->kind != FDT_CROP_EMBEDDING && spec->kind != FDT_CROP_FACE) return fail(h, FDT_ERR_BAD_ARG, "unknown crop kind");
    if (spec->layout & ~(FDT_CROP_RGB | FDT_CROP_CHW | FDT_CROP_F32)) return fail(h, FDT_ERR_BAD_ARG, "unknown crop layout bit");
    if (spec->out_size <= 0 || spec->out_size > 4096) return fail(h, FDT_ERR_BAD_ARG, "crop out_size must be 1..4096");
    for (int c = 0; c < 3; ++c)
      if (!std::isfinite(spec->scale[c]) || !std::isfinite(spec->bias[c])) return fail(h, FDT_ERR_BAD_ARG, "crop scale and bias must be finite");
  }
  for (fdt_handle* r : replicas(h)) {
    std::unique_lock<std::mutex> gl(r->mu, std::defer_lock);
    if (r != h) gl.lock();
    if (int rc = set_crops_single(r, spec)) { if (r != h) h->err = r->err; return rc; }
  }
  h->crops_on = spec != nullptr;
  if (spec) h->crop_spec = *spec;
  return FDT_OK;
}

int32_t fdt_get_face_crops(fdt_handle* h, int64_t* out_n, const void** out_dev) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  std::lock_guard<std::mutex> g(h->mu);
  if (out_dev && !h->shards.empty()) return fail(h, FDT_ERR_UNSUPPORTED, "the crops of a multi-device handle lie on several devices: fdt_copy_face_crops");
  long long n = 0;
  for (fdt_handle* r : replicas(h)) n += r->crop_n;
  if (out_n) *out_n = n;
  if (out_dev) *out_dev = h->d_crop_arena;
  return FDT_OK;
}

int32_t fdt_copy_face_crops(fdt_handle* h, void* dst, size_t capacity, int32_t mem_kind, int32_t* out_ok) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  std::lock_guard<std::mutex> g(h->mu);
  if (mem_kind != FDT_MEM_HOST && mem_kind != FDT_MEM_DEVICE) return fail(h, FDT_ERR_BAD_ARG, "unknown mem_kind");
  if (mem_kind == FDT_MEM_DEVICE && !h->shards.empty())
    return fail(h, FDT_ERR_UNSUPPORTED, "a multi-device handle copies its crops to host memory only");
  const std::vector<fdt_handle*> reps = replicas(h);
  size_t total = 0;
  for (fdt_handle* r : reps) total += (size_t)r->crop_n * crop_bytes(r->crop_spec);
  if (total && !dst) return fail(h, FDT_ERR_BAD_ARG, "null destination");
  if (capacity < total) return fail(h, FDT_ERR_SIZE_MISMATCH, "capacity smaller than n * crop bytes");
  size_t at = 0, k = 0;
  for (fdt_handle* r : reps) {
    const size_t bytes = (size_t)r->crop_n * crop_bytes(r->crop_spec);
    if (bytes) {
      cudaSetDevice(r->cfg.device);
      const cudaMemcpyKind kind = mem_kind == FDT_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
      if (!cuda_ok(h, cudaMemcpy(static_cast<uint8_t*>(dst) + at, r->d_crop_arena, bytes, kind), "face crop copy")) return FDT_ERR_CUDA;
    }
    if (out_ok) std::copy(r->crop_ok.begin(), r->crop_ok.end(), out_ok + k);
    at += bytes; k += r->crop_ok.size();
  }
  return FDT_OK;
}

int64_t fdt_last_launch_count(fdt_handle* h) { return h ? h->launches : 0; }
int64_t fdt_last_h2d_bytes(fdt_handle* h) { return h ? h->h2d_bytes : 0; }

int32_t fdt_set_stage_timing(fdt_handle* h, int32_t enable) {
  if (!h) return FDT_ERR_NOT_READY;
  primary(h)->stage_timing = enable != 0;
  return FDT_OK;
}
int32_t fdt_get_stage_ms(fdt_handle* h, int32_t stage, float* ms, int32_t* launches) {
  if (!h || stage < 0 || stage >= kNumStages) return FDT_ERR_BAD_ARG;
  h = primary(h);
  if (ms) *ms = h->stage_ms[stage];
  if (launches) *launches = h->stage_launches[stage];
  return FDT_OK;
}

int32_t fdt_timer_begin(fdt_handle* h) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  h = primary(h);
  std::lock_guard<std::mutex> g(h->mu);
  cudaSetDevice(h->cfg.device);
  for (int i = 0; i < kSlots; ++i) cudaStreamSynchronize(h->slots[i].stream);
  cudaEventRecord(h->tev[0], h->slots[0].stream);
  for (int i = 1; i < kSlots; ++i) cudaStreamWaitEvent(h->slots[i].stream, h->tev[0], 0);
  return FDT_OK;
}

int32_t fdt_timer_end(fdt_handle* h, float* ms) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  h = primary(h);
  std::lock_guard<std::mutex> g(h->mu);
  cudaSetDevice(h->cfg.device);
  for (int i = 1; i < kSlots; ++i) {
    cudaEventRecord(h->tev[2], h->slots[i].stream);
    cudaStreamWaitEvent(h->slots[0].stream, h->tev[2], 0);
  }
  cudaEventRecord(h->tev[1], h->slots[0].stream);
  if (!cuda_ok(h, cudaEventSynchronize(h->tev[1]), "timer")) return FDT_ERR_CUDA;
  float t = 0;
  cudaEventElapsedTime(&t, h->tev[0], h->tev[1]);
  if (ms) *ms = t;
  return FDT_OK;
}

int32_t fdt_profile_chunk(fdt_handle* h, const uint8_t* d_frames, int32_t n, int32_t width, int32_t height,
                          int32_t row_stride, int32_t mat_type, int32_t repeats, float* out_ms, int32_t capacity,
                          int32_t* out_launches) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  h = primary(h);
  std::lock_guard<std::mutex> g(h->mu);
  const int S = (int)h->det.plan().steps.size();
  if (out_launches) *out_launches = S + 2;
  FrameLayout lay;
  const char* msg = nullptr;
  if (!d_frames || n <= 0 || n > h->chunk || width <= 0 || height <= 0 || repeats <= 0 ||
      frame_layout(mat_type, width, height, row_stride, &lay, &msg) != FDT_OK)
    return fail(h, FDT_ERR_BAD_ARG, "bad profile arguments");
  if (!out_ms || capacity < S + 2) return fail(h, FDT_ERR_SIZE_MISMATCH, "out_ms too small");
  cudaSetDevice(h->cfg.device);
  if (!ensure_results(h, n)) return FDT_ERR_CUDA;
  const LbTables* tb = get_tables(h, width, height, 1);
  if (!tb) return fail(h, FDT_ERR_CUDA, "letterbox table upload failed");
  std::vector<cudaEvent_t> ev(S + 3);
  for (auto& e : ev) cudaEventCreate(&e);
  std::vector<double> acc(S + 2, 0.0);
  Slot& sl = h->slots[0];
  cudaStream_t s = sl.stream;
  const int S_w = h->det.in_w(), S_h = h->det.in_h();
  for (int r = 0; r < repeats; ++r) {
    cudaEventRecord(ev[0], s);
    if (lay.rgb) {
      LetterboxRgbP lb;
      fill_letterbox(lb.lb, tb, d_frames, lay.frame_bytes, row_stride, lay.channels, width, height, sl.d_lb, S_w, S_h, false);
      lb.pf = lay.px;
      launch_letterbox_rgb(lb, n, false, s);
    } else if (lay.yuv) {
      LetterboxYuvP lb;
      fill_letterbox_yuv(lb, tb, lay, d_frames, lay.frame_bytes, false, d_frames + lay.c_off, lay.frame_bytes, false, row_stride,
                         width, height, sl.d_lb, S_w, S_h);
      launch_letterbox_yuv(lb, n, s, lay.p010);
    } else {
      LetterboxP lb;
      fill_letterbox(lb, tb, d_frames, lay.frame_bytes, row_stride, lay.channels, width, height, sl.d_lb, S_w, S_h, false);
      launch_letterbox(lb, n, s);
    }
    h->det.run(sl.det_ctx, sl.d_lb, n, s, ev.data() + 1);
    DecodeP d;
    fill_decode(d, h, sl, tb, width, height);
    d.faces = h->d_faces; d.counts = h->d_counts;
    launch_decode_nms(d, n, s);
    cudaEventRecord(ev[S + 2], s);
    if (!cuda_ok(h, cudaStreamSynchronize(s), "profile")) { for (auto& e : ev) cudaEventDestroy(e); return FDT_ERR_CUDA; }
    for (int i = 0; i < S + 2; ++i) {
      float ms = 0;
      cudaEventElapsedTime(&ms, ev[i], ev[i + 1]);
      acc[i] += ms;
    }
  }
  for (int i = 0; i < S + 2; ++i) out_ms[i] = (float)(acc[i] / repeats);
  for (auto& e : ev) cudaEventDestroy(e);
  return FDT_OK;
}

static const char* kKernelNames[] = {"k_normalize", "k_naive_conv", "k_gemm_conv", "k_dwpw", "k_add", "k_act", "k_padc", "k_maxpool",
                                     "k_resize_bilinear", "k_stem", "k_block_ws", "k_stem_ws", "k_tail_ws", "k_fc_tc", "k_block_ts"};

static void step_info(const Plan& p, const PStep& st, int in_w, int in_h, std::string* kname, std::string* tname, double* macs, double* bytes) {
  *kname = kKernelNames[st.kind]; *tname = st.name; *macs = st.macs;
  const PTensor& o = p.tensors[st.out];
  double b = (double)o.H * o.W * o.C * 4;
  if (st.out2 >= 0) { const PTensor& o2 = p.tensors[st.out2]; b += (double)o2.H * o2.W * o2.C * 4; }
  if (st.in_u8) b += (double)in_w * in_h * 4;
  else if (st.in >= 0) { const PTensor& i = p.tensors[st.in]; b += (double)i.H * i.W * i.C * 4; }
  if (st.in2 >= 0 && st.in2 != st.in) { const PTensor& r = p.tensors[st.in2]; b += (double)r.H * r.W * r.C * 4; }
  for (int extra : st.extra_out) { const PTensor& e = p.tensors[extra]; b += (double)e.H * e.W * e.C * 4; }
  *bytes = b;
}

int32_t fdt_get_step_info(fdt_handle* h, int32_t launch, char* kernel, char* tensor, int32_t str_cap, double* macs_per_image,
                          double* bytes_per_image) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  h = primary(h);
  const Plan& p = h->det.plan();
  const int S = (int)p.steps.size();
  if (launch < 0 || launch > S + 1) return fail(h, FDT_ERR_BAD_ARG, "launch index out of range");
  std::string kname, tname;
  double macs = 0, bytes = 0;
  if (launch == 0) {
    kname = "k_letterbox"; tname = "letterboxed_u8";
    bytes = 0;  // depends on the frame size: 4 taps x 3 B per content pixel read + S*S*3 written (filled by the caller)
  } else if (launch == S + 1) {
    kname = "k_decode_nms"; tname = "faces";
    bytes = (double)h->num_anchors * 17 * 4;
  } else {
    step_info(p, p.steps[launch - 1], h->det.in_w(), h->det.in_h(), &kname, &tname, &macs, &bytes);
  }
  if (kernel && str_cap > 0) { std::snprintf(kernel, str_cap, "%s", kname.c_str()); }
  if (tensor && str_cap > 0) { std::snprintf(tensor, str_cap, "%s", tname.c_str()); }
  if (macs_per_image) *macs_per_image = macs;
  if (bytes_per_image) *bytes_per_image = bytes;
  return FDT_OK;
}

int32_t fdt_profile_net(fdt_handle* h, int32_t which, int32_t n, int32_t repeats, float* out_ms, int32_t capacity, int32_t* out_steps) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  h = primary(h);
  std::lock_guard<std::mutex> g(h->mu);
  if (which != 1 && which != 2) return fail(h, FDT_ERR_BAD_ARG, "which: 1 mesh, 2 iris");
  if ((which == 1 && !h->has_mesh) || (which == 2 && !h->has_iris)) return fail(h, FDT_ERR_NOT_READY, "model not loaded");
  const Engine& e = which == 1 ? h->mesh : h->iris;
  const int S = (int)e.plan().steps.size();
  if (out_steps) *out_steps = S;
  const int have = which == 1 ? h->last_mesh_faces : 2 * h->last_iris_faces;
  if (n <= 0 || n > have) n = have;                  // n <= 0: every crop the last call left
  if (out_steps) out_steps[0] = S;
  if (n <= 0 || repeats <= 0) return fail(h, FDT_ERR_BAD_ARG, "the last call left no crops in the stage buffers");
  if (!out_ms || capacity < S) return fail(h, FDT_ERR_SIZE_MISMATCH, "out_ms too small");
  cudaSetDevice(h->cfg.device);
  Slot& sl = h->slots[which == 1 ? h->last_mesh_slot : h->last_iris_slot];
  cudaStream_t s = sl.stream;
  std::vector<cudaEvent_t> ev(S + 1);
  for (auto& x : ev) cudaEventCreate(&x);
  std::vector<double> acc(S, 0.0);
  int rc = FDT_OK;
  for (int r = 0; r < repeats && rc == FDT_OK; ++r) {
    if (which == 1) h->mesh.run(sl.mesh_ctx, sl.d_crops, n, s, ev.data());
    else h->iris.run(sl.iris_ctx, sl.d_eye_crops, n, s, ev.data());
    if (!cuda_ok(h, cudaStreamSynchronize(s), "profile")) { rc = FDT_ERR_CUDA; break; }
    for (int i = 0; i < S; ++i) {
      float ms = 0;
      cudaEventElapsedTime(&ms, ev[i], ev[i + 1]);
      acc[i] += ms;
    }
  }
  for (int i = 0; i < S; ++i) out_ms[i] = (float)(acc[i] / repeats);
  for (auto& x : ev) cudaEventDestroy(x);
  return rc;
}

int32_t fdt_get_net_step_info(fdt_handle* h, int32_t which, int32_t step, char* kernel, char* tensor, int32_t str_cap,
                              double* macs_per_image, double* bytes_per_image) {
  if (!h || !h->ready) return fail(h, FDT_ERR_NOT_READY, "detector is not initialised");
  h = primary(h);
  if (which < 0 || which > 2 || (which == 1 && !h->has_mesh) || (which == 2 && !h->has_iris)) return fail(h, FDT_ERR_BAD_ARG, "which: 0 detector, 1 mesh, 2 iris");
  const Engine& e = which == 0 ? h->det : (which == 1 ? h->mesh : h->iris);
  const Plan& p = e.plan();
  if (step < 0 || step >= (int)p.steps.size()) return fail(h, FDT_ERR_BAD_ARG, "step index out of range");
  std::string kname, tname;
  double macs = 0, bytes = 0;
  step_info(p, p.steps[step], e.in_w(), e.in_h(), &kname, &tname, &macs, &bytes);
  if (kernel && str_cap > 0) { std::snprintf(kernel, str_cap, "%s", kname.c_str()); }
  if (tensor && str_cap > 0) { std::snprintf(tensor, str_cap, "%s", tname.c_str()); }
  if (macs_per_image) *macs_per_image = macs;
  if (bytes_per_image) *bytes_per_image = bytes;
  return FDT_OK;
}

int32_t fdt_host_anchors(int32_t model, double* out_xy, int32_t capacity_pairs) {
  std::vector<double> a = generate_anchors(ssd_options(model));
  int n = (int)a.size() / 2;
  if (out_xy) std::memcpy(out_xy, a.data(), (size_t)std::min(n, capacity_pairs) * 2 * sizeof(double));
  return n;
}

int32_t fdt_host_plan_describe(const uint8_t* tflite, size_t len, int32_t fuse_level, char* buf, size_t buf_len) {
  TfModel m;
  std::string err;
  Plan p;
  std::string text;
  int rc = FDT_OK;
  if (!m.parse(tflite, len, &err) || !p.build(m, fuse_level, &err)) { text = err; rc = FDT_ERR_MODEL; }
  else text = p.describe();
  if (buf && buf_len) {
    size_t n = std::min(buf_len - 1, text.size());
    std::memcpy(buf, text.data(), n);
    buf[n] = 0;
  }
  return rc;
}

int32_t fdt_host_resize_taps(int32_t src, int32_t dst, int32_t is_x_axis, int32_t* i0, int32_t* i1, int16_t* w0, int16_t* w1) {
  if (src <= 0 || dst <= 0 || !i0 || !i1 || !w0 || !w1) return FDT_ERR_BAD_ARG;
  resize_linear_taps(src, dst, is_x_axis != 0, i0, i1, w0, w1);
  return FDT_OK;
}

int32_t fdt_host_decode_box(const float* raw16, double ax, double ay, double scale, double* out_box4, double* out_kp12) {
  if (!raw16 || !out_box4 || !out_kp12) return FDT_ERR_BAD_ARG;
  decode_box(raw16, ax, ay, scale, out_box4, out_kp12);
  return FDT_OK;
}

int32_t fdt_host_tile_walk(int32_t first, int32_t stride, int32_t tiles_x, int32_t tiles_y, int32_t n, int32_t* out3) {
  if (!out3 || first < 0 || stride <= 0 || tiles_x <= 0 || tiles_y <= 0 || n < 0) return FDT_ERR_BAD_ARG;
  const int tpi = tiles_x * tiles_y;
  const TileStep step = tile_step(stride, tpi, tiles_x);
  TileAt at = tile_at(first, tpi, tiles_x);
  for (int i = 0; i < n; ++i) {
    out3[3 * i] = at.b; out3[3 * i + 1] = at.ty; out3[3 * i + 2] = at.tx;
    tile_advance(at, step, tiles_x, tiles_y);
  }
  return FDT_OK;
}

int32_t fdt_host_face_roi(const double* kp12, double img_w, double img_h, int32_t out_size, double* out10) {
  if (!kp12 || !out10) return 0;
  face_alignment(kp12, img_w, img_h, &out10[0], &out10[1], &out10[2], &out10[3]);
  return aligned_square_inverse(out10[1], out10[2], out10[3], -out10[0], out_size, &out10[4]) ? 1 : 0;
}

int32_t fdt_host_eye_rois(const double* corners8, double* out8) {
  if (!corners8 || !out8) return FDT_ERR_BAD_ARG;
  eye_rois_from_corners(corners8, out8);
  return FDT_OK;
}

int32_t fdt_host_embedding_roi(const double* l, const double* r, double* out4) {
  if (!l || !r || !out4) return FDT_ERR_BAD_ARG;
  embedding_alignment(l, r, out4);
  return FDT_OK;
}

const char* fdt_last_error(fdt_handle* h) {
  static thread_local std::string copy;
  if (h) {
    std::lock_guard<std::mutex> g(h->mu);
    copy = h->err;
    return copy.c_str();
  }
  std::lock_guard<std::mutex> g(g_create_mu);
  copy = g_create_error;
  return copy.c_str();
}

const char* fdt_version(void) { return "fdt-cuda 0.2.0 (sm_100a)"; }

}  // extern "C"
