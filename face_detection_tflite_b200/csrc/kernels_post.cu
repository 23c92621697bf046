// Geometry-side kernels, compiled with -fmad=false so that the f64 arithmetic is evaluated
// operation by operation exactly like the reference's Dart doubles / OpenCV's C++:
//   k_decode_nms       threshold -> ordered compaction -> decode -> sort -> weighted NMS ->
//                      letterbox removal -> gates   (one block per image)
//   k_warp_affine      cv::warpAffine(INTER_LINEAR, BORDER_CONSTANT 0) into square BGR crops (192 face / 64 eye);
//                      YUV 4:2:0 frames are converted tap by tap (in-frame taps only); RGB, RGBA and planar RGB frames
//                      and packed YUV 4:2:2 frames are read through their PixFmt; separate-plane YUV frames through their
//                      YuvPlaneD
//   k_mesh_post        _unpackLandmarks + transformMeshToAbsolute + face-flag sigmoid
//   k_iris_post        _unpackLandmarks(clamp: false) + transformIrisNormToAbsolute + iris-centre eye keypoints
#include "fdt_math.h"
#include "kernels.h"

namespace fdt {
namespace {

constexpr int kDecodeThreads = 128;
constexpr int kMaxDet = 100;          // weightedNms maxDet (lib/src/util/helpers.dart:187)
constexpr double kRawScoreLimit = 100.0;  // lib/src/shared/face_model_config.dart:49
constexpr int kTaken = -(1 << 30);        // s_order entry of a candidate already merged into an emitted cluster

struct NmsOut { double box[4]; double score; int cand; };

__global__ void __launch_bounds__(kDecodeThreads) k_decode_nms(DecodeP p) {
  extern __shared__ __align__(16) unsigned char dsm[];
  const int N = p.N;
  double* s_score = reinterpret_cast<double*>(dsm);            // [N]
  double* s_box = s_score + N;                                 // [N][4]
  int* s_idx = reinterpret_cast<int*>(s_box + 4 * (size_t)N);  // [N]
  int* s_order = s_idx + N;                                    // [N]
  unsigned char* s_alive = reinterpret_cast<unsigned char*>(s_order + N);  // [N]
  __shared__ int s_wcnt[kDecodeThreads / 32];
  __shared__ int s_n, s_nvalid, s_top, s_pos;
  __shared__ NmsOut s_out[kMaxDet];
  __shared__ fdt_face s_face[kMaxDet];
  __shared__ unsigned char s_pass[kMaxDet];
  __shared__ int s_dst[kMaxDet];

  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* scores = p.scores + (size_t)b * p.scores_istride;
  const float* boxes = p.boxes + (size_t)b * p.boxes_istride;
  if (tid == 0) { s_n = 0; s_nvalid = 0; }
  __syncthreads();

  // 1. candidates: raw >= logit(minScore), ascending anchor order (_collectCandidateScores)
  const double* pre = p.pre ? p.pre + (size_t)b * N * 17 : nullptr;
  if (pre) {
    // test entry (fdt_debug_nms): the N rows are detections already decoded by the caller
    for (int c = tid; c < N; c += kDecodeThreads) s_idx[c] = c;
    if (tid == 0) s_n = N;
    __syncthreads();
  } else {
    for (int base = 0; base < N; base += kDecodeThreads) {
      int i = base + tid;
      bool flag = i < N && (double)scores[i] >= p.raw_thresh;
      unsigned bal = __ballot_sync(0xffffffffu, flag);
      if (lane == 0) s_wcnt[warp] = __popc(bal);
      __syncthreads();
      int woff = 0, tot = 0;
#pragma unroll
      for (int w = 0; w < kDecodeThreads / 32; ++w) {
        if (w < warp) woff += s_wcnt[w];
        tot += s_wcnt[w];
      }
      if (flag) s_idx[s_n + woff + __popc(bal & ((1u << lane) - 1u))] = i;
      __syncthreads();
      if (tid == 0) s_n += tot;
      __syncthreads();
    }
  }
  const int n = s_n;
  if (p.cand_n) {
    if (tid == 0) p.cand_n[b] = n;
    for (int c = tid; c < n && c < p.cand_cap; c += kDecodeThreads) p.cand_idx[(size_t)b * p.cand_cap + c] = s_idx[c];
  }

  // 2. score + decode (+ degenerate-box filter, score >= kMinScore filter)
  for (int c = tid; c < n; c += kDecodeThreads) {
    int i = s_idx[c];
    double sc, box[4], kp[12];
    if (pre) {
      for (int k = 0; k < 4; ++k) box[k] = pre[(size_t)i * 17 + k];
      sc = pre[(size_t)i * 17 + 4];
      for (int k = 0; k < 12; ++k) kp[k] = pre[(size_t)i * 17 + 5 + k];
    } else {
      sc = sigmoid_clipped((double)scores[i], kRawScoreLimit);
      decode_box(boxes + (size_t)i * 16, p.anchors[2 * i], p.anchors[2 * i + 1], (double)p.input_h, box, kp);
    }
    bool valid = !(box[2] <= box[0] || box[3] <= box[1]) && sc >= p.score_thresh;
    s_score[c] = sc;
    s_box[4 * c + 0] = box[0]; s_box[4 * c + 1] = box[1];
    s_box[4 * c + 2] = box[2]; s_box[4 * c + 3] = box[3];
    s_alive[c] = valid ? 1 : 0;
    if (valid) atomicAdd(&s_nvalid, 1);
    if (p.dbg_dec) {
      double* d = p.dbg_dec + ((size_t)b * N + c) * 18;
      for (int k = 0; k < 4; ++k) d[k] = box[k];
      d[4] = sc;
      for (int k = 0; k < 12; ++k) d[5 + k] = kp[k];
      d[17] = valid ? 1.0 : 0.0;
    }
  }
  __syncthreads();
  const int nvalid = s_nvalid;

  // 3. stable sort by score descending (rank sort; ties keep ascending anchor order)
  for (int c = tid; c < n; c += kDecodeThreads) {
    if (!s_alive[c]) continue;
    double sc = s_score[c];
    int rank = 0;
    for (int j = 0; j < n; ++j) {
      if (!s_alive[j]) continue;
      double sj = s_score[j];
      rank += (sj > sc || (sj == sc && j < c)) ? 1 : 0;
    }
    s_order[rank] = c;
  }
  if (tid == 0) s_pos = 0;
  __syncthreads();

  // 4. weighted NMS (flutter_litert weightedNms; strict IoU > thr against the top box)
  int nout = 0;
  while (nout < kMaxDet) {
    if (tid == 0) {
      int pos = s_pos;
      while (pos < nvalid && (s_order[pos] < 0 || !s_alive[s_order[pos]])) ++pos;
      s_pos = pos;
      s_top = pos < nvalid ? s_order[pos] : -1;
    }
    __syncthreads();
    const int top = s_top, pos0 = s_pos;
    if (top < 0) break;
    double tb[4] = {s_box[4 * top], s_box[4 * top + 1], s_box[4 * top + 2], s_box[4 * top + 3]};
    // cluster membership in parallel (s_order of a cluster member is overwritten by -1 - candidate) ...
    for (int j = pos0 + tid; j < nvalid; j += kDecodeThreads) {
      int c = s_order[j];
      if (c < 0 || !s_alive[c]) continue;
      if ((c == top) || box_iou(&s_box[4 * c], tb) > p.iou_thresh) { s_alive[c] = 0; s_order[j] = -1 - c; }
    }
    __syncthreads();
    // ... and the score-weighted sum by ONE thread in sorted order, exactly the reference's sequential f64 accumulation
    // (a tree reduction would round differently): clusters hold a handful of boxes
    if (tid == 0) {
      double t[5] = {0, 0, 0, 0, 0};
      for (int j = pos0; j < nvalid; ++j) {
        int e = s_order[j];
        if (e >= 0 || e == kTaken) continue;
        int c = -1 - e;
        s_order[j] = kTaken;
        double sc = s_score[c];
        t[0] += sc;
        t[1] += s_box[4 * c + 0] * sc;
        t[2] += s_box[4 * c + 1] * sc;
        t[3] += s_box[4 * c + 2] * sc;
        t[4] += s_box[4 * c + 3] * sc;
      }
      NmsOut& o = s_out[nout];
      o.box[0] = t[1] / t[0]; o.box[1] = t[2] / t[0];
      o.box[2] = t[3] / t[0]; o.box[3] = t[4] / t[0];
      o.score = s_score[top];
      o.cand = top;
      s_pos = pos0 + 1;
    }
    ++nout;
    __syncthreads();
  }

  // 5. letterbox removal (helpers.dart:101-136), gates (face_gates.dart:130-146), ROI check
  //    (face_detector_core.dart:255-265 / helpers.dart:591-592)
  const double* g = p.geom ? p.geom + 6 * (size_t)b : nullptr;
  const double pad_t = g ? g[0] : p.pad_t, pad_b = g ? g[1] : p.pad_b, pad_l = g ? g[2] : p.pad_l, pad_r = g ? g[3] : p.pad_r;
  const double img_w = g ? g[4] : p.img_w, img_h = g ? g[5] : p.img_h;
  const double sx = 1.0 - (pad_l + pad_r), sy = 1.0 - (pad_t + pad_b);
  for (int f = tid; f < nout; f += kDecodeThreads) {
    const NmsOut& o = s_out[f];
    int i = s_idx[o.cand];
    double box[4], kp[12];
    if (pre) { for (int k = 0; k < 12; ++k) kp[k] = pre[(size_t)i * 17 + 5 + k]; }
    else decode_box(boxes + (size_t)i * 16, p.anchors[2 * i], p.anchors[2 * i + 1], (double)p.input_h, box, kp);
    fdt_face fc;
    fc.xmin = (o.box[0] - pad_l) / sx;
    fc.ymin = (o.box[1] - pad_t) / sy;
    fc.xmax = (o.box[2] - pad_l) / sx;
    fc.ymax = (o.box[3] - pad_t) / sy;
    fc.score = o.score;
    for (int k = 0; k < 12; k += 2) {
      fc.keypoints[k] = (kp[k] - pad_l) / sx;
      fc.keypoints[k + 1] = (kp[k + 1] - pad_t) / sy;
    }
    fc.mesh_score = nan("");
    fc.has_mesh = 0;
    fc.anchor_index = i;
    fc.has_iris = 0;            // every byte of the record is defined: callers read has_iris, tests compare records bitwise
    fc.reserved = 0;
    bool pass = true;
    if (p.min_score > 0.0 || p.min_face_size > 0.0) {
      pass = fc.score >= p.min_score &&
             (p.min_face_size <= 0.0 || visible_width_fraction(fc.xmin, fc.xmax, img_w) >= p.min_face_size);
    }
    double theta, cx, cy, size;
    face_alignment(fc.keypoints, img_w, img_h, &theta, &cx, &cy, &size);
    if (!p.skip_roi && !(dart_round(size) > 0)) pass = false;
    s_face[f] = fc;
    s_pass[f] = pass ? 1 : 0;
  }
  __syncthreads();
  if (tid == 0) {
    int cnt = 0;
    for (int f = 0; f < nout; ++f) {
      s_dst[f] = -1;
      if (s_pass[f] && cnt < p.max_faces) s_dst[f] = cnt++;
    }
    p.counts[b] = cnt;
  }
  __syncthreads();
  for (int f = tid; f < nout; f += kDecodeThreads)
    if (s_dst[f] >= 0) p.faces[(size_t)b * p.max_faces + s_dst[f]] = s_face[f];
}

// ------------------------------------------------------------------------------------------
constexpr bool kWarpYuv422 = false;   // warp_affine.cuh: chunks with a packed YUV 4:2:2 frame take kernels_warp422.cu
constexpr bool kWarp16 = false;       // and chunks with a 16-bit YUV 4:2:0 frame kernels_warp16.cu
#include "warp_affine.cuh"

// ------------------------------------------------------------------------------------------
__global__ void k_mesh_post(MeshPostP p) {
  const int f = blockIdx.x;
  if (f >= p.nfaces) return;
  const float* raw = p.raw + (size_t)f * p.raw_istride;
  const double cx = p.roi[6 * f + 1], cy = p.roi[6 * f + 2], size = p.roi[6 * f + 3];
  // transformMeshToAbsolute (lib/src/shared/face_geometry.dart:48-73); cos / sin come from the host libm
  const double ct = p.roi[6 * f + 4], st = p.roi[6 * f + 5];
  const double sct = size * ct, sst = size * st;
  const double tx = cx - 0.5 * sct + 0.5 * sst;
  const double ty = cy - 0.5 * sst - 0.5 * sct;
  // _unpackLandmarks with zero padding (lib/src/util/helpers.dart:138-172)
  const double inv_w = 1.0 / p.in_size, inv_h = 1.0 / p.in_size, inv_sx = 1.0 / (1.0 - 0.0), inv_sy = 1.0 / (1.0 - 0.0);
  for (int i = threadIdx.x; i < FDT_MESH_POINTS; i += blockDim.x) {
    double x = ((double)raw[3 * i] * inv_w - 0.0) * inv_sx;
    double y = ((double)raw[3 * i + 1] * inv_h - 0.0) * inv_sy;
    double z = (double)raw[3 * i + 2] * inv_w * inv_sx;
    x = x < 0.0 ? 0.0 : (x > 1.0 ? 1.0 : x);
    y = y < 0.0 ? 0.0 : (y > 1.0 ? 1.0 : y);
    const double ax = tx + sct * x - sst * y, ay = ty + sst * x + sct * y;
    float* o = p.mesh_out + (size_t)f * FDT_MESH_FLOATS + 3 * i;
    o[0] = (float)ax;
    o[1] = (float)ay;
    o[2] = (float)(z * size);
    // eyeRoisFromMesh reads the f64 points 33/133 (left) and 362/263 (right) (face_geometry.dart:155-168)
    if (p.eye_corners) {
      const int k = i == 33 ? 0 : (i == 133 ? 1 : (i == 362 ? 2 : (i == 263 ? 3 : -1)));
      if (k >= 0) { p.eye_corners[8 * f + 2 * k] = ax; p.eye_corners[8 * f + 2 * k + 1] = ay; }
    }
  }
  if (threadIdx.x == 0)
    p.score_out[f] = sigmoid_clipped((double)p.flag[(size_t)f * p.flag_istride], kRawScoreLimit);
}

// ------------------------------------------------------------------------------------------
// One block per face, 152 threads = 2 eyes x 76 points.  IrisLandmark.call unpacks every output in order
// (71 contour points then 5 iris points, clamp: false, z untouched; lib/src/models/iris_landmark.dart:328-360),
// transformIrisNormToAbsolute maps them into the frame and un-mirrors the right eye
// (lib/src/shared/face_geometry.dart:109-125); the detector's eye keypoints are replaced by the iris point closest
// to the iris centroid (irisCenterFromPoints, face_types.dart:976-997; face_detector_core.dart:356-373).
__global__ void k_iris_post(IrisPostP p) {
  const int f = blockIdx.x;
  if (f >= p.nfaces) return;
  __shared__ double s_xy[2][5][2];
  const int t = threadIdx.x;
  if (t < 2 * 76) {
    const int eye = t / 76, i = t - eye * 76;
    const int e = 2 * f + eye;
    const float* src = i < 71 ? p.contours + (size_t)e * p.contours_istride + 3 * i
                              : p.iris + (size_t)e * p.iris_istride + 3 * (i - 71);
    const double inv = 1.0 / p.in_size;
    const double x = ((double)src[0] * inv - 0.0) * (1.0 / (1.0 - 0.0));
    const double y = ((double)src[1] * inv - 0.0) * (1.0 / (1.0 - 0.0));
    const double z = (double)src[2];
    const double cx = p.roi[6 * e + 1], cy = p.roi[6 * e + 2], s = p.roi[6 * e + 3], ct = p.roi[6 * e + 4], st = p.roi[6 * e + 5];
    const double px = eye ? (1.0 - x) : x;
    const double lx2 = (px - 0.5) * s, ly2 = (y - 0.5) * s;
    const double ax = cx + lx2 * ct - ly2 * st, ay = cy + lx2 * st + ly2 * ct;
    float* o = p.iris_out + (size_t)f * FDT_IRIS_FLOATS + 3 * t;
    o[0] = (float)ax; o[1] = (float)ay; o[2] = (float)z;
    if (i >= 71) { s_xy[eye][i - 71][0] = ax; s_xy[eye][i - 71][1] = ay; }
  }
  __syncthreads();
  if (t < 2) {
    double mx = 0, my = 0;
    for (int k = 0; k < 5; ++k) { mx += s_xy[t][k][0]; my += s_xy[t][k][1]; }
    mx /= 5; my /= 5;
    int best = 0;
    double bd = INFINITY;
    for (int k = 0; k < 5; ++k) {
      const double dx = s_xy[t][k][0] - mx, dy = s_xy[t][k][1] - my, d = dx * dx + dy * dy;
      if (d < bd) { bd = d; best = k; }
    }
    const double iw = p.img_wh ? p.img_wh[2 * f] : p.img_w, ih = p.img_wh ? p.img_wh[2 * f + 1] : p.img_h;
    p.eye_kp[4 * f + 2 * t] = s_xy[t][best][0] / iw;
    p.eye_kp[4 * f + 2 * t + 1] = s_xy[t][best][1] / ih;
  }
}

}  // namespace

size_t decode_smem_bytes(int N) {
  return (size_t)N * (8 + 32 + 4 + 4 + 1) + 16;
}

void launch_decode_nms(const DecodeP& p, int B, cudaStream_t s) {
  size_t smem = decode_smem_bytes(p.N);
  cudaFuncSetAttribute(k_decode_nms, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  k_decode_nms<<<B, kDecodeThreads, smem, s>>>(p);
}

template <bool kFmt, bool kOut> void launch_warp(const WarpP& p, dim3 grid, cudaStream_t s, const CropOutP& o) {
  if (p.orientation != 1) {
    if (p.fr) k_warp_affine<true, true, kFmt, false, kOut><<<grid, 256, 0, s>>>(p, nullptr, o);
    else k_warp_affine<false, true, kFmt, false, kOut><<<grid, 256, 0, s>>>(p, nullptr, o);
  } else {
    if (p.fr) k_warp_affine<true, false, kFmt, false, kOut><<<grid, 256, 0, s>>>(p, nullptr, o);
    else k_warp_affine<false, false, kFmt, false, kOut><<<grid, 256, 0, s>>>(p, nullptr, o);
  }
}

template <bool kOut> void launch_warp_any(const WarpP& p, dim3 grid, cudaStream_t s, const YuvPlaneD* pl, const CropOutP& o,
                                          bool yuv422, bool yuv16) {
  if (yuv16) {
    launch_warp_affine_16(p, grid, s, pl, kOut ? &o : nullptr);
  } else if (pl) {
    if (p.orientation != 1) k_warp_affine<true, true, false, true, kOut><<<grid, 256, 0, s>>>(p, pl, o);
    else k_warp_affine<true, false, false, true, kOut><<<grid, 256, 0, s>>>(p, pl, o);
  } else if (p.pf && yuv422) {
    launch_warp_affine_422(p, grid, s, kOut ? &o : nullptr);
  } else if (p.pf) {
    launch_warp<true, kOut>(p, grid, s, o);
  } else {
    launch_warp<false, kOut>(p, grid, s, o);
  }
}

void launch_warp_affine(const WarpP& p, cudaStream_t s, const YuvPlaneD* pl, const CropOutP* out, bool yuv422, bool yuv16) {
  if (p.ncrops <= 0) return;
  dim3 grid((p.out_size * p.out_size + 255) / 256, p.ncrops);
  if (out) launch_warp_any<true>(p, grid, s, pl, *out, yuv422, yuv16);
  else launch_warp_any<false>(p, grid, s, pl, CropOutP(), yuv422, yuv16);
}

void launch_mesh_post(const MeshPostP& p, cudaStream_t s) {
  if (p.nfaces <= 0) return;
  k_mesh_post<<<p.nfaces, 128, 0, s>>>(p);
}

void launch_iris_post(const IrisPostP& p, cudaStream_t s) {
  if (p.nfaces <= 0) return;
  k_iris_post<<<p.nfaces, 160, 0, s>>>(p);
}

}  // namespace fdt
