// Geometry-side kernels, compiled with -fmad=false so that the f64 arithmetic is evaluated
// operation by operation exactly like the reference's Dart doubles / OpenCV's C++:
//   k_decode_nms       threshold -> ordered compaction -> decode -> sort -> weighted NMS ->
//                      letterbox removal -> gates   (one block per image)
//   k_warp_affine      cv::warpAffine(INTER_LINEAR, BORDER_CONSTANT 0) into square BGR crops (192 face / 64 eye);
//                      YUV 4:2:0 frames are converted tap by tap (in-frame taps only); RGB, RGBA and planar RGB frames
//                      are read through their PixFmt; separate-plane YUV frames through their YuvPlaneD
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
__device__ __forceinline__ long long sat_round_ll(double v) { return (long long)rint(v); }

// One thread per output pixel; blockIdx.y = crop.  The per-row / per-column fixed-point terms of
// imgproc/imgwarp.cpp WarpAffineInvoker (AB_BITS = 10, INTER_BITS = 5) are evaluated per pixel: two f64 rint each.
// kRagged: the crop's frame, its layout and size come from the descriptor table p.fr (chunks of frames of different sizes).
// kOriented: the frame is stored rotated / mirrored (EXIF orientation, p.orientation or the descriptor's).  Coordinates, weights
// and bounds are those of the upright image U; only each in-frame tap's address is mapped to the stored pixel (and chroma
// sample) it is.  Folding the orientation into the affine map instead would change the rint rounding above.
// kFmt: the frame (uniform) or some frame of the chunk (ragged) is RGB / RGBA / planar RGB; every packed or planar frame's taps
// are read through its PixFmt (p.pf[0], or p.pf[frame]), so a crop equals the crop of the BGR image.
// kPlanes (ragged only): every frame of the chunk is a separate-plane YUV frame, its chroma read through pl[frame].
// kOut: a face crop of the detect calls.  Only the epilogue differs: crop f goes to crop out.first + f of the packed arena in
// out.layout (FDT_CROP_RGB / _CHW / _F32); a warp's 32 pixels are consecutive in each CHW plane.
template <bool kRagged, bool kOriented, bool kFmt, bool kPlanes, bool kOut>
__global__ void k_warp_affine(WarpP p, const YuvPlaneD* pl, CropOutP out) {
  const int f = blockIdx.y;
  if (f >= p.ncrops) return;
  const int S = p.out_size;
  const double* A = p.affine + 6 * f;
  // every per-frame value is written as (kRagged ? descriptor : parameter), so the uniform instantiation is the plain kernel
  const FrameD* d = kRagged ? p.fr + p.crop_img[f] : nullptr;
  const uint8_t* src = kRagged ? d->y : p.frames + (size_t)p.crop_img[f] * p.frame_stride;
  const bool flip = p.flip_odd && (f & 1);
  const int orient = kOriented ? (kRagged ? d->orientation : p.orientation) : 1;
  const bool tr = orient >= 5;
  PixFmt pf;
  if (kFmt) pf = p.pf[kRagged ? p.crop_img[f] : 0];
  YuvPlaneD q;
  if (kPlanes) q = pl[p.crop_img[f]];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < S * S; i += gridDim.x * blockDim.x) {
    int y = i / S, x = i - y * S;
    long long adelta = sat_round_ll(A[0] * x * 1024.0);
    long long bdelta = sat_round_ll(A[3] * x * 1024.0);
    long long X0 = sat_round_ll((A[1] * y + A[2]) * 1024.0) + 16;
    long long Y0 = sat_round_ll((A[4] * y + A[5]) * 1024.0) + 16;
    long long X = (X0 + adelta) >> 5, Y = (Y0 + bdelta) >> 5;
    long long sxl = X >> 5, syl = Y >> 5;
    sxl = sxl < -32768 ? -32768 : (sxl > 32767 ? 32767 : sxl);
    syl = syl < -32768 ? -32768 : (syl > 32767 ? 32767 : syl);
    int sx = (int)sxl, sy = (int)syl;
    int iw[4];
    warp_weights((int)(X & 31), (int)(Y & 31), iw);
    int acc[3] = {0, 0, 0};
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      int yy = sy + (t >> 1), xx = sx + (t & 1);
      // bounds of U: the uniform src_w / src_h already are U's size; a descriptor holds the stored size
      if (yy < 0 || yy >= (kRagged ? (tr ? d->w : d->h) : p.src_h) || xx < 0 || xx >= (kRagged ? (tr ? d->h : d->w) : p.src_w)) continue;   // out-of-frame taps: BGR 0 (also for YUV frames)
      if (kOriented) {
        // U(xx, yy) = stored(column, row): flips first (2, 3, 6, 7 run U's x backwards, 3, 4, 7, 8 its y), then the transpose
        const int uw = kRagged ? (tr ? d->h : d->w) : p.src_w, uh = kRagged ? (tr ? d->w : d->h) : p.src_h;
        const int fx = (orient == 2 || orient == 3 || orient == 6 || orient == 7) ? uw - 1 - xx : xx;
        const int fy = (orient == 3 || orient == 4 || orient == 7 || orient == 8) ? uh - 1 - yy : yy;
        xx = tr ? fy : fx;
        yy = tr ? fx : fy;
      }
      const int row_stride = kRagged ? d->row_stride : p.row_stride;
      if (kPlanes) {
        int v[3];
        load_yuv_planes(src + (size_t)yy * row_stride, yy >> 1, xx, q, v);
        acc[0] += v[0] * iw[t]; acc[1] += v[1] * iw[t]; acc[2] += v[2] * iw[t];
        continue;
      }
      if (kRagged ? d->channels == 0 : p.yuv) {
        const uint8_t* c = (kRagged ? d->c : src + p.c_off) + (size_t)(yy >> 1) * (kRagged ? d->c_row_stride : p.c_row_stride) +
                           (size_t)(xx >> 1) * (kRagged ? d->c_step : p.c_step);
        int v[3];
        yuv_to_bgr(src[(size_t)yy * row_stride + xx], c[kRagged ? d->u_off : p.u_off], c[kRagged ? d->v_off : p.v_off], v);
        acc[0] += v[0] * iw[t]; acc[1] += v[1] * iw[t]; acc[2] += v[2] * iw[t];
        continue;
      }
      const int channels = kRagged ? d->channels : p.channels;
      const uint8_t* px = src + (size_t)yy * row_stride + (size_t)xx * channels;
      if (kFmt) {
        int v[3];
        load_pix(px, pf, v);
        acc[0] += v[0] * iw[t]; acc[1] += v[1] * iw[t]; acc[2] += v[2] * iw[t];
      } else if (channels == 1) {
        acc[0] += px[0] * iw[t]; acc[1] += px[0] * iw[t]; acc[2] += px[0] * iw[t];
      } else {
        acc[0] += px[0] * iw[t]; acc[1] += px[1] * iw[t]; acc[2] += px[2] * iw[t];
      }
    }
    uint8_t o[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      int v = (acc[c] + 16384) >> 15;
      o[c] = (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v));
    }
    if (kOut) {
      const size_t px = (size_t)S * S, k = (size_t)out.first + f;
      const bool chw = out.layout & FDT_CROP_CHW;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const uint8_t v = o[(out.layout & FDT_CROP_RGB) ? 2 - c : c];
        const size_t at = chw ? (3 * k + c) * px + i : (k * px + i) * 3 + c;
        if (out.layout & FDT_CROP_F32) reinterpret_cast<float*>(out.dst)[at] = __fadd_rn(__fmul_rn((float)v, out.scale[c]), out.bias[c]);
        else reinterpret_cast<uint8_t*>(out.dst)[at] = v;
      }
      continue;
    }
    const int xo = flip ? S - 1 - x : x;
    reinterpret_cast<uchar4*>(p.crops)[(size_t)f * S * S + (size_t)y * S + xo] = make_uchar4(o[0], o[1], o[2], 0);
  }
}

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

template <bool kOut> void launch_warp_any(const WarpP& p, dim3 grid, cudaStream_t s, const YuvPlaneD* pl, const CropOutP& o) {
  if (pl) {
    if (p.orientation != 1) k_warp_affine<true, true, false, true, kOut><<<grid, 256, 0, s>>>(p, pl, o);
    else k_warp_affine<true, false, false, true, kOut><<<grid, 256, 0, s>>>(p, pl, o);
  } else if (p.pf) {
    launch_warp<true, kOut>(p, grid, s, o);
  } else {
    launch_warp<false, kOut>(p, grid, s, o);
  }
}

void launch_warp_affine(const WarpP& p, cudaStream_t s, const YuvPlaneD* pl, const CropOutP* out) {
  if (p.ncrops <= 0) return;
  dim3 grid((p.out_size * p.out_size + 255) / 256, p.ncrops);
  if (out) launch_warp_any<true>(p, grid, s, pl, *out);
  else launch_warp_any<false>(p, grid, s, pl, CropOutP());
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
