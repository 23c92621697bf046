// Preprocessing kernels: fused letterbox (cv::resize INTER_LINEAR 8U fixed point +
// copyMakeBorder(0) + BGRA/GRAY->BGR, or cvtColor YUV2BGR for NV12 / NV21 / I420 frames; k_letterbox_multi for chunks of
// frames of different sizes and formats; k_letterbox_tr for frames stored transposed; k_letterbox_rgb for RGB, RGBA and planar
// RGB frames, read through their PixFmt, and packed YUV 4:2:2 frames; k_letterbox_multi<., ., true> for separate-plane YUV frames;
// the k16 variants for 16-bit YUV 4:2:0, P010 and fdt_detect_yuv_planes16 frames) and the [-1,1] normalisation.
// Reference: convertImageToTensor / bgrMatToSignedFloat32 (lib/src/util/helpers.dart:303-421).
#include "kernels.h"

namespace fdt {
namespace {

__device__ __forceinline__ void load_bgr(const uint8_t* px, int channels, int* v) {
  if (channels == 1) { v[0] = v[1] = v[2] = px[0]; }
  else { v[0] = px[0]; v[1] = px[1]; v[2] = px[2]; }
}

// HResizeLinear (11-bit) then VResizeLinear<uchar,int,short> fixed point (resize.cpp) of one channel of four taps
__device__ __forceinline__ int resize_linear(int t00, int t01, int t10, int t11, int wa, int wb, int va, int vb) {
  int h0 = t00 * wa + t01 * wb;
  int h1 = t10 * wa + t11 * wb;
  int v = ((va * (h0 >> 4)) >> 16) + ((vb * (h1 >> 4)) >> 16);
  v = (v + 2) >> 2;
  return v < 0 ? 0 : (v > 255 ? 255 : v);
}

// One thread per output pixel: four 3-byte taps (byte loads; neighbouring threads share the sectors through L1) and one uchar4
// store; grid = (columns / 64, rows / 4, frames), so no index is divided (the flat 64-bit index this kernel started with cost two
// 64-bit divisions per pixel: 125 -> 122 us per 1024 1280x720 frames).
// Measured alternatives (round 2), both SLOWER on B200:
//  * the 6 bytes of the two neighbouring taps of a row from two aligned 32-bit loads + a funnel shift instead of six byte loads
//    (a third of the load instructions, same sectors): 168-172 us vs 122;
//  * a row-staged kernel - one warp per output row, the two source rows fetched with coalesced 16-byte streaming loads into shared
//    memory, taps read from there: 148 vs 126 us (97 vs 73 us per 256 1920x1080 frames).
// The DRAM traffic is the same in all three (every 32-byte sector of the 2-in-10 source rows) and this form already sits at 68 % of
// peak DRAM throughput.
__global__ void __launch_bounds__(256) k_letterbox(LetterboxP p, int B) {
  const int x = blockIdx.x * 64 + (threadIdx.x & 63), y = blockIdx.y * 4 + (threadIdx.x >> 6);
  if (x >= p.dst_w || y >= p.dst_h) return;
  for (int b = blockIdx.z; b < B; b += gridDim.z) {
    const int dy = y - p.pad_top, dx = x - p.pad_left;
    uchar3 o = make_uchar3(0, 0, 0);
    if (dy >= 0 && dy < p.new_h && dx >= 0 && dx < p.new_w) {
      const uint8_t* src = p.frames + (size_t)b * p.frame_stride;
      if (p.identity) {
        int v[3];
        load_bgr(src + (size_t)dy * p.row_stride + (size_t)dx * p.channels, p.channels, v);
        o = make_uchar3((unsigned char)v[0], (unsigned char)v[1], (unsigned char)v[2]);
      } else {
        const int xa = p.x0[dx], xb = p.x1[dx], wa = p.ax0[dx], wb = p.ax1[dx];
        const int ya = p.y0[dy], yb = p.y1[dy], va = p.by0[dy], vb = p.by1[dy];
        int t00[3], t01[3], t10[3], t11[3];
        const uint8_t* r0 = src + (size_t)ya * p.row_stride;
        const uint8_t* r1 = src + (size_t)yb * p.row_stride;
        load_bgr(r0 + (size_t)xa * p.channels, p.channels, t00);
        load_bgr(r0 + (size_t)xb * p.channels, p.channels, t01);
        load_bgr(r1 + (size_t)xa * p.channels, p.channels, t10);
        load_bgr(r1 + (size_t)xb * p.channels, p.channels, t11);
        int res[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) res[c] = resize_linear(t00[c], t01[c], t10[c], t11[c], wa, wb, va, vb);
        o = make_uchar3((unsigned char)res[0], (unsigned char)res[1], (unsigned char)res[2]);
      }
    }
    reinterpret_cast<uchar4*>(p.out)[((size_t)b * p.dst_h + y) * p.dst_w + x] = make_uchar4(o.x, o.y, o.z, 0);
  }
}

// The Y sample of pixel x: its byte, or for P010 (k16) the high byte of its 16-bit word, (s >> 8) & 0xFF.  A P010 frame's chroma
// step and offsets (4, 1, 3) already name the high bytes of its U and V words.
template <bool k16>
__device__ __forceinline__ int y_sample(const uint8_t* yrow, int x) { return k16 ? yrow[(size_t)x * 2 + 1] : yrow[x]; }

// One YUV 4:2:0 tap: the Y byte and the chroma pair of its 2x2 block, converted to BGR (cvtColor first, then resize).
template <bool k16 = false>
__device__ __forceinline__ void load_yuv(const uint8_t* yrow, const uint8_t* crow, int x, const LetterboxYuvP& p, int* v) {
  const uint8_t* c = crow + (size_t)(x >> 1) * p.c_step;
  yuv_to_bgr(y_sample<k16>(yrow, x), c[p.u_off], c[p.v_off], v);
}
// the same for a frame of a ragged chunk
template <bool k16 = false>
__device__ __forceinline__ void load_yuv(const uint8_t* yrow, const uint8_t* crow, int x, const FrameD& f, int* v) {
  const uint8_t* c = crow + (size_t)(x >> 1) * f.c_step;
  yuv_to_bgr(y_sample<k16>(yrow, x), c[f.u_off], c[f.v_off], v);
}

// k_letterbox for NV12 / NV21 / I420 frames: same grid and fixed-point resize; every tap is converted before it is weighted
// (the conversion is per pixel, so this equals resizing the converted frame).  Padding stays BGR 0.
// k16: P010 frames; each tap's samples are reduced to 8 bits on load (y_sample), so the output equals that of the NV12 frame
// made of the words' high bytes.
template <bool k16>
__global__ void __launch_bounds__(256) k_letterbox_yuv(LetterboxYuvP p, int B) {
  const LetterboxP& q = p.lb;
  const int x = blockIdx.x * 64 + (threadIdx.x & 63), y = blockIdx.y * 4 + (threadIdx.x >> 6);
  if (x >= q.dst_w || y >= q.dst_h) return;
  for (int b = blockIdx.z; b < B; b += gridDim.z) {
    const int dy = y - q.pad_top, dx = x - q.pad_left;
    uchar3 o = make_uchar3(0, 0, 0);
    if (dy >= 0 && dy < q.new_h && dx >= 0 && dx < q.new_w) {
      const uint8_t* ys = q.frames + (size_t)b * q.frame_stride;
      const uint8_t* cs = p.chroma + (size_t)b * p.c_frame_stride;
      if (q.identity) {
        int v[3];
        load_yuv<k16>(ys + (size_t)dy * q.row_stride, cs + (size_t)(dy >> 1) * p.c_row_stride, dx, p, v);
        o = make_uchar3((unsigned char)v[0], (unsigned char)v[1], (unsigned char)v[2]);
      } else {
        const int xa = q.x0[dx], xb = q.x1[dx], wa = q.ax0[dx], wb = q.ax1[dx];
        const int ya = q.y0[dy], yb = q.y1[dy], va = q.by0[dy], vb = q.by1[dy];
        const int ca = p.cy0[dy], cb = p.cy1[dy];
        int t00[3], t01[3], t10[3], t11[3];
        const uint8_t* r0 = ys + (size_t)ya * q.row_stride;
        const uint8_t* r1 = ys + (size_t)yb * q.row_stride;
        const uint8_t* c0 = cs + (size_t)ca * p.c_row_stride;
        const uint8_t* c1 = cs + (size_t)cb * p.c_row_stride;
        load_yuv<k16>(r0, c0, xa, p, t00);
        load_yuv<k16>(r0, c0, xb, p, t01);
        load_yuv<k16>(r1, c1, xa, p, t10);
        load_yuv<k16>(r1, c1, xb, p, t11);
        int res[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) res[c] = resize_linear(t00[c], t01[c], t10[c], t11[c], wa, wb, va, vb);
        o = make_uchar3((unsigned char)res[0], (unsigned char)res[1], (unsigned char)res[2]);
      }
    }
    reinterpret_cast<uchar4*>(q.out)[((size_t)b * q.dst_h + y) * q.dst_w + x] = make_uchar4(o.x, o.y, o.z, 0);
  }
}

// Frames stored transposed (orientations 5-8): the grid and fixed-point resize of k_letterbox over the upright image U, whose
// pixel (x, y) is the stored pixel (row x', column y') - x' from the x taps, y' from the y taps, flips already folded into both.
// So U's four taps t00 = U(xa, ya), t01 = U(xb, ya), t10 = U(xa, yb), t11 = U(xb, yb) are read from stored rows xa / xb and stored
// columns ya / yb, and resize_linear weights them exactly as it weights an upright frame's taps: the output bytes are those of
// letterboxing U itself.  No identity branch: at equal sizes the taps are (i, weight 2048 / 0), which resize_linear returns exactly.
// k16 (with kYuv): P010 frames, read as k_letterbox_yuv<true> reads them.
template <bool kYuv, bool k16>
__global__ void __launch_bounds__(256) k_letterbox_tr(LetterboxTrP p, int B) {
  const LetterboxP& q = p.yp.lb;
  const int x = blockIdx.x * 64 + (threadIdx.x & 63), y = blockIdx.y * 4 + (threadIdx.x >> 6);
  if (x >= q.dst_w || y >= q.dst_h) return;
  for (int b = blockIdx.z; b < B; b += gridDim.z) {
    const int dy = y - q.pad_top, dx = x - q.pad_left;
    uchar3 o = make_uchar3(0, 0, 0);
    if (dy >= 0 && dy < q.new_h && dx >= 0 && dx < q.new_w) {
      const uint8_t* src = q.frames + (size_t)b * q.frame_stride;
      const int ra = q.x0[dx], rb = q.x1[dx], wa = q.ax0[dx], wb = q.ax1[dx];   // stored rows, U's x weights
      const int ca = q.y0[dy], cb = q.y1[dy], va = q.by0[dy], vb = q.by1[dy];   // stored columns, U's y weights
      int t00[3], t01[3], t10[3], t11[3];
      const uint8_t* r0 = src + (size_t)ra * q.row_stride;
      const uint8_t* r1 = src + (size_t)rb * q.row_stride;
      if (kYuv) {
        const uint8_t* cs = p.yp.chroma + (size_t)b * p.yp.c_frame_stride;
        const uint8_t* c0 = cs + (size_t)p.yp.cy0[dx] * p.yp.c_row_stride;
        const uint8_t* c1 = cs + (size_t)p.yp.cy1[dx] * p.yp.c_row_stride;
        load_yuv<k16>(r0, c0, ca, p.yp, t00);
        load_yuv<k16>(r1, c1, ca, p.yp, t01);
        load_yuv<k16>(r0, c0, cb, p.yp, t10);
        load_yuv<k16>(r1, c1, cb, p.yp, t11);
      } else {
        load_bgr(r0 + (size_t)ca * q.channels, q.channels, t00);
        load_bgr(r1 + (size_t)ca * q.channels, q.channels, t01);
        load_bgr(r0 + (size_t)cb * q.channels, q.channels, t10);
        load_bgr(r1 + (size_t)cb * q.channels, q.channels, t11);
      }
      int res[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) res[c] = resize_linear(t00[c], t01[c], t10[c], t11[c], wa, wb, va, vb);
      o = make_uchar3((unsigned char)res[0], (unsigned char)res[1], (unsigned char)res[2]);
    }
    reinterpret_cast<uchar4*>(q.out)[((size_t)b * q.dst_h + y) * q.dst_w + x] = make_uchar4(o.x, o.y, o.z, 0);
  }
}

// Ragged batches: the grid of k_letterbox, one frame per blockIdx.z step, its geometry and layout from a descriptor table.  The
// format is the same for every thread of a block, so the packed / YUV branch does not diverge; the arithmetic is that of
// k_letterbox / k_letterbox_yuv, so a frame letterboxes to the same bytes in a ragged chunk as in a uniform one.
// kTransposed: the chunk also holds frames of orientations 5-8, gathered as in k_letterbox_tr (block-uniform branch; their
// chroma rows are the stored rows halved, mixed calls upload whole frames).  Orientations 2-4 need nothing here: their flips are
// folded into the taps.
// kFmt: the chunk also holds RGB / RGBA / planar RGB frames; every packed or planar frame is read through its PixFmt pfs[b]
// (launched with kTransposed = true, for a chunk of any orientations).
// kPlanes: every frame of the chunk is a separate-plane YUV frame whose chroma is read through its YuvPlaneD pls[b] (launched with
// kTransposed = true and kFmt = false); the chroma row of a tap is the same as above, only its address differs.
// k422: the chunk also holds packed YUV 4:2:2 frames (launched with kTransposed = kFmt = true); their taps are read with load_422,
// which needs the tap's column as well as its row.
// k16 (launched with kTransposed = true): the chunk holds P010 frames (c_step 4), whose Y samples are read by y_sample<true>, or
// (with kPlanes) every frame is an fdt_detect_yuv_planes16 frame, read with load_yuv_planes16 and its YuvPlaneD::shift.  Only the
// loads differ; every tap's samples are 8-bit before yuv_to_bgr, so the output is that of the 8-bit frame.
template <bool kFmt>
__device__ __forceinline__ void load_packed(const uint8_t* px, int channels, const PixFmt& pf, int* v) {
  if (kFmt) load_pix(px, pf, v);
  else load_bgr(px, channels, v);
}
// pixel x of a packed or planar frame's row; k422: the chunk also holds packed YUV 4:2:2 frames (pf.yuv422, block-uniform)
template <bool kFmt, bool k422>
__device__ __forceinline__ void load_packed_at(const uint8_t* row, int x, int channels, const PixFmt& pf, int* v) {
  if (k422 && pf.yuv422) load_422(row, x, pf, v);
  else load_packed<kFmt>(row + (size_t)x * channels, channels, pf, v);
}
// a YUV 4:2:0 tap of a ragged chunk's frame; k16: the chunk may hold P010 frames (c_step 4, block-uniform)
template <bool k16>
__device__ __forceinline__ void load_yuv_frame(const uint8_t* yrow, const uint8_t* crow, int x, const FrameD& f, int* v) {
  if (k16 && f.c_step == 4) load_yuv<true>(yrow, crow, x, f, v);
  else load_yuv(yrow, crow, x, f, v);
}
// a tap of a separate-plane frame; k16: planes of 16-bit words
template <bool k16>
__device__ __forceinline__ void load_planes(const uint8_t* yrow, int crow, int x, const YuvPlaneD& q, int* v) {
  if (k16) load_yuv_planes16(yrow, crow, x, q, v);
  else load_yuv_planes(yrow, crow, x, q, v);
}

template <bool kTransposed, bool kFmt, bool kPlanes, bool k422, bool k16>
__global__ void __launch_bounds__(256) k_letterbox_multi(LetterboxMultiP p, int B, const PixFmt* pfs, const YuvPlaneD* pls) {
  const int x = blockIdx.x * 64 + (threadIdx.x & 63), y = blockIdx.y * 4 + (threadIdx.x >> 6);
  if (x >= p.dst_w || y >= p.dst_h) return;
  for (int b = blockIdx.z; b < B; b += gridDim.z) {
    const FrameD f = p.fr[b];
    PixFmt pf;
    if (kFmt) pf = pfs[b];
    YuvPlaneD pl;
    if (kPlanes) pl = pls[b];
    const int dy = y - f.pad_top, dx = x - f.pad_left;
    uchar3 o = make_uchar3(0, 0, 0);
    if (dy >= 0 && dy < f.new_h && dx >= 0 && dx < f.new_w) {
      int res[3];
      if (kTransposed && f.orientation >= 5) {
        const int* tx = p.taps + f.tx;
        const int* ty = p.taps + f.ty;
        const int ra = tx[dx], rb = tx[f.new_w + dx], wa = tx[2 * f.new_w + dx], wb = tx[3 * f.new_w + dx];
        const int ca = ty[dy], cb = ty[f.new_h + dy], va = ty[2 * f.new_h + dy], vb = ty[3 * f.new_h + dy];
        int t00[3], t01[3], t10[3], t11[3];
        const uint8_t* r0 = f.y + (size_t)ra * f.row_stride;
        const uint8_t* r1 = f.y + (size_t)rb * f.row_stride;
        if (kPlanes) {
          load_planes<k16>(r0, ra >> 1, ca, pl, t00);
          load_planes<k16>(r1, rb >> 1, ca, pl, t01);
          load_planes<k16>(r0, ra >> 1, cb, pl, t10);
          load_planes<k16>(r1, rb >> 1, cb, pl, t11);
        } else if (f.channels) {
          load_packed_at<kFmt, k422>(r0, ca, f.channels, pf, t00);
          load_packed_at<kFmt, k422>(r1, ca, f.channels, pf, t01);
          load_packed_at<kFmt, k422>(r0, cb, f.channels, pf, t10);
          load_packed_at<kFmt, k422>(r1, cb, f.channels, pf, t11);
        } else {
          const uint8_t* c0 = f.c + (size_t)(ra >> 1) * f.c_row_stride;
          const uint8_t* c1 = f.c + (size_t)(rb >> 1) * f.c_row_stride;
          load_yuv_frame<k16>(r0, c0, ca, f, t00);
          load_yuv_frame<k16>(r1, c1, ca, f, t01);
          load_yuv_frame<k16>(r0, c0, cb, f, t10);
          load_yuv_frame<k16>(r1, c1, cb, f, t11);
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) res[c] = resize_linear(t00[c], t01[c], t10[c], t11[c], wa, wb, va, vb);
      } else if (f.identity) {
        if (kPlanes) load_planes<k16>(f.y + (size_t)dy * f.row_stride, dy >> 1, dx, pl, res);
        else if (f.channels) load_packed_at<kFmt, k422>(f.y + (size_t)dy * f.row_stride, dx, f.channels, pf, res);
        else load_yuv_frame<k16>(f.y + (size_t)dy * f.row_stride, f.c + (size_t)(dy >> 1) * f.c_row_stride, dx, f, res);
      } else {
        const int* tx = p.taps + f.tx;
        const int* ty = p.taps + f.ty;
        const int xa = tx[dx], xb = tx[f.new_w + dx], wa = tx[2 * f.new_w + dx], wb = tx[3 * f.new_w + dx];
        const int ya = ty[dy], yb = ty[f.new_h + dy], va = ty[2 * f.new_h + dy], vb = ty[3 * f.new_h + dy];
        int t00[3], t01[3], t10[3], t11[3];
        const uint8_t* r0 = f.y + (size_t)ya * f.row_stride;
        const uint8_t* r1 = f.y + (size_t)yb * f.row_stride;
        if (kPlanes) {
          const int ca = ty[4 * f.new_h + dy], cb = ty[5 * f.new_h + dy];
          load_planes<k16>(r0, ca, xa, pl, t00);
          load_planes<k16>(r0, ca, xb, pl, t01);
          load_planes<k16>(r1, cb, xa, pl, t10);
          load_planes<k16>(r1, cb, xb, pl, t11);
        } else if (f.channels) {
          load_packed_at<kFmt, k422>(r0, xa, f.channels, pf, t00);
          load_packed_at<kFmt, k422>(r0, xb, f.channels, pf, t01);
          load_packed_at<kFmt, k422>(r1, xa, f.channels, pf, t10);
          load_packed_at<kFmt, k422>(r1, xb, f.channels, pf, t11);
        } else {
          const uint8_t* c0 = f.c + (size_t)ty[4 * f.new_h + dy] * f.c_row_stride;
          const uint8_t* c1 = f.c + (size_t)ty[5 * f.new_h + dy] * f.c_row_stride;
          load_yuv_frame<k16>(r0, c0, xa, f, t00);
          load_yuv_frame<k16>(r0, c0, xb, f, t01);
          load_yuv_frame<k16>(r1, c1, xa, f, t10);
          load_yuv_frame<k16>(r1, c1, xb, f, t11);
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) res[c] = resize_linear(t00[c], t01[c], t10[c], t11[c], wa, wb, va, vb);
      }
      o = make_uchar3((unsigned char)res[0], (unsigned char)res[1], (unsigned char)res[2]);
    }
    reinterpret_cast<uchar4*>(p.out)[((size_t)b * p.dst_h + y) * p.dst_w + x] = make_uchar4(o.x, o.y, o.z, 0);
  }
}

// pixel x of a row through its PixFmt: load_pix, or for packed YUV 4:2:2 frames (k422) load_422
template <bool k422>
__device__ __forceinline__ void load_fmt(const uint8_t* row, int x, int step, const PixFmt& pf, int* v) {
  if (k422) load_422(row, x, pf, v);
  else load_pix(row + (size_t)x * step, pf, v);
}

// RGB, RGBA and planar RGB frames (uniform chunks): the grid, taps and fixed-point resize of k_letterbox (kTransposed = false,
// identity branch included) or of k_letterbox_tr (true, orientations 5-8: x taps name stored rows, y taps stored columns), with
// every tap's B, G, R read through p.pf.  Swapping channels or reading three planes only changes which bytes a tap loads, so the
// output equals letterboxing the BGR image.  k422: packed YUV 4:2:2 frames, every tap converted as cvtColor converts it before
// it is weighted (as k_letterbox_yuv does), so the output equals letterboxing the converted frame.
template <bool kTransposed, bool k422>
__global__ void __launch_bounds__(256) k_letterbox_rgb(LetterboxRgbP p, int B) {
  const LetterboxP& q = p.lb;
  const int x = blockIdx.x * 64 + (threadIdx.x & 63), y = blockIdx.y * 4 + (threadIdx.x >> 6);
  if (x >= q.dst_w || y >= q.dst_h) return;
  const int step = p.pf.step;
  for (int b = blockIdx.z; b < B; b += gridDim.z) {
    const int dy = y - q.pad_top, dx = x - q.pad_left;
    uchar3 o = make_uchar3(0, 0, 0);
    if (dy >= 0 && dy < q.new_h && dx >= 0 && dx < q.new_w) {
      const uint8_t* src = q.frames + (size_t)b * q.frame_stride;
      int res[3];
      if (!kTransposed && q.identity) {
        load_fmt<k422>(src + (size_t)dy * q.row_stride, dx, step, p.pf, res);
      } else {
        const int xa = q.x0[dx], xb = q.x1[dx], wa = q.ax0[dx], wb = q.ax1[dx];
        const int ya = q.y0[dy], yb = q.y1[dy], va = q.by0[dy], vb = q.by1[dy];
        int t00[3], t01[3], t10[3], t11[3];
        if (kTransposed) {
          const uint8_t* r0 = src + (size_t)xa * q.row_stride;
          const uint8_t* r1 = src + (size_t)xb * q.row_stride;
          load_fmt<k422>(r0, ya, step, p.pf, t00);
          load_fmt<k422>(r1, ya, step, p.pf, t01);
          load_fmt<k422>(r0, yb, step, p.pf, t10);
          load_fmt<k422>(r1, yb, step, p.pf, t11);
        } else {
          const uint8_t* r0 = src + (size_t)ya * q.row_stride;
          const uint8_t* r1 = src + (size_t)yb * q.row_stride;
          load_fmt<k422>(r0, xa, step, p.pf, t00);
          load_fmt<k422>(r0, xb, step, p.pf, t01);
          load_fmt<k422>(r1, xa, step, p.pf, t10);
          load_fmt<k422>(r1, xb, step, p.pf, t11);
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) res[c] = resize_linear(t00[c], t01[c], t10[c], t11[c], wa, wb, va, vb);
      }
      o = make_uchar3((unsigned char)res[0], (unsigned char)res[1], (unsigned char)res[2]);
    }
    reinterpret_cast<uchar4*>(q.out)[((size_t)b * q.dst_h + y) * q.dst_w + x] = make_uchar4(o.x, o.y, o.z, 0);
  }
}

__global__ void k_normalize(const uint8_t* in, TV out, long long total) {
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    int c = (int)(idx % out.Cs);
    long long pix = idx / out.Cs;
    long long hw = (long long)out.H * out.W;
    int b = (int)(pix / hw);
    long long sp = pix % hw;
    float v = 0.f;
    if (c < 3) v = fmaf((float)in[((size_t)b * hw + sp) * 4 + (2 - c)], 1.0f / 127.5f, -1.0f);
    out.p[b * out.istride + sp * out.Cs + c] = v;
  }
}

}  // namespace

void launch_letterbox(const LetterboxP& p, int B, cudaStream_t s) {
  if (B <= 0) return;
  dim3 grid((unsigned)((p.dst_w + 63) / 64), (unsigned)((p.dst_h + 3) / 4), (unsigned)(B < 65535 ? B : 65535));
  k_letterbox<<<grid, 256, 0, s>>>(p, B);
}

void launch_letterbox_yuv(const LetterboxYuvP& p, int B, cudaStream_t s, bool p010) {
  if (B <= 0) return;
  dim3 grid((unsigned)((p.lb.dst_w + 63) / 64), (unsigned)((p.lb.dst_h + 3) / 4), (unsigned)(B < 65535 ? B : 65535));
  if (p010) k_letterbox_yuv<true><<<grid, 256, 0, s>>>(p, B);
  else k_letterbox_yuv<false><<<grid, 256, 0, s>>>(p, B);
}

void launch_letterbox_tr(const LetterboxTrP& p, int B, cudaStream_t s, bool p010) {
  if (B <= 0) return;
  dim3 grid((unsigned)((p.yp.lb.dst_w + 63) / 64), (unsigned)((p.yp.lb.dst_h + 3) / 4), (unsigned)(B < 65535 ? B : 65535));
  if (p.yuv && p010) k_letterbox_tr<true, true><<<grid, 256, 0, s>>>(p, B);
  else if (p.yuv) k_letterbox_tr<true, false><<<grid, 256, 0, s>>>(p, B);
  else k_letterbox_tr<false, false><<<grid, 256, 0, s>>>(p, B);
}

void launch_letterbox_multi(const LetterboxMultiP& p, int B, bool transposed, cudaStream_t s, const PixFmt* pf, const YuvPlaneD* pl,
                            bool yuv422, bool yuv16) {
  if (B <= 0) return;
  dim3 grid((unsigned)((p.dst_w + 63) / 64), (unsigned)((p.dst_h + 3) / 4), (unsigned)(B < 65535 ? B : 65535));
  if (yuv16) {
    if (pl) k_letterbox_multi<true, false, true, false, true><<<grid, 256, 0, s>>>(p, B, pf, pl);
    else if (pf && yuv422) k_letterbox_multi<true, true, false, true, true><<<grid, 256, 0, s>>>(p, B, pf, pl);
    else if (pf) k_letterbox_multi<true, true, false, false, true><<<grid, 256, 0, s>>>(p, B, pf, pl);
    else k_letterbox_multi<true, false, false, false, true><<<grid, 256, 0, s>>>(p, B, pf, pl);
  } else if (pl) k_letterbox_multi<true, false, true, false, false><<<grid, 256, 0, s>>>(p, B, pf, pl);
  else if (pf && yuv422) k_letterbox_multi<true, true, false, true, false><<<grid, 256, 0, s>>>(p, B, pf, pl);
  else if (pf) k_letterbox_multi<true, true, false, false, false><<<grid, 256, 0, s>>>(p, B, pf, pl);
  else if (transposed) k_letterbox_multi<true, false, false, false, false><<<grid, 256, 0, s>>>(p, B, pf, pl);
  else k_letterbox_multi<false, false, false, false, false><<<grid, 256, 0, s>>>(p, B, pf, pl);
}

void launch_letterbox_rgb(const LetterboxRgbP& p, int B, bool transposed, cudaStream_t s) {
  if (B <= 0) return;
  dim3 grid((unsigned)((p.lb.dst_w + 63) / 64), (unsigned)((p.lb.dst_h + 3) / 4), (unsigned)(B < 65535 ? B : 65535));
  if (p.pf.yuv422) {
    if (transposed) k_letterbox_rgb<true, true><<<grid, 256, 0, s>>>(p, B);
    else k_letterbox_rgb<false, true><<<grid, 256, 0, s>>>(p, B);
  } else {
    if (transposed) k_letterbox_rgb<true, false><<<grid, 256, 0, s>>>(p, B);
    else k_letterbox_rgb<false, false><<<grid, 256, 0, s>>>(p, B);
  }
}

void launch_normalize(const uint8_t* in, TV out, int B, cudaStream_t s) {
  long long total = (long long)B * out.H * out.W * out.Cs;
  long long g = (total + 255) / 256;
  if (g > 148LL * 32) g = 148LL * 32;
  k_normalize<<<(int)(g < 1 ? 1 : g), 256, 0, s>>>(in, out, total);
}

}  // namespace fdt
