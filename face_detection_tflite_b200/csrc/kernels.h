// Kernel parameter blocks and launchers for the BlazeFace / face-mesh hot path (sm_100a).
// Layout: activations are NHWC fp32 in HBM, channel stride Cs = roundup4(C) (padded lanes are
// always written as 0) except for views into graph outputs, which are dense (Cs == C).
#pragma once
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdint>

#include "../../include/fdt_api.h"
#include "tail_layer.h"

namespace fdt {

enum { kActNone = 0, kActRelu = 1, kActPrelu = 2 };

// Division by a runtime-constant divisor as multiply-high + shift (n < 2^31), so the index
// arithmetic of the staging / epilogue loops costs 3 instructions instead of ~30.
struct FastDiv {
  unsigned mul = 0, shr = 0, d = 1;
  FastDiv() {}
  explicit FastDiv(int div) {
    d = div < 1 ? 1u : (unsigned)div;
    unsigned l = 0;
    while ((1ull << l) < d) ++l;
    shr = l;
    mul = (unsigned)(((1ull << 32) * ((1ull << l) - d)) / d + 1);
  }
#ifdef __CUDACC__
  __device__ __forceinline__ int div(int n) const { return (int)((__umulhi(mul, (unsigned)n) + (unsigned)n) >> shr); }
  __device__ __forceinline__ void divmod(int n, int& q, int& r) const { q = div(n); r = n - q * (int)d; }
#endif
};

struct TV {  // tensor view (device)
  float* p = nullptr;       // image 0
  long long istride = 0;    // floats between consecutive images
  int H = 1, W = 1, C = 1, Cs = 1;
};

// ---- generic one-thread-per-element kernels (fuse_level 0 and shapes the tiled kernels skip) ----
struct NaiveConvP {
  TV in, out;
  const float* w;      // OHWI [Cout][kh][kw][Cin]  (depthwise: [kh][kw][C])
  const float* bias;   // [Cout] or nullptr
  const float* alpha;  // PReLU slopes [Cout] or nullptr
  int kh, kw, sh, sw, pt, pl, act, depthwise;
};
struct EltP {
  TV a, b, out;        // b unused for unary ops
  const float* alpha;
  int act;
};
struct PoolP { TV in, out; int fh, fw, sh, sw, pt, pl; };
struct ResizeP { TV in, out; int align_corners, half_pixel; TV add; int has_add, act; };   // has_add: out = resize(in) + add [ReLU]

void launch_naive_conv(const NaiveConvP& p, int B, cudaStream_t s);
void launch_add(const EltP& p, int B, cudaStream_t s);
void launch_act(const EltP& p, int B, cudaStream_t s);
void launch_padc(const EltP& p, int B, cudaStream_t s);
void launch_maxpool(const PoolP& p, int B, cudaStream_t s);
void launch_resize_bilinear(const ResizeP& p, int B, cudaStream_t s);

// ---- preprocessing ----
#ifdef __CUDACC__
// cv::cvtColor COLOR_YUV2BGR_NV12 / _NV21 / _I420 for one sample (BT.601 limited range, 20-bit fixed point, imgproc/color_yuv):
// v[0..2] = B, G, R.
__device__ __forceinline__ int sat_u8(int v) { return v < 0 ? 0 : (v > 255 ? 255 : v); }
__device__ __forceinline__ void yuv_to_bgr(int Y, int U, int V, int* v) {
  const int yy = max(Y - 16, 0) * 1220542 + (1 << 19), u = U - 128, w = V - 128;
  v[0] = sat_u8((yy + 2116026 * u) >> 20);
  v[1] = sat_u8((yy - 852492 * w - 409993 * u) >> 20);
  v[2] = sat_u8((yy + 1673527 * w) >> 20);
}
#endif
struct LetterboxP {
  const uint8_t* frames;   // [B][H][row_stride]
  long long frame_stride;  // bytes between frames
  int row_stride, channels, src_w, src_h;
  uint8_t* out;            // [B][S_h][S_w][4] BGRX (X = 0)
  int dst_w, dst_h, new_w, new_h, pad_top, pad_left;
  // INTER_LINEAR tap tables (device): x: [new_w], y: [new_h]
  const int* x0; const int* x1; const short* ax0; const short* ax1;
  const int* y0; const int* y1; const short* by0; const short* by1;
  int identity;            // 1: no resize (new == src)
};
void launch_letterbox(const LetterboxP& p, int B, cudaStream_t s);
// YUV 4:2:0 frames (k_letterbox_yuv): lb.frames is the Y plane, lb.row_stride its row stride, lb.channels unused.  The chroma of
// frame b starts at chroma + b * c_frame_stride; the chroma sample of pixel (x, y) sits in chroma row cy0 / cy1 (the rows of
// lb.y0 / lb.y1, halved and, for a compacted upload, renumbered), byte (x >> 1) * c_step + u_off (U) / v_off (V):
// NV12 c_step 2, u_off 0, v_off 1; NV21 2, 1, 0; I420 1, 0, offset of the V plane behind the U plane.
// (A struct of its own: LetterboxP keeps its size, so k_letterbox keeps its parameter layout.)
struct LetterboxYuvP {
  LetterboxP lb;
  const uint8_t* chroma;
  long long c_frame_stride;
  int c_row_stride, c_step, u_off, v_off;
  const int* cy0; const int* cy1;
};
// p010: the frames are FDT_FMT_P010 (c_step 4, u_off 1, v_off 3: the chroma words' high bytes); launches k_letterbox_yuv<true>,
// which reads the Y sample of pixel x as byte 2x + 1 of its row.
void launch_letterbox_yuv(const LetterboxYuvP& p, int B, cudaStream_t s, bool p010 = false);
// Frames stored transposed (EXIF orientations 5-8, see fdt_detect_batch_oriented), k_letterbox_tr: the letterbox of the upright
// image U.  The tables are U's (x taps from U's width, y taps from U's height, flips folded in on the host), but the x taps,
// indexed by the output column, name stored ROWS and the y taps, indexed by the output row, stored COLUMNS.  YUV frames (yuv = 1):
// yp.cy0 / yp.cy1 are the chroma rows of lb.x0 / lb.x1 (indexed by the output column); a chroma byte sits at
// (column >> 1) * c_step.  (A struct of its own: LetterboxP and LetterboxYuvP keep their layouts.)
struct LetterboxTrP {
  LetterboxYuvP yp;
  int yuv;
};
// p010 (with yuv = 1): FDT_FMT_P010 frames, as for launch_letterbox_yuv.
void launch_letterbox_tr(const LetterboxTrP& p, int B, cudaStream_t s, bool p010 = false);
// RGB, RGBA and planar RGB frames (FDT_FMT_RGB / _RGBA / _RGB_PLANAR): every non-YUV format is a pixel step and the byte offsets
// of its B, G and R samples from the pixel's first byte (row + x * step):
//   BGR 3: 0, 1, 2   RGB 3: 2, 1, 0   BGRA 4: 0, 1, 2   RGBA 4: 2, 1, 0   GRAY 1: 0, 0, 0   planar RGB 1: 2P, P, 0
// with P the bytes of one plane as it lies on the device (after a compacted upload, the compacted plane).
// Packed YUV 4:2:2 frames (FDT_FMT_YUYV / _UYVY / _YVYU, yuv422 = 1): step 2, and b, g, r are the offsets of the pixel's Y from
// byte 2x of its row and of U and V from its 4-byte macropixel, byte 4 * (x / 2):  YUYV 0, 1, 3   UYVY 1, 0, 2   YVYU 0, 3, 1.
// They are read by load_422 (k_letterbox_rgb<., true>, k_letterbox_multi<., ., ., true>, yuv422::k_warp_affine), which needs the
// pixel's column as well as its row.
struct PixFmt {
  long long b = 0, g = 0, r = 0;
  int step = 0;            // 0: no PixFmt (the existing formats' own kernels)
  int yuv422 = 0;          // 1: packed YUV 4:2:2 (in the struct's tail padding: PixFmt keeps its 32 bytes)
};
#ifdef __CUDACC__
__device__ __forceinline__ void load_pix(const uint8_t* px, const PixFmt& f, int* v) { v[0] = px[f.b]; v[1] = px[f.g]; v[2] = px[f.r]; }
// Pixel x of a packed YUV 4:2:2 row, converted as cv::cvtColor COLOR_YUV2BGR_YUYV / _UYVY / _YVYU converts it.
__device__ __forceinline__ void load_422(const uint8_t* row, int x, const PixFmt& f, int* v) {
  const uint8_t* m = row + (size_t)(x >> 1) * 4;
  yuv_to_bgr(row[(size_t)x * 2 + f.b], m[f.g], m[f.r], v);
}
#endif
// Ragged batches (fdt_detect_frames): one descriptor per frame of a chunk.  It says where the frame's bytes are and how the
// letterbox maps it; the crop warps read the same table, indexed by WarpP::crop_img.
struct FrameD {
  const uint8_t* y;        // the packed frame, or the Y plane
  const uint8_t* c;        // YUV 4:2:0: the chroma area, addressed as in LetterboxYuvP (v_off relative to it)
  int w, h, row_stride;
  int channels;            // 1 / 3 / 4 (RGB-family frames: their pixel step); 2: packed YUV 4:2:2; 0: YUV 4:2:0
  // YUV 4:2:0: c_step 4 (u_off 1, v_off 3) is a P010 frame, 16-bit words read by their high bytes (the Y sample of pixel x at
  // byte 2x + 1 of its row); only the k16 variants (k_letterbox_multi<., ., ., ., true>, yuv16::k_warp_affine) take such frames
  int c_row_stride, c_step, u_off, v_off;
  int new_w, new_h, pad_top, pad_left, identity;
  int tx, ty;              // offsets (ints) of the frame's x taps [4][new_w] and y taps [6][new_h] in the chunk's tap table
  int orientation;         // EXIF 1..8: the upright image is exif_transform(stored frame, orientation); w, h are the stored size
};
// Separate-plane YUV 4:2:0 frames (fdt_detect_yuv_planes) in device memory whose U and V planes FrameD cannot describe (different
// strides, or more than an int apart): the chroma samples of pixel (x, y) are u[(y / 2) * u_stride + (x / 2) * ps] and
// v[(y / 2) * v_stride + (x / 2) * ps]; the frame's FrameD gives the Y plane.  One entry per frame of the chunk, in the chunk blob.
// fdt_detect_yuv_planes16 (every frame, host or device, through this table): the planes hold 16-bit words, strides count bytes,
// ps and x count samples, and shift = sample_bits - 8 (load_yuv_planes16).  8-bit frames leave shift 0 and unread.
struct YuvPlaneD {
  const uint8_t* u;
  const uint8_t* v;
  int u_stride, v_stride, ps, shift;
};
#ifdef __CUDACC__
__device__ __forceinline__ void load_yuv_planes(const uint8_t* yrow, int crow, int x, const YuvPlaneD& q, int* v) {
  const size_t cx = (size_t)(x >> 1) * q.ps;
  yuv_to_bgr(yrow[x], q.u[(size_t)crow * q.u_stride + cx], q.v[(size_t)crow * q.v_stride + cx], v);
}
// The 8-bit sample of a 16-bit word with shift + 8 significant bits from bit 0: (s >> shift) & 0xFF (truncation; bits above the
// significant ones are ignored).
__device__ __forceinline__ int sample16(const uint8_t* p, int shift) { return (*reinterpret_cast<const uint16_t*>(p) >> shift) & 0xFF; }
// load_yuv_planes over planes of 16-bit words: every sample reduced to 8 bits first, then the 8-bit conversion.
__device__ __forceinline__ void load_yuv_planes16(const uint8_t* yrow, int crow, int x, const YuvPlaneD& q, int* v) {
  const size_t cx = (size_t)(x >> 1) * q.ps * 2;
  yuv_to_bgr(sample16(yrow + (size_t)x * 2, q.shift), sample16(q.u + (size_t)crow * q.u_stride + cx, q.shift),
             sample16(q.v + (size_t)crow * q.v_stride + cx, q.shift), v);
}
#endif
// k_letterbox_multi: k_letterbox / k_letterbox_yuv per frame.  taps (host-built, resize_linear_taps): per distinct size and
// orientation x0, x1, ax0, ax1 (new_w each), then y0, y1, by0, by1, cy0, cy1 (new_h each; cy = y / 2, read for YUV frames only),
// all of the upright image with the flips folded in.  transposed = true launches the variant that also takes frames of
// orientations 5-8 (their x taps name stored rows, as in k_letterbox_tr); a chunk without such frames runs the plain one.
struct LetterboxMultiP {
  const FrameD* fr;        // [B]
  const int* taps;
  uint8_t* out;            // [B][S_h][S_w][4] BGRX
  int dst_w, dst_h;
};
// pf (device, [B]): the chunk holds an RGB / RGBA / planar RGB frame, and pf[b] is frame b's PixFmt (offsets from FrameD::y, whole
// frames; unused for YUV frames), FrameD::channels its pixel step.  Non-null launches the variant that reads every packed or planar
// frame through pf, whatever its orientation.  (A kernel argument of its own, behind B: FrameD and LetterboxMultiP keep their
// sizes, which the existing variants' code depends on.)
// pl (device, [B]): the chunk's frames are all separate-plane YUV frames read through their YuvPlaneD (any orientation; pf null).
// (A kernel argument of its own, behind pfs, for the same reason.)
// yuv422: the chunk holds a packed YUV 4:2:2 frame (pf non-null); launches the variant that also knows that pixel rule.
// yuv16: the chunk holds a P010 frame (FrameD::c_step 4), or its frames are fdt_detect_yuv_planes16 frames (pl non-null, every
// frame's shift set); launches the k16 variant, which reduces every 16-bit sample to 8 bits before the conversion.
void launch_letterbox_multi(const LetterboxMultiP& p, int B, bool transposed, cudaStream_t s, const PixFmt* pf = nullptr,
                            const YuvPlaneD* pl = nullptr, bool yuv422 = false, bool yuv16 = false);
// k_letterbox_rgb: k_letterbox (transposed = 0) or k_letterbox_tr (transposed = 1, orientations 5-8) with every tap read through
// pf; lb.channels unused.  pf.yuv422 launches the instantiation that reads the taps with load_422.  (A struct of its own: the
// existing parameter blocks keep their layouts.)
struct LetterboxRgbP {
  LetterboxP lb;
  PixFmt pf;
};
void launch_letterbox_rgb(const LetterboxRgbP& p, int B, bool transposed, cudaStream_t s);
// u8 [B][S][S][4] BGRX -> f32 [B][S][S][3] RGB, v*(1/127.5)-1
void launch_normalize(const uint8_t* in, TV out, int B, cudaStream_t s);

// ---- stem: k x k / stride 2 conv of the u8x4 BGRX image (normalise + BGR->RGB on load) ----
struct StemP {
  const uint8_t* in8;       // [B][H][W][4] BGRX
  int H, W, OH, OW, kw, pt, pl, K, KP;
  float* out; long long out_istride; int Cout, CoutS, vec_store;
  const float* w;           // [KP][CoutP], row k = (ky*kw + kx)*3 + c
  const float* bias; const float* alpha;
  int act, CoutP, NC;
  size_t smem_bytes;
};
void launch_stem(const StemP& p, int B, cudaStream_t s, int max_ctas);

// ---- tiled conv kernels: im2col + register-tiled fp32 GEMM ----
struct GemmConvP {
  const float* in;          // f32 NHWC (or nullptr when in8 is used)
  const uint8_t* in8;       // u8 [B][H][W][4] BGRX image: normalised + swapped on load
  long long in_istride;
  int H, W, Cin, CinS;
  int kh, kw, sh, sw, pt, pl, OH, OW;
  int K, KP, KS;
  float* out; long long out_istride; int Cout, CoutS, vec_store;
  const float* w;           // [KP][CoutP], row k = (ky,kx,c)
  const float* bias;        // [CoutP]
  const float* alpha;       // [CoutP] or nullptr
  int act, CoutP, NC, nchunks, NPG, TM;
  int flat;                 // 1: the kernel window is the whole (dense) input image -> im2col row = plain copy
  FastDiv fd_KP, fd_kwc, fd_Cin, fd_OW, fd_OH, fd_NQ;
  size_t smem_bytes;
};
void launch_gemm_conv(const GemmConvP& p, int B, cudaStream_t s, int max_ctas);

// ---- fused BlazeBlock: [DW3x3] -> PW1x1 + bias [+ residual(maxpool, channel pad)] + act ----
struct DwPwP {
  const float* in; long long in_istride; int H, W, Cin, CinS;
  int has_dw, s, dpt, dpl, OH, OW;
  const float* dww;         // [9][KP]
  const float* dwb;         // [KP]
  int KP, KS;
  float* out; long long out_istride; int Cout, CoutS, vec_store;
  const float* w;           // [KP][CoutP]
  const float* bias; const float* alpha;
  int act, CoutP, NC, nchunks, NPG, TM;
  const float* res; long long res_istride; int res_H, res_W, res_C, res_Cs, res_pool;
  int res_mode;             // 0 none, 1 from the staged input tile (shared memory), 2 from global
  int TH, TW, G, IH, IW, tilesX, tilesY;
  FastDiv fd_Q, fd_IW, fd_IH, fd_TW, fd_thw, fd_NQ, fd_tpg, fd_tilesX;
  size_t smem_bytes;
};
void launch_dwpw(const DwPwP& p, int B, cudaStream_t s, int max_ctas);

// ---- fused BlazeBlock with the pointwise conv on tcgen05 tensor cores (TF32 hi/lo split) ----
struct DwPwTcP {
  const float* in; long long in_istride; int H, W, Cin, CinS;
  int has_dw, s, dpt, dpl, OH, OW;
  const float* dww;         // [9][K8]
  const float* dwb;         // [K8]
  int K8, KS;               // K padded to 8; smem pixel stride of the staged tile
  float* out; long long out_istride; int Cout, CoutS, vec_store;
  const float* wB;          // [Npad x K8] in the UMMA K-major core-matrix layout
  const float* bias; const float* alpha;   // [Npad]
  int act, Npad, tmem_cols, a_rows, RS;
  int in_floats, n_chunks, n_items;   // staged tile size (floats), staging-table / depthwise-table entries
  int nr, KSr, res_stage_floats;      // residual from another HBM tensor staged by TMA: ring stages (0 = direct loads), record stride, floats per stage
  int deint, plane_floats, PW;        // stride 2: the stage holds the even and the odd input columns as two planes [G][IH][PW][KS] (see kernels_ts.cu)
  int w_parts;              // 1: weights exact in TF32; 2: W = W_hi + W_lo (fp32 weights), wB holds both
  int nbuf;                 // 2: double-buffered input tile (the next tile is prefetched during compute)
  int ns, na, nd, nt;       // k_block_ws: input ring stages, A-operand buffers, depthwise warps, TMEM accumulators
  int no, KSo, out_stage_floats;   // k_block_ws TMA-store epilogue: output tile buffers (0 = direct stores), its pixel stride, floats per buffer
  float* out2; long long out2_istride; int Cs2, c1, c2;   // second output of a merged head pair (c2 == 0: none)
  long long* trace;         // FDT_WS_TRACE=1: per-role clock64 stamps of CTA 0 ([4 roles][64 tiles][3]); null in production
  const float* res; long long res_istride; int res_H, res_W, res_C, res_Cs, res_pool, res_mode, res_lim;
  int TH, TW, G, IH, IW, tilesX, tilesY;
  FastDiv fd_Q8, fd_IW, fd_IH, fd_TW, fd_thw, fd_tpg, fd_tilesX, fd_nstrips, fd_nslots;
  size_t smem_bytes;
};
// warp-specialised TMA / mbarrier pipeline version (kernels_ws.cu); `cap` = images the input tensor is allocated for.
// Returns false when the tensor map could not be encoded (nothing launched).
bool launch_block_ws(const DwPwTcP& p, int B, int cap, cudaStream_t s);

// ---- stem, warp-specialised: TMA patch ring -> exact fp16 im2col (16-byte copies) -> tcgen05 kind::f16 ----
struct StemWsP {
  const uint8_t* in8;       // [cap][H][W][4] BGRX
  int H, W, OH, OW, kw, pt, pl;
  float* out; long long out_istride; int Cout, CoutS, vec_store;
  const float* wB;          // w_parts x [Npad x K8] fp16, UMMA K-major core-matrix layout (see plan.cpp)
  const float* bias; const float* alpha;
  int act, Npad, K8, tmem_cols, w_parts;
  float out_scale;
  size_t smem_bytes;
};
bool launch_stem_ws(const StemWsP& p, int B, int cap, cudaStream_t s);

// ---- BlazeBlock with the GEMM operand in tensor memory (kernels_ts.cu): fp16-weight detectors, K16 <= 64, Npad <= 64 ----
struct BlockTsP {
  const float* in; long long in_istride; int H, W, CinS;
  float* out; long long out_istride; int OH, OW, CoutS;
  const float* rec;         // [W fp16 Npad x K16 (UMMA K-major core matrices) | depthwise taps 9 x K16 | depthwise bias K16]
  const float* bias;        // pointwise bias [Npad]
  int rec_bytes;
  int Cin, K16, Npad, KS;   // KS: staged pixel stride (floats), an odd number of 16-byte quads
  int stride;               // depthwise stride 1 (16x16 output tiles) or 2 (8x16)
  int res;                  // 0 none, 1 the block input, 2 its 2x2 max-pool (stride 2); zero channel pad either way
  int relu, wide;           // wide: pixel records 32-byte aligned -> 256-bit stores
  int ns, stage_bytes;      // input ring
  size_t smem_bytes;
  // depthwise taps and bias once more, quad-major ([16 quads][9 taps + bias][4 channels]), as KERNEL PARAMETERS: the taps of a channel quad are the same for every lane, and as
  // broadcast LDS.128 they made up 40 of the 88 shared-memory wavefronts per quad and pixel pair; from the constant bank they cost none
  alignas(16) float dw[10 * 64];
};
size_t ts_smem_bytes(int rec_bytes, int Npad, int ns, int stage_bytes);
bool launch_block_ts(const BlockTsP& p, int B, int cap, cudaStream_t s);

// ---- image-resident tail (kernels_tail.cu): every 16x16 / 8x8 BlazeBlock and both head pairs in one launch ----
struct TailP {
  const float* in; long long in_istride; int H, W, CinS;   // first layer's input activation (HBM, NHWC f32) -> buffer 0 by TMA
  const float* blob;            // the engine's weight blob
  const TailLayerD* layers;     // device copy of the layer program
  int nlayers;
  int nbuf;                     // shared-memory activation buffers
  int buf_off[kTailMaxBufs];    // float offset of each inside the activation area
  int buf_ks[kTailMaxBufs];     // pixel stride (floats): an odd number of 16-byte quads
  int act_floats;               // size of the activation area
  int in_bytes;                 // bytes the TMA of one image delivers into buffer 0
  int last_a_layer;             // last layer that touches buffer 0 (the next image's input is fetched after it)
  int wbuf_bytes, wdepth;       // pointwise-weight ring: wdepth (1 or 2) buffers of wbuf_bytes
  int tbuf_bytes;               // depthwise-record ring (always two deep)
  int generic;                  // 1: the program needs the GEN = true kernel (see kernels_tail.cu); 2: k_chain_wide
  // k_chain_wide only: W block table (device), shared-memory bias area, residual tensors read from HBM
  const TailBlk* blks; int nblks; int bias_floats; int in_px;
  const float* rsrc[2]; long long rs_istride[2]; int rs_cs[2], rs_w[2], rs_c[2];
  float* outs[4]; long long out_istride[4]; int out_pix[4];   // HBM tensors the layers write: image 0, floats per image / per pixel
  size_t smem_bytes;
};
size_t tail_smem_bytes(int act_floats, int wbuf_bytes, int wdepth, int tbuf_bytes);
size_t wide_smem_bytes(int act_floats, int wbuf_bytes, int wdepth, int tbuf_bytes, int bias_floats);
bool launch_tail_ws(const TailP& p, int B, int cap, cudaStream_t s);

// ---- k_fc_tc (kernels_fc.cu): whole-map convolution = one dense contraction per image, tcgen05 GEMM over the chunk ----
struct FcP {
  const float* in; long long in_istride;     // [B][K] (the NHWC map, Cs == C, read as one row)
  float* out; long long out_istride;         // [B][N]
  const float* w;                            // per 128-channel tile: [w_parts][128][K16] fp16, UMMA K-major core matrices
  const float* bias;                         // [N]
  int K, K16, N, w_parts, tile_bytes;
  float wscale;
};
bool launch_fc_tc(const FcP& p, int B, cudaStream_t s);

// ---- JPEG front end (kernels_jpeg.cu): coefficients -> component planes -> BGR frame ----
struct JpegIdctP {
  const int16_t* coef;      // [bh][bw][64] quantised coefficients, natural order
  const uint16_t* q;        // [64] quantisation table, natural order
  int bw, bh;
  uint8_t* plane; int pitch;   // [bh * 8][pitch = bw * 8]
};
struct JpegColorP {
  const uint8_t* py; const uint8_t* pcb; const uint8_t* pcr;
  int pitch_y, pitch_c;
  int W, H, ncomp;
  int cdw, cdh, hs, vs;     // chroma plane size in samples, subsampling factors (1 or 2)
  int orientation;          // EXIF 1..8
  uint8_t* out; int out_w;  // packed BGR, out_w = W (orientations 1-4) or H (5-8)
};
void launch_jpeg_idct(const JpegIdctP& p, cudaStream_t s);
void launch_jpeg_color(const JpegColorP& p, cudaStream_t s);

// ---- detector post-processing: one block per image ----
struct DecodeP {
  const float* boxes; long long boxes_istride;    // [B][N][16]
  const float* scores; long long scores_istride;  // [B][N]
  const double* anchors;                          // [N][2]
  int N, input_h;
  double raw_thresh, score_thresh, iou_thresh;
  double pad_t, pad_b, pad_l, pad_r;              // normalised letterbox padding
  double min_score, min_face_size, img_w, img_h;
  int max_faces;
  fdt_face* faces;                                // [B][max_faces]
  int* counts;                                    // [B]
  int* cand_idx; int cand_cap; int* cand_n;       // debug taps (may be null)
  // test hooks (fdt_debug_decode / fdt_debug_nms); null / 0 in production
  const double* pre;                              // [B][N][17] already decoded detections (box4, score, kp12): skips threshold + decode
  double* dbg_dec;                                // [B][N][18] decoded candidates in anchor order: box4, score, kp12, kept flag
  int skip_roi;                                   // 1: keep faces whose alignment ROI is degenerate (round(size) <= 0)
  // ragged batches: [B][6] = pad_t, pad_b, pad_l, pad_r, img_w, img_h per image; null: the scalars above
  const double* geom = nullptr;
};
size_t decode_smem_bytes(int N);
void launch_decode_nms(const DecodeP& p, int B, cudaStream_t s);

// ---- aligned crops: cv::warpAffine(INTER_LINEAR, BORDER_CONSTANT 0) of a list of ROIs ----
// The ROI list (source image + inverse affine map per crop) is built on the host from the detections /
// mesh points with the host libm, exactly as the reference does (extractAlignedSquare, helpers.dart:583-625).
struct WarpP {
  const uint8_t* frames; long long frame_stride; int row_stride, channels, src_w, src_h;
  const int* crop_img;     // [ncrops] frame index inside `frames`
  const double* affine;    // [ncrops][6] inverse map (dst -> src), cv::warpAffine convention
  int ncrops, out_size;
  int flip_odd;            // 1: odd crops are mirrored horizontally (cv.flip(rightEye, 1), face_detector_core.dart:567)
  uint8_t* crops;          // [ncrops][out][out][4] BGRX
  // yuv = 1: YUV 4:2:0 frames (channels unused), `frames` dense: chroma at frame + c_off, addressed as in LetterboxP
  int yuv = 0;
  long long c_off = 0;
  int c_row_stride = 0, c_step = 0, u_off = 0, v_off = 0;
  // ragged batches: the frame of crop f is fr[crop_img[f]] (its layout and size replace the fields above); null: uniform
  const FrameD* fr = nullptr;
  // EXIF orientation of the frames (fdt_detect_batch_oriented): src_w / src_h are then the upright size, and each in-frame tap
  // of the upright image is mapped to its stored pixel right before the load.  Ragged: 1 when every frame of the chunk is
  // upright, else 0 (each frame's own FrameD::orientation applies).  Anything but 1 launches the oriented instantiation.
  int orientation = 1;
  // RGB / RGBA / planar RGB frames (device memory): uniform, pf[0] is the frames' PixFmt (whole frames); ragged, pf is the chunk's
  // table (k_letterbox_multi's), indexed like fr.  Non-null launches the format-aware instantiation, which reads every packed or
  // planar frame's taps through it; out-of-frame taps stay BGR 0.  (One pointer: a larger WarpP changes the code the compiler
  // makes for the existing instantiations.)
  const PixFmt* pf = nullptr;
};
// Face crops of the detect calls (fdt_set_face_crops): the warp's epilogue writes crop f of the pass as crop first + f of a packed
// arena, in the caller's layout (FDT_CROP_* flags: RGB channel order, CHW planes, f32 = (float)u8 * scale[c] + bias[c] rounded
// per operation, c in output order), instead of BGRX into WarpP::crops.  (A kernel argument of its own: WarpP has no room left.)
struct CropOutP {
  void* dst = nullptr;
  long long first = 0;
  int layout = 0;
  float scale[3] = {1.f, 1.f, 1.f}, bias[3] = {0.f, 0.f, 0.f};
};
// pl: ragged chunks of separate-plane YUV frames (k_letterbox_multi's table, indexed like fr); non-null launches the instantiation
// that reads every frame's chroma through it.  (A kernel argument of its own: WarpP has no room left, see pf.)
// out: non-null launches the face-crop instantiation that writes the packed arena out->dst (WarpP::crops and flip_odd unused).
// yuv422: the frame (uniform) or some frame of the chunk (ragged) is packed YUV 4:2:2 (p.pf non-null); launches the crop warps of
// kernels_warp422.cu, which read such frames with load_422.  (WarpP has no room for the flag, see pf.)
// yuv16: the frame (uniform) or some frame of the chunk (ragged) is P010 (c_step 4), or pl holds fdt_detect_yuv_planes16 frames;
// launches the crop warps of kernels_warp16.cu, which reduce every 16-bit sample to 8 bits before the conversion.
void launch_warp_affine(const WarpP& p, cudaStream_t s, const YuvPlaneD* pl = nullptr, const CropOutP* out = nullptr,
                        bool yuv422 = false, bool yuv16 = false);
// kernels_warp422.cu: yuv422::k_warp_affine on launch_warp_affine's grid (out: the face-crop epilogue, else BGRX crops).
void launch_warp_affine_422(const WarpP& p, dim3 grid, cudaStream_t s, const CropOutP* out);
// kernels_warp16.cu: yuv16::k_warp_affine on launch_warp_affine's grid (pl: the plane table of fdt_detect_yuv_planes16 frames).
void launch_warp_affine_16(const WarpP& p, dim3 grid, cudaStream_t s, const YuvPlaneD* pl, const CropOutP* out);

// ---- mesh / iris post-processing ----
struct MeshPostP {
  const float* raw; long long raw_istride;     // [F][1404]
  const float* flag; long long flag_istride;   // [F][1]
  const double* roi;                           // [F][6] theta, cx, cy, size, cos(theta), sin(theta) (host libm)
  int nfaces, in_size;
  float* mesh_out;                             // [F][1404] absolute pixels
  double* score_out;                           // [F]
  double* eye_corners;                         // [F][8] mesh points 33, 133, 362, 263 (x, y) in f64 (eyeRoisFromMesh input)
};
void launch_mesh_post(const MeshPostP& p, cudaStream_t s);

struct IrisPostP {
  const float* contours; long long contours_istride;   // [2F][213] eye contour + brow points of each eye crop (input-pixel units)
  const float* iris; long long iris_istride;           // [2F][15]  iris points
  const double* roi;                                   // [2F][6] theta, cx, cy, size, cos, sin per eye (even = left, odd = right/flipped)
  int nfaces, in_size;
  double img_w, img_h;
  const double* img_wh = nullptr;                      // ragged batches: [F][2] frame size per face; null: img_w, img_h
  float* iris_out;                                    // [F][456] 76 points of the left eye then 76 of the right, absolute pixels
  double* eye_kp;                                      // [F][4] iris-refined leftEye / rightEye keypoints, normalised
};
void launch_iris_post(const IrisPostP& p, cudaStream_t s);

}  // namespace fdt
