// k_warp_affine: cv::warpAffine(INTER_LINEAR, BORDER_CONSTANT 0) of a list of ROIs into square crops.  Included by
// kernels_post.cu with kWarpYuv422 = kWarp16 = false (the crop warps of every 8-bit format but packed YUV 4:2:2), by
// kernels_warp422.cu, inside namespace yuv422, with kWarpYuv422 = true (a chunk or frame that holds packed YUV 4:2:2), and by
// kernels_warp16.cu, inside namespace yuv16, with both true (a chunk or frame that holds 16-bit YUV 4:2:0), so every translation
// unit compiles the same source and the first keeps its code.  Both compile with -fmad=false: the f64 map is evaluated operation by operation.
// Included inside an anonymous namespace of fdt, after kernels.h and fdt_math.h.

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
// kWarpYuv422 (a constexpr bool of the including scope): with kFmt, a frame whose PixFmt says yuv422 has its taps read with
// load_422 (the stored column, after the orientation mapping, picks the macropixel).
// kWarp16 (a constexpr bool of the including scope): a YUV 4:2:0 frame with c_step 4 is P010 (its Y sample the high byte of the
// word, byte 2x + 1; the chroma offsets already name high bytes), and kPlanes frames are fdt_detect_yuv_planes16 frames
// (load_yuv_planes16).  Every sample is 8-bit before yuv_to_bgr, so a crop equals the crop of the 8-bit frame.
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
        if (kWarp16) load_yuv_planes16(src + (size_t)yy * row_stride, yy >> 1, xx, q, v);
        else load_yuv_planes(src + (size_t)yy * row_stride, yy >> 1, xx, q, v);
        acc[0] += v[0] * iw[t]; acc[1] += v[1] * iw[t]; acc[2] += v[2] * iw[t];
        continue;
      }
      if (kRagged ? d->channels == 0 : p.yuv) {
        const uint8_t* c = (kRagged ? d->c : src + p.c_off) + (size_t)(yy >> 1) * (kRagged ? d->c_row_stride : p.c_row_stride) +
                           (size_t)(xx >> 1) * (kRagged ? d->c_step : p.c_step);
        int v[3];
        const int ys = kWarp16 && (kRagged ? d->c_step : p.c_step) == 4 ? src[(size_t)yy * row_stride + (size_t)xx * 2 + 1]
                                                                          : src[(size_t)yy * row_stride + xx];
        yuv_to_bgr(ys, c[kRagged ? d->u_off : p.u_off], c[kRagged ? d->v_off : p.v_off], v);
        acc[0] += v[0] * iw[t]; acc[1] += v[1] * iw[t]; acc[2] += v[2] * iw[t];
        continue;
      }
      const int channels = kRagged ? d->channels : p.channels;
      const uint8_t* px = src + (size_t)yy * row_stride + (size_t)xx * channels;
      if (kFmt) {
        int v[3];
        if (kWarpYuv422 && pf.yuv422) load_422(src + (size_t)yy * row_stride, xx, pf, v);
        else load_pix(px, pf, v);
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

