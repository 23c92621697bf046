// Crop warps over chunks that hold a 16-bit YUV 4:2:0 frame (FDT_FMT_P010, fdt_detect_yuv_planes16): k_warp_affine of
// warp_affine.cuh with kWarp16 = true, as yuv16::k_warp_affine.  Every 16-bit sample is reduced to 8 bits before the conversion, the
// other frames of a mixed chunk are read as in kernels_post.cu and kernels_warp422.cu, so a crop equals the crop of the 8-bit
// frame.  A translation unit of its own, so that kernels_post.cu's k_warp_affine instantiations keep their names and code.
#include "fdt_math.h"
#include "kernels.h"

namespace fdt {
namespace {
namespace yuv16 {

constexpr bool kWarpYuv422 = true;   // a mixed chunk may hold a packed YUV 4:2:2 frame next to a P010 one
constexpr bool kWarp16 = true;
#include "warp_affine.cuh"

template <bool kOut> void launch(const WarpP& p, dim3 grid, cudaStream_t s, const YuvPlaneD* pl, const CropOutP& o) {
  const bool oriented = p.orientation != 1;
  if (pl) {
    // fdt_detect_yuv_planes16: every frame through the plane table
    if (oriented) k_warp_affine<true, true, false, true, kOut><<<grid, 256, 0, s>>>(p, pl, o);
    else k_warp_affine<true, false, false, true, kOut><<<grid, 256, 0, s>>>(p, pl, o);
  } else if (p.pf) {
    // a mixed chunk that also holds RGB-family or packed YUV 4:2:2 frames
    if (oriented) k_warp_affine<true, true, true, false, kOut><<<grid, 256, 0, s>>>(p, nullptr, o);
    else k_warp_affine<true, false, true, false, kOut><<<grid, 256, 0, s>>>(p, nullptr, o);
  } else if (p.fr) {
    if (oriented) k_warp_affine<true, true, false, false, kOut><<<grid, 256, 0, s>>>(p, nullptr, o);
    else k_warp_affine<true, false, false, false, kOut><<<grid, 256, 0, s>>>(p, nullptr, o);
  } else {
    if (oriented) k_warp_affine<false, true, false, false, kOut><<<grid, 256, 0, s>>>(p, nullptr, o);
    else k_warp_affine<false, false, false, false, kOut><<<grid, 256, 0, s>>>(p, nullptr, o);
  }
}

}  // namespace yuv16
}  // namespace

void launch_warp_affine_16(const WarpP& p, dim3 grid, cudaStream_t s, const YuvPlaneD* pl, const CropOutP* out) {
  if (out) yuv16::launch<true>(p, grid, s, pl, *out);
  else yuv16::launch<false>(p, grid, s, pl, CropOutP());
}

}  // namespace fdt
