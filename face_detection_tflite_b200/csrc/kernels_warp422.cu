// Crop warps over chunks that hold a packed YUV 4:2:2 frame (FDT_FMT_YUYV / _UYVY / _YVYU): k_warp_affine of warp_affine.cuh with
// kWarpYuv422 = true, as yuv422::k_warp_affine<kRagged, kOriented, true, false, kOut>.  Every frame is read through its PixFmt;
// a 4:2:2 frame's taps with load_422, the others' as in kernels_post.cu, so a crop equals the crop of the BGR image.  A
// translation unit of its own, so that kernels_post.cu's k_warp_affine instantiations keep their names and code.
#include "fdt_math.h"
#include "kernels.h"

namespace fdt {
namespace {
namespace yuv422 {

constexpr bool kWarpYuv422 = true;
constexpr bool kWarp16 = false;
#include "warp_affine.cuh"

template <bool kOut> void launch(const WarpP& p, dim3 grid, cudaStream_t s, const CropOutP& o) {
  if (p.orientation != 1) {
    if (p.fr) k_warp_affine<true, true, true, false, kOut><<<grid, 256, 0, s>>>(p, nullptr, o);
    else k_warp_affine<false, true, true, false, kOut><<<grid, 256, 0, s>>>(p, nullptr, o);
  } else {
    if (p.fr) k_warp_affine<true, false, true, false, kOut><<<grid, 256, 0, s>>>(p, nullptr, o);
    else k_warp_affine<false, false, true, false, kOut><<<grid, 256, 0, s>>>(p, nullptr, o);
  }
}

}  // namespace yuv422
}  // namespace

void launch_warp_affine_422(const WarpP& p, dim3 grid, cudaStream_t s, const CropOutP* out) {
  if (out) yuv422::launch<true>(p, grid, s, *out);
  else yuv422::launch<false>(p, grid, s, CropOutP());
}

}  // namespace fdt
