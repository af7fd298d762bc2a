// Host build of csrc/ops.cu (softsplat, the 81-displacement volumes, the tiled K = 51 separable convolution - kernels with
// shared-memory tiles and __syncthreads) through cuda_shim_block.h: every block on a host thread, its threads as fibers.
#include "cuda_shim_block.h"

#include <string>

#include "../../comfyui-frame-interpolation_b200/csrc/vfi_internal.h"
namespace vfi {
void set_error(const std::string&) {}
}
#include "../../comfyui-frame-interpolation_b200/csrc/ops.cu"

extern "C" {
int emu_softsplat(const float* in, const float* flow, float* out, int N, int C, int H, int W) {
  return (int)vfi::launch_softsplat_sum(in, flow, out, N, C, H, W, nullptr);
}
int emu_softsplat_weighted(const float* in, const float* flow, const float* metric, int mode, int eps, float* out, float* norm,
                          int N, int C, int H, int W) {
  return (int)vfi::launch_softsplat_weighted(in, flow, metric, mode, eps, out, norm, N, C, H, W, nullptr);
}
int emu_softsplat_weighted_nhwc(const float* in, const float* flow, const float* metric, int mode, int eps, float* out, float* norm,
                               float* sa, float* sb, int N, int C, int H, int W) {
  return (int)vfi::launch_softsplat_weighted_nhwc(in, flow, metric, mode, eps, out, norm, sa, sb, N, C, H, W, nullptr);
}
int emu_volume81_warp(int dot, const float* one, const float* two, float* out, float* sa, float* sb, int N, int C, int H, int W) {
  return (int)vfi::launch_volume81_warp(dot != 0, one, two, out, sa, sb, N, C, H, W, nullptr);
}
int emu_volume81(int dot, const float* one, const float* two, float* out, int N, int C, int H, int W) {
  return (int)vfi::launch_volume81(dot != 0, one, two, out, N, C, H, W, nullptr);
}
int emu_sepconv(const float* in, const float* ver, const float* hor, float* out, int N, int C, int H, int W, int Kv, int Kh) {
  return (int)vfi::launch_sepconv(in, ver, hor, out, N, C, H, W, Kv, Kh, nullptr);
}
// the forms that VFI_OPS_TILED / VFI_SEPCONV_PY select, chosen per call (the environment is read once per process)
int emu_volume81_form(int tiled, int dot, const float* one, const float* two, float* out, int N, int C, int H, int W) {
  return (int)vfi::launch_volume81_form(tiled != 0, dot != 0, one, two, out, N, C, H, W, nullptr);
}
int emu_sepconv_form(int py, const float* in, const float* ver, const float* hor, float* out, int N, int C, int H, int W, int Kv,
                     int Kh) {
  return (int)vfi::launch_sepconv_form(py, in, ver, hor, out, N, C, H, W, Kv, Kh, nullptr);
}
}
