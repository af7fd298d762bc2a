// The reference's custom CUDA ops (vfi_models/ops/cupy_ops, CUDA-C strings JIT-compiled through cupy/NVRTC), rebuilt as
// ahead-of-time sm_100a kernels behind the C ABI.  Same tensor contract as the reference: contiguous NCHW fp32.
//   softsplat_sum  : forward summation splat                      cupy_ops/softsplat.py:140-192
//   costvol_l1     : 9x9 L1 cost volume (81 ch)                   cupy_ops/costvol.py:4-43
//   corr_dot       : 9x9 dot-product correlation (81 ch)          cupy_ops/correlation.py:4-99
//   sepconv        : adaptive separable convolution, Kahan sums   cupy_ops/sepconv.py:86-117
// One thread per pixel computes everything that does not depend on the channel ONCE (the reference launches one
// thread per (pixel, channel) and recomputes flow taps / weights C times) and keeps the 81 volume entries in registers.
// The volume and sepconv kernels stage their input window in shared memory (zero fill outside the image = the
// reference's boundary rule) so that the inner loops are LDS + FMA only; sepconv additionally keeps each pixel's 51
// horizontal weights in registers and shares every loaded input value between vertically stacked output pixels.
#include <cstdlib>

#include "vfi_internal.h"

namespace vfi {
namespace {

// Top-left corner (x0, y0) of the four targets of a splat source moved to (fx, fy); false when none of them is in the
// image.  The test is made on the floored floats, so the int conversion only sees values in [-1, W) x [-1, H): a flow of
// 2^31 or more converts to INT_MAX on the GPU (saturation), and x0 + 1 would then overflow, which the compiler is free to
// assume never happens (it tests x0 + 1 >= 0 as x0 > -2 next to a wrapped x0 + 1 < W, accepting x1 = INT_MIN).
__device__ __forceinline__ bool splat_corner(float fx, float fy, int W, int H, int& x0, int& y0) {
  const float lx = floorf(fx), ly = floorf(fy);
  if (!(lx >= -1.f && lx < (float)W && ly >= -1.f && ly < (float)H)) return false;
  x0 = (int)lx;
  y0 = (int)ly;
  return true;
}

__global__ void softsplat_sum_kernel(const float* __restrict__ in, const float* __restrict__ flow,
                                     float* __restrict__ out, int N, int C, int H, int W) {
  const size_t hw = (size_t)H * W;
  const size_t total = (size_t)N * hw;
  for (size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x; id < total; id += (size_t)gridDim.x * blockDim.x) {
    const int x = (int)(id % W);
    const int y = (int)((id / W) % H);
    const int n = (int)(id / hw);
    const size_t pix = (size_t)y * W + x;
    const float fx = (float)x + __ldg(flow + ((size_t)n * 2 + 0) * hw + pix);
    const float fy = (float)y + __ldg(flow + ((size_t)n * 2 + 1) * hw + pix);
    if (!isfinite(fx) || !isfinite(fy)) continue;  // softsplat.py:158-159
    int x0, y0;
    if (!splat_corner(fx, fy, W, H, x0, y0)) continue;
    const int x1 = x0 + 1, y1 = y0 + 1;
    const float wnw = ((float)x1 - fx) * ((float)y1 - fy);
    const float wne = (fx - (float)x0) * ((float)y1 - fy);
    const float wsw = ((float)x1 - fx) * (fy - (float)y0);
    const float wse = (fx - (float)x0) * (fy - (float)y0);
    const bool inx0 = x0 >= 0 && x0 < W, inx1 = x1 >= 0 && x1 < W;
    const bool iny0 = y0 >= 0 && y0 < H, iny1 = y1 >= 0 && y1 < H;
    const float* src = in + (size_t)n * C * hw + pix;
    float* dst = out + (size_t)n * C * hw;
    for (int c = 0; c < C; ++c) {
      const float v = __ldg(src + (size_t)c * hw);
      float* d = dst + (size_t)c * hw;
      if (inx0 && iny0) atomicAdd(d + (size_t)y0 * W + x0, v * wnw);
      if (inx1 && iny0) atomicAdd(d + (size_t)y0 * W + x1, v * wne);
      if (inx0 && iny1) atomicAdd(d + (size_t)y1 * W + x0, v * wsw);
      if (inx1 && iny1) atomicAdd(d + (size_t)y1 * W + x1, v * wse);
    }
  }
}

// Fused avg / linear / soft splat (the wrapper modes of cupy_ops/softsplat.py:382-435 without their temporaries): the source
// pixel's weight (1, metric or exp(metric)) is applied on the fly, the weights are splatted into a one-channel `norm` plane
// next to the C channels, and a second kernel divides.  Same association of the products as the reference's
// softsplat_out on cat(in * weight, weight): (in * weight) rounded first, then times the corner weight.
__global__ void softsplat_weighted_kernel(const float* __restrict__ in, const float* __restrict__ flow,
                                          const float* __restrict__ metric, int mode, float* __restrict__ out,
                                          float* __restrict__ norm, int N, int C, int H, int W) {
  const size_t hw = (size_t)H * W;
  const size_t total = (size_t)N * hw;
  for (size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x; id < total; id += (size_t)gridDim.x * blockDim.x) {
    const int x = (int)(id % W);
    const int y = (int)((id / W) % H);
    const int n = (int)(id / hw);
    const size_t pix = (size_t)y * W + x;
    const float fx = (float)x + __ldg(flow + ((size_t)n * 2 + 0) * hw + pix);
    const float fy = (float)y + __ldg(flow + ((size_t)n * 2 + 1) * hw + pix);
    if (!isfinite(fx) || !isfinite(fy)) continue;
    const float ws = mode == 0 ? 1.f : (mode == 1 ? __ldg(metric + (size_t)n * hw + pix) : expf(__ldg(metric + (size_t)n * hw + pix)));
    int x0, y0;
    if (!splat_corner(fx, fy, W, H, x0, y0)) continue;
    const int x1 = x0 + 1, y1 = y0 + 1;
    const float wnw = ((float)x1 - fx) * ((float)y1 - fy);
    const float wne = (fx - (float)x0) * ((float)y1 - fy);
    const float wsw = ((float)x1 - fx) * (fy - (float)y0);
    const float wse = (fx - (float)x0) * (fy - (float)y0);
    const bool inx0 = x0 >= 0 && x0 < W, inx1 = x1 >= 0 && x1 < W;
    const bool iny0 = y0 >= 0 && y0 < H, iny1 = y1 >= 0 && y1 < H;
    const float* src = in + (size_t)n * C * hw + pix;
    float* dst = out + (size_t)n * C * hw;
    float* nd = norm + (size_t)n * hw;
    if (inx0 && iny0) atomicAdd(nd + (size_t)y0 * W + x0, ws * wnw);
    if (inx1 && iny0) atomicAdd(nd + (size_t)y0 * W + x1, ws * wne);
    if (inx0 && iny1) atomicAdd(nd + (size_t)y1 * W + x0, ws * wsw);
    if (inx1 && iny1) atomicAdd(nd + (size_t)y1 * W + x1, ws * wse);
    for (int c = 0; c < C; ++c) {
      const float v = __ldg(src + (size_t)c * hw) * ws;
      float* d = dst + (size_t)c * hw;
      if (inx0 && iny0) atomicAdd(d + (size_t)y0 * W + x0, v * wnw);
      if (inx1 && iny0) atomicAdd(d + (size_t)y0 * W + x1, v * wne);
      if (inx0 && iny1) atomicAdd(d + (size_t)y1 * W + x0, v * wsw);
      if (inx1 && iny1) atomicAdd(d + (size_t)y1 * W + x1, v * wse);
    }
  }
}

// eps: 0 addeps (norm + 1e-7, the default), 1 zeroeps (0 -> 1), 2 clipeps (max(norm, 1e-7))  - softsplat.py:418-431
__global__ void softsplat_normalize_kernel(float* __restrict__ out, const float* __restrict__ norm, int eps, int N, int C,
                                           size_t hw) {
  const size_t total = (size_t)N * C * hw;
  for (size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x; id < total; id += (size_t)gridDim.x * blockDim.x) {
    const size_t pix = id % hw;
    const int n = (int)(id / (hw * C));
    float d = norm[(size_t)n * hw + pix];
    d = eps == 0 ? d + 0.0000001f : (eps == 1 ? (d == 0.f ? 1.f : d) : fmaxf(d, 0.0000001f));
    out[id] = out[id] / d;
  }
}

// kDot = false: mean_c |one - two(shifted)|, outside -> mean_c |one|      (costvol)
// kDot = true : mean_c one * two(shifted), outside -> 0                   (correlation, zero padded)
template <bool kDot>
__global__ void volume81_kernel(const float* __restrict__ one, const float* __restrict__ two, float* __restrict__ out,
                                int N, int C, int H, int W) {
  const size_t hw = (size_t)H * W;
  const size_t total = (size_t)N * hw;
  for (size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x; id < total; id += (size_t)gridDim.x * blockDim.x) {
    const int x = (int)(id % W);
    const int y = (int)((id / W) % H);
    const int n = (int)(id / hw);
    float acc[81];
#pragma unroll
    for (int k = 0; k < 81; ++k) acc[k] = 0.f;
    for (int c = 0; c < C; ++c) {
      const float a = __ldg(one + ((size_t)n * C + c) * hw + (size_t)y * W + x);
      const float* t = two + ((size_t)n * C + c) * hw;
#pragma unroll
      for (int dy = -4; dy <= 4; ++dy) {
        const int yy = y + dy;
        const bool yin = yy >= 0 && yy < H;
#pragma unroll
        for (int dx = -4; dx <= 4; ++dx) {
          const int xx = x + dx;
          const float b = (yin && xx >= 0 && xx < W) ? __ldg(t + (size_t)yy * W + xx) : 0.f;
          const int k = (dy + 4) * 9 + (dx + 4);
          if (kDot)
            acc[k] = fmaf(a, b, acc[k]);
          else
            acc[k] += fabsf(a - b);
        }
      }
    }
    const float inv = 1.f / (float)C;
    float* o = out + (size_t)n * 81 * hw + (size_t)y * W + x;
#pragma unroll
    for (int k = 0; k < 81; ++k) o[(size_t)k * hw] = kDot ? acc[k] / (float)C : acc[k] / (float)C;
    (void)inv;
  }
}

// in [N, C, H+Kv-1, W+Kh-1], ver [N, Kv, H, W], hor [N, Kh, H, W] -> out [N, C, H, W]; C <= 4 per pass
template <int CB>
__global__ void sepconv_kernel(const float* __restrict__ in, const float* __restrict__ ver,
                               const float* __restrict__ hor, float* __restrict__ out, int N, int C, int c0, int H,
                               int W, int Kv, int Kh) {
  const size_t hw = (size_t)H * W;
  const size_t total = (size_t)N * hw;
  const int Hp = H + Kv - 1, Wp = W + Kh - 1;
  const size_t hwp = (size_t)Hp * Wp;
  for (size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x; id < total; id += (size_t)gridDim.x * blockDim.x) {
    const int x = (int)(id % W);
    const int y = (int)((id / W) % H);
    const int n = (int)(id / hw);
    const size_t pix = (size_t)y * W + x;
    float sum[CB], comp[CB];
#pragma unroll
    for (int c = 0; c < CB; ++c) sum[c] = comp[c] = 0.f;
    const float* vp = ver + (size_t)n * Kv * hw + pix;
    const float* hp = hor + (size_t)n * Kh * hw + pix;
    for (int fy = 0; fy < Kv; ++fy) {
      const float v = __ldg(vp + (size_t)fy * hw);
      for (int fx = 0; fx < Kh; ++fx) {
        const float h = __ldg(hp + (size_t)fx * hw);
#pragma unroll
        for (int c = 0; c < CB; ++c) {
          if (c0 + c < C) {
            const float i = __ldg(in + ((size_t)n * C + c0 + c) * hwp + (size_t)(y + fy) * Wp + (x + fx));
            // Kahan summation exactly as sepconv.py:103-110
            float yk = i * v * h;
            yk = yk - comp[c];
            const float t = sum[c] + yk;
            comp[c] = (t - sum[c]) - yk;
            sum[c] = t;
          }
        }
      }
    }
#pragma unroll
    for (int c = 0; c < CB; ++c)
      if (c0 + c < C) out[((size_t)n * C + c0 + c) * hw + pix] = sum[c];
  }
}


// ---- shared-memory tiled 9x9 volume: block = 32 x 8 pixels, `two` window (40 x 16) staged for kVolCh channels at a time
constexpr int kVolCh = 8;
template <bool kDot>
__global__ void __launch_bounds__(256) volume81_tile_kernel(const float* __restrict__ one, const float* __restrict__ two,
                                                            float* __restrict__ out, int N, int C, int H, int W) {
  __shared__ float tile[kVolCh][16][40];
  const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;
  const int x0 = blockIdx.x * 32, y0 = blockIdx.y * 8, n = blockIdx.z;
  const int x = x0 + lx, y = y0 + ly;
  const bool valid = x < W && y < H;
  const size_t hw = (size_t)H * W;
  float acc[81];
#pragma unroll
  for (int k = 0; k < 81; ++k) acc[k] = 0.f;
  for (int cb = 0; cb < C; cb += kVolCh) {
    const int nc = min(kVolCh, C - cb);
    __syncthreads();  // the previous chunk has been consumed
    for (int i = threadIdx.x; i < nc * 16 * 40; i += 256) {
      const int c = i / (16 * 40), r = (i / 40) % 16, q = i % 40;
      const int yy = y0 + r - 4, xx = x0 + q - 4;
      float v = 0.f;  // outside the image: 0 (correlation: zero padding; cost volume: |one - 0| = |one|, costvol.py:27-31)
      if (yy >= 0 && yy < H && xx >= 0 && xx < W) v = __ldg(two + ((size_t)n * C + cb + c) * hw + (size_t)yy * W + xx);
      tile[c][r][q] = v;
    }
    __syncthreads();
    for (int c = 0; c < nc; ++c) {
      const float a = valid ? __ldg(one + ((size_t)n * C + cb + c) * hw + (size_t)y * W + x) : 0.f;
#pragma unroll
      for (int dy = 0; dy < 9; ++dy)
#pragma unroll
        for (int dx = 0; dx < 9; ++dx) {
          const float b = tile[c][ly + dy][lx + dx];
          if (kDot)
            acc[dy * 9 + dx] = fmaf(a, b, acc[dy * 9 + dx]);
          else
            acc[dy * 9 + dx] += fabsf(a - b);
        }
    }
  }
  if (!valid) return;
  float* o = out + (size_t)n * 81 * hw + (size_t)y * W + x;
#pragma unroll
  for (int k = 0; k < 81; ++k) o[(size_t)k * hw] = acc[k] / (float)C;
}

// ------------------------------------------------------------------------------------------------------------------------
// Channel-last forms (r02).  The reference's tensors are NCHW, and both ops above pay for it: the splat issues four scalar
// atomics per (pixel, channel) into four different planes (r01 / r02 measurements: 4 - 14 % of HBM bandwidth), the volumes
// read one value per (channel, displacement) from shared memory (one LDS per multiply-add, 6.7 % of the fp32 rate).  With
// the channels of a pixel contiguous, a splat corner is ONE 16-byte vector atomic per four channels and a displacement of
// the volume is a dot product of two contiguous channel vectors, reduced over the lanes of a warp with shuffles.  The C-ABI
// keeps the reference's NCHW contract: the inputs are transposed into context-owned scratch first (coalesced both ways),
// the results are transposed back by the kernel that finishes them (normalise / the block's staging of the 81 values).

// [N, C, HW] -> [N, HW, Cp] (channels padded with zeros to Cp), 32 x 32 tiles through shared memory
__global__ void __launch_bounds__(256) nchw_to_nhwc_kernel(const float* __restrict__ src, float* __restrict__ dst, int C, int Cp,
                                                           size_t HW) {
  __shared__ float tile[32][33];
  const int n = blockIdx.z;
  const size_t p0 = (size_t)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int j = ty; j < 32; j += 8) {
    const int c = c0 + j;
    const size_t p = p0 + tx;
    tile[j][tx] = (c < C && p < HW) ? src[((size_t)n * C + c) * HW + p] : 0.f;
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    const size_t p = p0 + j;
    const int c = c0 + tx;
    if (p < HW && c < Cp) dst[((size_t)n * HW + p) * Cp + c] = tile[tx][j];
  }
}

// Soft / linear / average splat on channel-last data: thread = (source pixel, four channels); the pixel's weight (1, metric
// or exp(metric)) and its four corner weights are recomputed per thread (a handful of FLOPs against a 16-byte atomic), the
// first thread of a pixel also splats the weight into the normalisation plane.  acc [N, HW, Cp], norm [N, HW], both zeroed.
__global__ void softsplat_nhwc_kernel(const float* __restrict__ in, const float* __restrict__ flow, const float* __restrict__ metric,
                                      int mode, float* __restrict__ acc, float* __restrict__ norm, int N, int Cp, int H, int W) {
  const size_t hw = (size_t)H * W;
  const int cq = Cp >> 2;
  const size_t total = (size_t)N * hw * cq;
  for (size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x; id < total; id += (size_t)gridDim.x * blockDim.x) {
    const int q = (int)(id % cq);
    const size_t pid = id / cq;  // n * hw + pixel
    const size_t pix = pid % hw;
    const int n = (int)(pid / hw);
    const int x = (int)(pix % W), y = (int)(pix / W);
    const float fx = (float)x + __ldg(flow + ((size_t)n * 2 + 0) * hw + pix);
    const float fy = (float)y + __ldg(flow + ((size_t)n * 2 + 1) * hw + pix);
    if (!isfinite(fx) || !isfinite(fy)) continue;  // softsplat.py:158-159
    const float ws = mode == 0 ? 1.f : (mode == 1 ? __ldg(metric + pid) : expf(__ldg(metric + pid)));
    int x0, y0;
    if (!splat_corner(fx, fy, W, H, x0, y0)) continue;
    const int x1 = x0 + 1, y1 = y0 + 1;
    const float wnw = ((float)x1 - fx) * ((float)y1 - fy);
    const float wne = (fx - (float)x0) * ((float)y1 - fy);
    const float wsw = ((float)x1 - fx) * (fy - (float)y0);
    const float wse = (fx - (float)x0) * (fy - (float)y0);
    const bool inx0 = x0 >= 0 && x0 < W, inx1 = x1 >= 0 && x1 < W;
    const bool iny0 = y0 >= 0 && y0 < H, iny1 = y1 >= 0 && y1 < H;
    float4 v = __ldg(reinterpret_cast<const float4*>(in + pid * Cp) + q);
    v.x *= ws; v.y *= ws; v.z *= ws; v.w *= ws;   // (in * weight) rounded first, then times the corner weight: the reference's order
    float* base = acc + (size_t)n * hw * Cp + 4 * q;
    float* nd = norm + (size_t)n * hw;
    auto put = [&](int yy, int xx, float wc) {
      atomicAdd(reinterpret_cast<float4*>(base + ((size_t)yy * W + xx) * Cp), make_float4(v.x * wc, v.y * wc, v.z * wc, v.w * wc));
      if (q == 0) atomicAdd(nd + (size_t)yy * W + xx, ws * wc);
    };
    if (inx0 && iny0) put(y0, x0, wnw);
    if (inx1 && iny0) put(y0, x1, wne);
    if (inx0 && iny1) put(y1, x0, wsw);
    if (inx1 && iny1) put(y1, x1, wse);
  }
}

// out[n, c, p] = acc[n, p, c] / f(norm[n, p])  (eps: 0 addeps, 1 zeroeps, 2 clipeps; -1: no division = "sum" mode)
__global__ void __launch_bounds__(256) nhwc_normalize_to_nchw_kernel(const float* __restrict__ acc, const float* __restrict__ norm,
                                                                     float* __restrict__ out, int C, int Cp, size_t HW, int eps) {
  __shared__ float tile[32][33];
  const int n = blockIdx.z;
  const size_t p0 = (size_t)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int j = ty; j < 32; j += 8) {
    const size_t p = p0 + j;
    const int c = c0 + tx;
    float v = 0.f;
    if (p < HW && c < Cp) {
      v = acc[((size_t)n * HW + p) * Cp + c];
      if (eps >= 0) {
        float d = norm[(size_t)n * HW + p];
        d = eps == 0 ? d + 0.0000001f : (eps == 1 ? (d == 0.f ? 1.f : d) : fmaxf(d, 0.0000001f));
        v = v / d;
      }
    }
    tile[j][tx] = v;
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    const int c = c0 + j;
    const size_t p = p0 + tx;
    if (c < C && p < HW) out[((size_t)n * C + c) * HW + p] = tile[tx][j];
  }
}

// 9 x 9 volume on channel-last data, one WARP per output pixel, eight pixels (consecutive x) per block: for each of the 81
// displacements the lanes walk the two channel vectors 32 channels at a time (128-byte coalesced loads, the 81-fold reuse of
// `two` comes out of L1 / L2) and the lanes' partial sums are reduced with five shuffles; lane 0 parks the value in shared
// memory so that the block writes each displacement plane 32 contiguous bytes at a time.
template <bool kDot>
__global__ void __launch_bounds__(256) volume81_warp_kernel(const float* __restrict__ one, const float* __restrict__ two,
                                                            float* __restrict__ out, int C, int Cp, int H, int W) {
  __shared__ float res[81][8];
  const int lane = threadIdx.x & 31, wq = threadIdx.x >> 5;
  const int x = blockIdx.x * 8 + wq, y = blockIdx.y, n = blockIdx.z;
  const size_t hw = (size_t)H * W;
  const bool valid = x < W;
  const float* a = one + ((size_t)n * hw + (size_t)y * W + (valid ? x : 0)) * Cp;
  for (int d = 0; d < 81; ++d) {
    const int yy = y + d / 9 - 4, xx = x + d % 9 - 4;
    const bool in = valid && yy >= 0 && yy < H && xx >= 0 && xx < W;
    const float* b = two + ((size_t)n * hw + (size_t)(in ? yy : 0) * W + (in ? xx : 0)) * Cp;
    float s = 0.f;
    for (int c = lane; c < C; c += 32) {
      const float av = a[c];
      const float bv = in ? b[c] : 0.f;   // outside the image: 0 (correlation: zero padding; cost volume: |one|, costvol.py:27-31)
      s = kDot ? fmaf(av, bv, s) : s + fabsf(av - bv);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) res[d][wq] = s / (float)C;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 81 * 8; i += 256) {
    const int d = i >> 3, j = i & 7;
    const int xo = blockIdx.x * 8 + j;
    if (xo < W) out[((size_t)n * 81 + d) * hw + (size_t)y * W + xo] = res[d][j];
  }
}

// ---- shared-memory tiled separable convolution, K x K taps (K compile time), up to 4 channels per pass.
// Block = 32 x (8*PY) output pixels, 256 threads; thread (lx, ly) owns the PY vertically adjacent pixels
// (y0 + ly*PY + j, x0 + lx).  The input window of the block, (8*PY + K-1) x (32 + K-1) positions x 4 channels, sits in
// shared memory as float4 (one conflict-free LDS.128 per tap); every loaded value feeds PY pixels, whose K horizontal
// weights live in registers.  out = sum_fy ver[fy] * (sum_fx hor[fx] * in[y+fy][x+fx]): the inner sums are FMA chains,
// the outer sum over the K rows is Kahan-compensated (the reference compensates every one of the K*K additions,
// sepconv.py:103-110; both are accurately rounded fp32 sums and agree to ~1e-6 relative).
template <int K, int PY>
__global__ void __launch_bounds__(256) sepconv_tile_kernel(const float* __restrict__ in, const float* __restrict__ ver,
                                                           const float* __restrict__ hor, float* __restrict__ out,
                                                           int N, int C, int c0, int H, int W) {
  VFI_DYN_SMEM(float4, sep_tile);  // [8*PY + K-1][32 + K-1]
  constexpr int TW = 32 + K - 1, TH = 8 * PY + K - 1;
  const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;
  const int x0 = blockIdx.x * 32, y0 = blockIdx.y * (8 * PY), n = blockIdx.z;
  const int Hp = H + K - 1, Wp = W + K - 1;
  const size_t hw = (size_t)H * W, hwp = (size_t)Hp * Wp;
  const int nch = min(4, C - c0);
  for (int i = threadIdx.x; i < TH * TW; i += 256) {
    const int r = i / TW, q = i - r * TW;
    const int gy = y0 + r, gx = x0 + q;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (gy < Hp && gx < Wp) {
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (c < nch) v[c] = __ldg(in + ((size_t)n * C + c0 + c) * hwp + (size_t)gy * Wp + gx);
    }
    sep_tile[i] = make_float4(v[0], v[1], v[2], v[3]);
  }
  __syncthreads();
  const int x = x0 + lx;
  const int yb = y0 + ly * PY;  // first of this thread's PY rows
  bool ok[PY];
  float h[PY][K];
#pragma unroll
  for (int j = 0; j < PY; ++j) {
    ok[j] = (x < W) && (yb + j < H);
#pragma unroll
    for (int fx = 0; fx < K; ++fx)
      h[j][fx] = ok[j] ? __ldg(hor + ((size_t)n * K + fx) * hw + (size_t)(yb + j) * W + x) : 0.f;
  }
  float sum[PY][4], comp[PY][4];
#pragma unroll
  for (int j = 0; j < PY; ++j)
#pragma unroll
    for (int c = 0; c < 4; ++c) sum[j][c] = comp[j][c] = 0.f;
  for (int r = 0; r < K + PY - 1; ++r) {  // input row yb + r serves pixel row j with vertical tap fy = r - j
    const float4* row = sep_tile + (ly * PY + r) * TW + lx;
    float rd[PY][4];
#pragma unroll
    for (int j = 0; j < PY; ++j)
#pragma unroll
      for (int c = 0; c < 4; ++c) rd[j][c] = 0.f;
#pragma unroll
    for (int fx = 0; fx < K; ++fx) {
      const float4 a = row[fx];
#pragma unroll
      for (int j = 0; j < PY; ++j) {
        rd[j][0] = fmaf(h[j][fx], a.x, rd[j][0]);
        rd[j][1] = fmaf(h[j][fx], a.y, rd[j][1]);
        rd[j][2] = fmaf(h[j][fx], a.z, rd[j][2]);
        rd[j][3] = fmaf(h[j][fx], a.w, rd[j][3]);
      }
    }
#pragma unroll
    for (int j = 0; j < PY; ++j) {
      const int fy = r - j;
      if (fy < 0 || fy >= K || !ok[j]) continue;
      const float v = __ldg(ver + ((size_t)n * K + fy) * hw + (size_t)(yb + j) * W + x);
#pragma unroll
      for (int c = 0; c < 4; ++c) {  // Kahan step with the row's contribution
        const float yk = v * rd[j][c] - comp[j][c];
        const float t = sum[j][c] + yk;
        comp[j][c] = (t - sum[j][c]) - yk;
        sum[j][c] = t;
      }
    }
  }
#pragma unroll
  for (int j = 0; j < PY; ++j) {
    if (!ok[j]) continue;
#pragma unroll
    for (int c = 0; c < 4; ++c)
      if (c < nch) out[((size_t)n * C + c0 + c) * hw + (size_t)(yb + j) * W + x] = sum[j][c];
  }
}

inline int grid_for(size_t total, int block) {
  size_t g = (total + block - 1) / block;
  const size_t cap = 148 * 16;
  return (int)(g < cap ? (g ? g : 1) : cap);
}

}  // namespace

cudaError_t launch_softsplat_sum(const float* in, const float* flow, float* out, int N, int C, int H, int W,
                                 cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(out, 0, (size_t)N * C * H * W * sizeof(float), st);
  if (e != cudaSuccess) return e;
  const size_t total = (size_t)N * H * W;
  VFI_LAUNCH((softsplat_sum_kernel), grid_for(total, 256), 256, 0, st, in, flow, out, N, C, H, W);
  return cudaGetLastError();
}

cudaError_t launch_softsplat_weighted(const float* in, const float* flow, const float* metric, int mode, int eps, float* out,
                                      float* norm, int N, int C, int H, int W, cudaStream_t st) {
  if (mode < 0 || mode > 2 || eps < 0 || eps > 2 || (mode != 0 && metric == nullptr)) return cudaErrorInvalidValue;
  cudaError_t e = cudaMemsetAsync(out, 0, (size_t)N * C * H * W * sizeof(float), st);
  if (e != cudaSuccess) return e;
  e = cudaMemsetAsync(norm, 0, (size_t)N * H * W * sizeof(float), st);
  if (e != cudaSuccess) return e;
  VFI_LAUNCH((softsplat_weighted_kernel), grid_for((size_t)N * H * W, 256), 256, 0, st, in, flow, metric, mode, out, norm, N, C, H,
             W);
  VFI_LAUNCH((softsplat_normalize_kernel), grid_for((size_t)N * C * H * W, 256), 256, 0, st, out, norm, eps, N, C, (size_t)H * W);
  return cudaGetLastError();
}

// tiled = false: the first-version per-pixel kernels; N > 65535 (more images than grid.z holds) takes them as well
cudaError_t launch_volume81_form(bool tiled, bool dot, const float* one, const float* two, float* out, int N, int C, int H, int W,
                                 cudaStream_t st) {
  if (tiled && N <= 65535) {
    const dim3 g((unsigned)((W + 31) / 32), (unsigned)((H + 7) / 8), (unsigned)N);
    if (dot)
      VFI_LAUNCH((volume81_tile_kernel<true>), g, 256, 0, st, one, two, out, N, C, H, W);
    else
      VFI_LAUNCH((volume81_tile_kernel<false>), g, 256, 0, st, one, two, out, N, C, H, W);
    return cudaGetLastError();
  }
  const size_t total = (size_t)N * H * W;
  if (dot)
    VFI_LAUNCH((volume81_kernel<true>), grid_for(total, 128), 128, 0, st, one, two, out, N, C, H, W);
  else
    VFI_LAUNCH((volume81_kernel<false>), grid_for(total, 128), 128, 0, st, one, two, out, N, C, H, W);
  return cudaGetLastError();
}

cudaError_t launch_volume81(bool dot, const float* one, const float* two, float* out, int N, int C, int H, int W,
                            cudaStream_t st) {
  static const bool tiled = [] {  // VFI_OPS_TILED=0: the first-version per-pixel kernels (A/B runs)
    const char* e = std::getenv("VFI_OPS_TILED");
    return !(e && e[0] == '0');
  }();
  return launch_volume81_form(tiled, dot, one, two, out, N, C, H, W, st);
}

// channel-last forms: `sa` / `sb` are caller-provided scratch of N * H * W * round4(C) floats each (context-owned)
size_t ops_scratch_floats(int N, int C, int H, int W) { return (size_t)N * H * W * (size_t)((C + 3) & ~3); }

cudaError_t launch_softsplat_weighted_nhwc(const float* in, const float* flow, const float* metric, int mode, int eps, float* out,
                                           float* norm, float* sa, float* sb, int N, int C, int H, int W, cudaStream_t st) {
  if (mode < 0 || mode > 2 || eps < -1 || eps > 2 || (mode != 0 && metric == nullptr) || N > 65535) return cudaErrorInvalidValue;
  const int Cp = (C + 3) & ~3;
  const size_t hw = (size_t)H * W;
  cudaError_t e = cudaMemsetAsync(sb, 0, (size_t)N * hw * Cp * sizeof(float), st);
  if (e != cudaSuccess) return e;
  e = cudaMemsetAsync(norm, 0, (size_t)N * hw * sizeof(float), st);
  if (e != cudaSuccess) return e;
  const dim3 gt((unsigned)((hw + 31) / 32), (unsigned)((Cp + 31) / 32), (unsigned)N);
  VFI_LAUNCH((nchw_to_nhwc_kernel), gt, 256, 0, st, in, sa, C, Cp, hw);
  VFI_LAUNCH((softsplat_nhwc_kernel), grid_for((size_t)N * hw * (Cp / 4), 256), 256, 0, st, sa, flow, metric, mode, sb, norm, N, Cp, H, W);
  VFI_LAUNCH((nhwc_normalize_to_nchw_kernel), gt, 256, 0, st, sb, norm, out, C, Cp, hw, eps);
  return cudaGetLastError();
}

cudaError_t launch_volume81_warp(bool dot, const float* one, const float* two, float* out, float* sa, float* sb, int N, int C, int H,
                                 int W, cudaStream_t st) {
  if (N > 65535 || H > 65535) return cudaErrorInvalidValue;
  const int Cp = (C + 3) & ~3;
  const size_t hw = (size_t)H * W;
  const dim3 gt((unsigned)((hw + 31) / 32), (unsigned)((Cp + 31) / 32), (unsigned)N);
  VFI_LAUNCH((nchw_to_nhwc_kernel), gt, 256, 0, st, one, sa, C, Cp, hw);
  VFI_LAUNCH((nchw_to_nhwc_kernel), gt, 256, 0, st, two, sb, C, Cp, hw);
  const dim3 g((unsigned)((W + 7) / 8), (unsigned)H, (unsigned)N);
  if (dot)
    VFI_LAUNCH((volume81_warp_kernel<true>), g, 256, 0, st, sa, sb, out, C, Cp, H, W);
  else
    VFI_LAUNCH((volume81_warp_kernel<false>), g, 256, 0, st, sa, sb, out, C, Cp, H, W);
  return cudaGetLastError();
}

// py = 0: the first-version per-pixel kernel, 1 - 3: the tiled K = 51 kernel with py pixels per thread
cudaError_t launch_sepconv_form(int py, const float* in, const float* ver, const float* hor, float* out, int N, int C, int H, int W,
                                int Kv, int Kh, cudaStream_t st) {
  // the reference's only kernel size is 51 (sepconv_enhanced.py: 51-tap heads): shared-memory tiled fast path
  if (Kv == 51 && Kh == 51 && py > 0 && N <= 65535) {
    auto go = [&](auto kern, int PY) -> cudaError_t {
      const size_t smem = (size_t)(8 * PY + 50) * (32 + 50) * sizeof(float4);
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return e;
      const dim3 g((unsigned)((W + 31) / 32), (unsigned)((H + 8 * PY - 1) / (8 * PY)), (unsigned)N);
      for (int c0 = 0; c0 < C; c0 += 4) VFI_LAUNCH((kern), g, 256, smem, st, in, ver, hor, out, N, C, c0, H, W);
      return cudaGetLastError();
    };
    if (py == 1) return go(sepconv_tile_kernel<51, 1>, 1);
    if (py == 3) return go(sepconv_tile_kernel<51, 3>, 3);
    return go(sepconv_tile_kernel<51, 2>, 2);
  }
  const size_t total = (size_t)N * H * W;
  for (int c0 = 0; c0 < C; c0 += 4) {
    VFI_LAUNCH((sepconv_kernel<4>), grid_for(total, 128), 128, 0, st, in, ver, hor, out, N, C, c0, H, W, Kv, Kh);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

cudaError_t launch_sepconv(const float* in, const float* ver, const float* hor, float* out, int N, int C, int H, int W,
                           int Kv, int Kh, cudaStream_t st) {
  static const int py = [] {  // VFI_SEPCONV_PY = 0 (first-version kernel), 1, 2 (default) or 3 pixels per thread
    const char* e = std::getenv("VFI_SEPCONV_PY");
    return (e && e[0] >= '0' && e[0] <= '3') ? e[0] - '0' : 2;
  }();
  return launch_sepconv_form(py, in, ver, hor, out, N, C, H, W, Kv, Kh, st);
}

}  // namespace vfi
