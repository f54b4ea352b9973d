// Bilinear (align_corners=True) sampling of fp32 NHWC class logits, shared by the fused up-sampling
// kernels (loss.cu) and the multi-scale combine (msc.cu).
#pragma once

#include <stdint.h>

namespace b200 {

struct Interp {
  int i0, i1;
  float l0, l1;
};
// PyTorch's align_corners=True source index: src = dst * (in-1)/(out-1), fp32.
__device__ __forceinline__ Interp interp_at(int dst, float scale, int in_size) {
  const float src = scale * dst;
  Interp r;
  r.i0 = (int)src;
  if (r.i0 > in_size - 1) r.i0 = in_size - 1;
  r.i1 = r.i0 + (r.i0 < in_size - 1 ? 1 : 0);
  r.l1 = src - r.i0;
  r.l0 = 1.f - r.l1;
  return r;
}

// Interpolated logits of one full-resolution pixel (four corner pixels read as float4 vectors;
// lr_ld is a multiple of 4 and the padding classes are readable).
template <int NC>
__device__ __forceinline__ void sample_logits(const float* __restrict__ lr, int lr_ld, int h_lr,
                                              int w_lr, int n, const Interp& ih, const Interp& iw,
                                              float (&v)[NC]) {
  const float4* p00 = reinterpret_cast<const float4*>(lr + (((int64_t)n * h_lr + ih.i0) * w_lr + iw.i0) * lr_ld);
  const float4* p01 = reinterpret_cast<const float4*>(lr + (((int64_t)n * h_lr + ih.i0) * w_lr + iw.i1) * lr_ld);
  const float4* p10 = reinterpret_cast<const float4*>(lr + (((int64_t)n * h_lr + ih.i1) * w_lr + iw.i0) * lr_ld);
  const float4* p11 = reinterpret_cast<const float4*>(lr + (((int64_t)n * h_lr + ih.i1) * w_lr + iw.i1) * lr_ld);
  const float w00 = ih.l0 * iw.l0, w01 = ih.l0 * iw.l1, w10 = ih.l1 * iw.l0, w11 = ih.l1 * iw.l1;
  constexpr int NV = (NC + 3) / 4;
#pragma unroll
  for (int q = 0; q < NV; ++q) {
    const float4 a = __ldg(p00 + q), b = __ldg(p01 + q), c = __ldg(p10 + q), d = __ldg(p11 + q);
    const float r[4] = {w00 * a.x + w01 * b.x + w10 * c.x + w11 * d.x,
                        w00 * a.y + w01 * b.y + w10 * c.y + w11 * d.y,
                        w00 * a.z + w01 * b.z + w10 * c.z + w11 * d.z,
                        w00 * a.w + w01 * b.w + w10 * c.w + w11 * d.w};
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (4 * q + k < NC) v[4 * q + k] = r[k];
  }
}

// Floats per staged low-res pixel: the class count rounded up to a float4 (20 for 19 classes).  The
// staging copies exactly that many floats of each pixel, which the host check lr_ld >= round_up(NC, 4)
// keeps inside the pixel.
template <int NC>
__host__ __device__ constexpr int staged_width() { return (NC + 3) / 4 * 4; }

}  // namespace b200
