// Bilinear (align_corners=True) up-sampling of the low-resolution class logits fused with its
// consumers, so that the full-resolution logit tensor (the largest tensor of the reference step)
// is only materialised when the caller asks for it.
//   reference: F.interpolate(..., mode='bilinear', align_corners=True)  model/model_stages.py:240-242
//              CrossEntropyLoss(ignore_index=255)                       train.py:66,86-89,135,214-217
//              (a label outside [0, classes) that is not ignore_index is EXCLUDED from the loss, its
//               gradient and the pixel count -- torch raises a device-side assert for such a label; the
//               Python wrapper can check for it first, losses.VALIDATE_LABELS)
//              F.softmax(output, dim=1) feeding the discriminator       train.py:230,248,257
//              reverse_one_hot (argmax over classes)                    utils.py:98-122
//              OHEM_CrossEntroy_Loss                                    utils.py:256-271
// Low-resolution logits are fp32 NHWC with a pixel stride of `lr_ld` floats (classes padded).
// Every kernel is a template on the class count NC; b200_upsample_fwd / _bwd pick the exact instance
// for 2..32 classes, so the per-class loops have no masking and no padding class is ever read.
#include <stdint.h>

#include <atomic>

#include "ptx.cuh"
#include "status.h"
#include "b200seg.h"

namespace b200 {

constexpr int kMaxCls = 32;
constexpr int TW = 32, TH = 8;       // full-resolution tile of the backward kernels
constexpr int MAXJ = 8, MAXI = 4;    // low-resolution footprint of a tile (host-checked)

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

template <int NC>
__device__ __forceinline__ float softmax_inplace(float (&v)[NC], float* lse) {
  float m = v[0];
#pragma unroll
  for (int c = 1; c < NC; ++c) m = fmaxf(m, v[c]);
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    v[c] = __expf(v[c] - m);
    s += v[c];
  }
  const float inv = 1.f / s;
#pragma unroll
  for (int c = 0; c < NC; ++c) v[c] *= inv;
  *lse = __logf(s) + m;
  return inv;
}

// Fast-path staging for up-sampling factors >= 7 (every configuration of the reference: 64x128 ->
// 512x1024, 90x160 -> 720x1280, 128x256 -> 1024x2048).  The low-resolution pixels under a CTA's
// tile are loaded once into shared memory (coalesced float4) and every full-resolution pixel
// reads its four corners from there as broadcast LDS.128 (a 32-pixel row touches <= 6 distinct
// low-resolution columns).  Both fast kernels were instruction-issue bound in ncu, so the
// per-pixel instruction count is what these helpers are written for.
constexpr int LJ = 6;        // low-res columns under a 32-pixel wide tile: 31 * sw + 2 <= 6
constexpr int LI_ROW = 3;    // low-res rows under 8 full-resolution rows:   7 * sh + 2 <= 3
constexpr int SH_ROWS = 64;  // rows of a backward strip (8 warps x 8 rows)
constexpr int LI = 11;       // low-res rows under a strip:                 63 * sh + 2 <= 11
// Floats per staged low-res pixel: the class count rounded up to a float4 (20 for 19 classes).  The
// staging copies exactly that many floats of each pixel, which the host check lr_ld >= round_up(NC, 4)
// keeps inside the pixel.
template <int NC>
__host__ __device__ constexpr int staged_width() { return (NC + 3) / 4 * 4; }

template <int ROWS, int NC>
__device__ __forceinline__ void stage_lowres(const float* __restrict__ lr, int lr_ld, int h_lr, int w_lr, int n,
                                             int i_min, int j_min, float* s_lr) {
  constexpr int NV = staged_width<NC>() / 4;
  for (int idx = threadIdx.x; idx < ROWS * LJ * NV; idx += blockDim.x) {
    const int q = idx % NV, pix = idx / NV, jj = pix % LJ, ii = pix / LJ;
    const int i = min(i_min + ii, h_lr - 1), j = min(j_min + jj, w_lr - 1);
    reinterpret_cast<float4*>(s_lr)[pix * NV + q] =
        __ldg(reinterpret_cast<const float4*>(lr + (((int64_t)n * h_lr + i) * w_lr + j) * lr_ld) + q);
  }
}
template <int NC>
__device__ __forceinline__ void sample_smem(const float* s_lr, const Interp& ih, const Interp& iw, int i_min,
                                            int j_min, float (&v)[NC]) {
  constexpr int LP = staged_width<NC>();
  const float4* p00 = reinterpret_cast<const float4*>(s_lr + ((ih.i0 - i_min) * LJ + iw.i0 - j_min) * LP);
  const float4* p01 = reinterpret_cast<const float4*>(s_lr + ((ih.i0 - i_min) * LJ + iw.i1 - j_min) * LP);
  const float4* p10 = reinterpret_cast<const float4*>(s_lr + ((ih.i1 - i_min) * LJ + iw.i0 - j_min) * LP);
  const float4* p11 = reinterpret_cast<const float4*>(s_lr + ((ih.i1 - i_min) * LJ + iw.i1 - j_min) * LP);
  const float w00 = ih.l0 * iw.l0, w01 = ih.l0 * iw.l1, w10 = ih.l1 * iw.l0, w11 = ih.l1 * iw.l1;
  constexpr int NV = (NC + 3) / 4;
#pragma unroll
  for (int q = 0; q < NV; ++q) {
    const float4 a = p00[q], b = p01[q], c = p10[q], d = p11[q];
    const float r[4] = {w00 * a.x + w01 * b.x + w10 * c.x + w11 * d.x,
                        w00 * a.y + w01 * b.y + w10 * c.y + w11 * d.y,
                        w00 * a.z + w01 * b.z + w10 * c.z + w11 * d.z,
                        w00 * a.w + w01 * b.w + w10 * c.w + w11 * d.w};
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (4 * q + k < NC) v[4 * q + k] = r[k];
  }
}

// Zero-bordered probability layout (out_flag / grad flag == 2 in mode 2): the map is stored as
// [N][H+2][W+2][p_ld] with the image at rows/cols 1..H / 1..W and a zero border, i.e. the conv padding is
// materialised.  The dense discriminator's 4x4/stride-2/pad-1 first layer then reads column PAIRS of it as
// 128-byte, stride-1 TMA rows (model/discriminator.py); the forward writes the border zeros itself.
__device__ __forceinline__ int64_t padded_pixel(int n, int h, int w, int H, int W) {
  return ((int64_t)n * (H + 2) + (h + 1)) * (W + 2) + (w + 1);
}
__device__ __forceinline__ void zero_pixel(__nv_bfloat16* q, int p_ld) {
  for (int c = 0; c < p_ld / 8; ++c) reinterpret_cast<uint4*>(q)[c] = make_uint4(0u, 0u, 0u, 0u);
}
__device__ __forceinline__ void zero_border(__nv_bfloat16* base, int n, int h, int w, int H, int W, int p_ld) {
  const bool top = h == 0, bot = h == H - 1, left = w == 0, right = w == W - 1;
  if (!(top | bot | left | right)) return;
  if (top) zero_pixel(base + padded_pixel(n, -1, w, H, W) * p_ld, p_ld);
  if (bot) zero_pixel(base + padded_pixel(n, H, w, H, W) * p_ld, p_ld);
  if (left) zero_pixel(base + padded_pixel(n, h, -1, H, W) * p_ld, p_ld);
  if (right) zero_pixel(base + padded_pixel(n, h, W, H, W) * p_ld, p_ld);
  if (top && left) zero_pixel(base + padded_pixel(n, -1, -1, H, W) * p_ld, p_ld);
  if (top && right) zero_pixel(base + padded_pixel(n, -1, W, H, W) * p_ld, p_ld);
  if (bot && left) zero_pixel(base + padded_pixel(n, H, -1, H, W) * p_ld, p_ld);
  if (bot && right) zero_pixel(base + padded_pixel(n, H, W, H, W) * p_ld, p_ld);
}

// ------------------------------------------------------------------ forward
// mode 0: full-resolution logits, NCHW (fp32 or bf16)        -> out_full
// mode 1: cross-entropy: acc[0] += sum loss, acc[1] += #valid; optional per-pixel loss map
// mode 2: softmax probabilities, bf16 NHWC with pixel stride p_ld (padding channels zeroed)
// mode 3: argmax class map (int64 or uint8)
template <int NC>
__global__ void __launch_bounds__(256)
upsample_fwd_kernel(const float* __restrict__ lr, int lr_ld, int N, int h_lr, int w_lr, int H, int W,
                    int mode, void* __restrict__ out, int out_is_bf16_or_u8, int p_ld,
                    const int64_t* __restrict__ labels, int ignore_index, double* __restrict__ acc,
                    float* __restrict__ loss_map) {
  const float sh = H > 1 ? (float)(h_lr - 1) / (float)(H - 1) : 0.f;
  const float sw = W > 1 ? (float)(w_lr - 1) / (float)(W - 1) : 0.f;
  const int64_t total = (int64_t)N * H * W;
  float loss_sum = 0.f, valid = 0.f;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < total;
       p += (int64_t)gridDim.x * blockDim.x) {
    const int w = (int)(p % W);
    const int h = (int)((p / W) % H);
    const int n = (int)(p / ((int64_t)W * H));
    const Interp ih = interp_at(h, sh, h_lr), iw = interp_at(w, sw, w_lr);
    float v[NC];
    sample_logits<NC>(lr, lr_ld, h_lr, w_lr, n, ih, iw, v);
    if (mode == 0) {
      const int64_t plane = (int64_t)H * W;
      const int64_t o = (int64_t)n * NC * plane + (int64_t)h * W + w;
      if (out_is_bf16_or_u8) {
        __nv_bfloat16* q = static_cast<__nv_bfloat16*>(out);
#pragma unroll
        for (int c = 0; c < NC; ++c) q[o + c * plane] = __float2bfloat16(v[c]);
      } else {
        float* q = static_cast<float*>(out);
#pragma unroll
        for (int c = 0; c < NC; ++c) q[o + c * plane] = v[c];
      }
    } else if (mode == 1) {
      const int64_t lab = labels[p];
      float l = 0.f;
      if (lab != ignore_index && (unsigned long long)lab < (unsigned long long)NC) {
        float tgt = 0.f;
#pragma unroll
        for (int c = 0; c < NC; ++c) tgt = (c == lab) ? v[c] : tgt;
        float lse;
        softmax_inplace<NC>(v, &lse);
        l = fmaxf(lse - tgt, 0.f);
        loss_sum += l;
        valid += 1.f;
      }
      if (loss_map != nullptr) loss_map[p] = l;
    } else if (mode == 2) {
      float lse;
      softmax_inplace<NC>(v, &lse);
      __nv_bfloat16* q = static_cast<__nv_bfloat16*>(out) + p * p_ld;
      if (out_is_bf16_or_u8 == 2) {
        q = static_cast<__nv_bfloat16*>(out) + padded_pixel(n, h, w, H, W) * p_ld;
        zero_border(static_cast<__nv_bfloat16*>(out), n, h, w, H, W, p_ld);
      }
      uint32_t pk[kMaxCls / 2];
#pragma unroll
      for (int c = 0; c < kMaxCls / 2; ++c) {
        const float a = (2 * c < NC) ? v[2 * c < NC ? 2 * c : 0] : 0.f;
        const float b = (2 * c + 1 < NC) ? v[2 * c + 1 < NC ? 2 * c + 1 : 0] : 0.f;
        pk[c] = pack_bf16(a, b);
      }
#pragma unroll
      for (int c = 0; c < kMaxCls / 8; ++c)
        if (c < p_ld / 8)
          reinterpret_cast<uint4*>(q)[c] = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
    } else {
      int best = 0;
      float bv = v[0];
#pragma unroll
      for (int c = 1; c < NC; ++c)
        if (v[c] > bv) {
          bv = v[c];
          best = c;
        }
      if (out_is_bf16_or_u8)
        static_cast<uint8_t*>(out)[p] = (uint8_t)best;
      else
        static_cast<int64_t*>(out)[p] = best;
    }
  }
  if (mode == 1) {
    loss_sum = warp_sum(loss_sum);
    valid = warp_sum(valid);
    __shared__ float s_part[2][8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) {
      s_part[0][warp] = loss_sum;
      s_part[1][warp] = valid;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      double a = 0.0, b = 0.0;
      for (int i = 0; i < (int)(blockDim.x >> 5); ++i) {
        a += s_part[0][i];
        b += s_part[1][i];
      }
      atomicAdd(&acc[0], a);
      atomicAdd(&acc[1], b);
    }
  }
}

// Tiled variant of the forward (one CTA = one 8 x 32 pixel tile, same modes), used whenever the
// up-sampling factor is >= 7 so that a tile's low-resolution footprint fits LI_ROW x LJ.
template <int NC>
__global__ void __launch_bounds__(TH * TW)
upsample_fwd_tiled_kernel(const float* __restrict__ lr, int lr_ld, int N, int h_lr, int w_lr, int H, int W,
                          int mode, void* __restrict__ out, int out_is_bf16_or_u8, int p_ld,
                          const int64_t* __restrict__ labels, int ignore_index,
                          double* __restrict__ acc, float* __restrict__ loss_map) {
  __shared__ __align__(16) float s_lr[LI_ROW * LJ * staged_width<NC>()];
  __shared__ Interp s_iw[TW], s_ih[TH];
  __shared__ float s_part[2][TH];
  const float sh = H > 1 ? (float)(h_lr - 1) / (float)(H - 1) : 0.f;
  const float sw = W > 1 ? (float)(w_lr - 1) / (float)(W - 1) : 0.f;
  const int tiles_w = (W + TW - 1) / TW, tiles_h = (H + TH - 1) / TH;
  const int n = blockIdx.x / (tiles_w * tiles_h);
  const int t_in = blockIdx.x - n * tiles_w * tiles_h;
  const int h_base = (t_in / tiles_w) * TH, w_base = (t_in % tiles_w) * TW;
  const int tx = threadIdx.x % TW, ty = threadIdx.x / TW;
  if (threadIdx.x < TW) s_iw[threadIdx.x] = interp_at(min(w_base + threadIdx.x, W - 1), sw, w_lr);
  if (threadIdx.x >= TW && threadIdx.x < TW + TH)
    s_ih[threadIdx.x - TW] = interp_at(min(h_base + threadIdx.x - TW, H - 1), sh, h_lr);
  __syncthreads();
  stage_lowres<LI_ROW, NC>(lr, lr_ld, h_lr, w_lr, n, s_ih[0].i0, s_iw[0].i0, s_lr);
  __syncthreads();
  const int h = h_base + ty, w = w_base + tx;
  float loss = 0.f, valid = 0.f;
  if (h < H && w < W) {
    const int64_t p = ((int64_t)n * H + h) * W + w;
    float v[NC];
    sample_smem<NC>(s_lr, s_ih[ty], s_iw[tx], s_ih[0].i0, s_iw[0].i0, v);
    if (mode == 0) {
      const int64_t plane = (int64_t)H * W;
      const int64_t o = (int64_t)n * NC * plane + (int64_t)h * W + w;
      if (out_is_bf16_or_u8) {
        __nv_bfloat16* q = static_cast<__nv_bfloat16*>(out);
#pragma unroll
        for (int c = 0; c < NC; ++c) q[o + c * plane] = __float2bfloat16(v[c]);
      } else {
        float* q = static_cast<float*>(out);
#pragma unroll
        for (int c = 0; c < NC; ++c) q[o + c * plane] = v[c];
      }
    } else if (mode == 1) {
      const int64_t lab = labels[p];
      float l = 0.f;
      if (lab != ignore_index && (unsigned long long)lab < (unsigned long long)NC) {
        float tgt = 0.f;
#pragma unroll
        for (int c = 0; c < NC; ++c) tgt = (c == lab) ? v[c] : tgt;
        float lse;
        softmax_inplace<NC>(v, &lse);
        l = fmaxf(lse - tgt, 0.f);
        loss = l;
        valid = 1.f;
      }
      if (loss_map != nullptr) loss_map[p] = l;
    } else if (mode == 2) {
      float lse;
      softmax_inplace<NC>(v, &lse);
      __nv_bfloat16* q = static_cast<__nv_bfloat16*>(out) + p * p_ld;
      if (out_is_bf16_or_u8 == 2) {
        q = static_cast<__nv_bfloat16*>(out) + padded_pixel(n, h, w, H, W) * p_ld;
        zero_border(static_cast<__nv_bfloat16*>(out), n, h, w, H, W, p_ld);
      }
      uint32_t pk[kMaxCls / 2];
#pragma unroll
      for (int c = 0; c < kMaxCls / 2; ++c) {
        const float a = (2 * c < NC) ? v[2 * c < NC ? 2 * c : 0] : 0.f;
        const float b = (2 * c + 1 < NC) ? v[2 * c + 1 < NC ? 2 * c + 1 : 0] : 0.f;
        pk[c] = pack_bf16(a, b);
      }
#pragma unroll
      for (int c = 0; c < kMaxCls / 8; ++c)
        if (c < p_ld / 8)
          reinterpret_cast<uint4*>(q)[c] = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
    } else {
      int best = 0;
      float bv = v[0];
#pragma unroll
      for (int c = 1; c < NC; ++c)
        if (v[c] > bv) {
          bv = v[c];
          best = c;
        }
      if (out_is_bf16_or_u8)
        static_cast<uint8_t*>(out)[p] = (uint8_t)best;
      else
        static_cast<int64_t*>(out)[p] = best;
    }
  }
  if (mode == 1) {
    const float wl = warp_sum(loss), wv = warp_sum(valid);
    if (tx == 0) {
      s_part[0][ty] = wl;
      s_part[1][ty] = wv;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      double a = 0.0, b = 0.0;
      for (int i = 0; i < TH; ++i) {
        a += s_part[0][i];
        b += s_part[1][i];
      }
      if (b > 0.0) {
        atomicAdd(&acc[0], a);
        atomicAdd(&acc[1], b);
      }
    }
  }
}

// ------------------------------------------------------------------ backward
// d_lr[n, i, j, c] += sum over full-resolution pixels of  wh(h, i) * ww(w, j) * G[n, h, w, c]
// with G produced per pixel according to `mode`:
//   mode 0: G = d_full (NCHW fp32 / bf16)                                     (plain up-sampling)
//   mode 1: G = (softmax - onehot(label)) * pixel_weight * coef, 0 if ignored (cross-entropy)
//           coef = *coef_num / max(*coef_den, tiny)   (device scalars; den = #valid or #kept)
//           pixel_weight: nullptr (all ones) or the OHEM selection weights
//   mode 2: G = P * (dP - sum_k P_k dP_k)   with dP bf16 NHWC (stride p_ld)   (softmax)
// One CTA = one TH x TW tile; the separable transposed interpolation runs in shared memory.
// Per-pixel class strides of the backward kernels' shared buffers, odd so that the 32 lanes of a warp, one
// pixel each, write one class into 32 different banks (an even stride folds them onto NC/2..1 banks: 16 classes
// made the strip kernel 1.7x slower than 19).  19 classes keep their strides (19 and 21).
template <int NC>
__host__ __device__ constexpr int strip_class_stride() { return NC | 1; }
template <int NC>
__host__ __device__ constexpr int tile_class_stride() { return (NC + 2) | 1; }

template <int NC>
__global__ void __launch_bounds__(TH * TW)
upsample_bwd_kernel(const float* __restrict__ lr, int lr_ld, int N, int h_lr, int w_lr, int H, int W,
                    int mode, const void* __restrict__ grad_in, int grad_is_bf16, int p_ld,
                    const int64_t* __restrict__ labels, int ignore_index,
                    const float* __restrict__ pixel_weight, const float* __restrict__ coef_num,
                    const double* __restrict__ coef_den, float coef_scale, float* __restrict__ d_lr,
                    double* __restrict__ loss_acc) {
  __shared__ float s_g[TH][TW][tile_class_stride<NC>()];
  __shared__ float s_loss[2][TH];
  __shared__ float s_a[TH][MAXJ][NC + 1];
  __shared__ Interp s_iw[TW], s_ih[TH];
  const float sh = H > 1 ? (float)(h_lr - 1) / (float)(H - 1) : 0.f;
  const float sw = W > 1 ? (float)(w_lr - 1) / (float)(W - 1) : 0.f;
  const int tiles_w = (W + TW - 1) / TW, tiles_h = (H + TH - 1) / TH;
  const int n = blockIdx.x / (tiles_w * tiles_h);
  const int t_in = blockIdx.x - n * tiles_w * tiles_h;
  const int h_base = (t_in / tiles_w) * TH, w_base = (t_in % tiles_w) * TW;
  const int tx = threadIdx.x % TW, ty = threadIdx.x / TW;
  if (threadIdx.x < TW) s_iw[threadIdx.x] = interp_at(min(w_base + threadIdx.x, W - 1), sw, w_lr);
  if (threadIdx.x >= TW && threadIdx.x < TW + TH)
    s_ih[threadIdx.x - TW] = interp_at(min(h_base + threadIdx.x - TW, H - 1), sh, h_lr);
  __syncthreads();
  const int h = h_base + ty, w = w_base + tx;
  float g[NC];
  float my_loss = 0.f, my_valid = 0.f;
#pragma unroll
  for (int c = 0; c < NC; ++c) g[c] = 0.f;
  if (h < H && w < W) {
    const int64_t p = ((int64_t)n * H + h) * W + w;
    if (mode == 0) {
      const int64_t plane = (int64_t)H * W;
      const int64_t o = (int64_t)n * NC * plane + (int64_t)h * W + w;
      if (grad_is_bf16) {
        const __nv_bfloat16* q = static_cast<const __nv_bfloat16*>(grad_in);
#pragma unroll
        for (int c = 0; c < NC; ++c) g[c] = __bfloat162float(q[o + c * plane]);
      } else {
        const float* q = static_cast<const float*>(grad_in);
#pragma unroll
        for (int c = 0; c < NC; ++c) g[c] = q[o + c * plane];
      }
    } else {
      float v[NC];
      sample_logits<NC>(lr, lr_ld, h_lr, w_lr, n, s_ih[ty], s_iw[tx], v);
      float tgt = 0.f;
      const int64_t lab_ce = (mode == 1) ? labels[p] : -1;
#pragma unroll
      for (int c = 0; c < NC; ++c) tgt = (c == lab_ce) ? v[c] : tgt;
      float lse;
      softmax_inplace<NC>(v, &lse);
      if (mode == 1) {
        const int64_t lab = lab_ce;
        if (lab != ignore_index && (unsigned long long)lab < (unsigned long long)NC) {
          my_loss = fmaxf(lse - tgt, 0.f);
          my_valid = 1.f;
          float cf = coef_scale * (coef_num != nullptr ? *coef_num : 1.f);
          if (coef_den != nullptr) cf /= (float)fmax(*coef_den, 1e-30);
          if (pixel_weight != nullptr) cf *= pixel_weight[p];
#pragma unroll
          for (int c = 0; c < NC; ++c) g[c] = (v[c] - (c == lab ? 1.f : 0.f)) * cf;
        }
      } else {
        const __nv_bfloat16* q = static_cast<const __nv_bfloat16*>(grad_in) +
                                 (grad_is_bf16 == 2 ? padded_pixel(n, h, w, H, W) : p) * p_ld;
        float dp[NC];
        float dot = 0.f;
#pragma unroll
        for (int c = 0; c < NC; ++c) {
          dp[c] = __bfloat162float(q[c]);
          dot += dp[c] * v[c];
        }
        const float cf = coef_scale * (coef_num != nullptr ? *coef_num : 1.f);
#pragma unroll
        for (int c = 0; c < NC; ++c) g[c] = v[c] * (dp[c] - dot) * cf;
      }
    }
  }
#pragma unroll
  for (int c = 0; c < NC; ++c) s_g[ty][tx][c] = g[c];
  if (loss_acc != nullptr) {  // fused forward: this tile's loss sum and valid-pixel count
    const float wl = warp_sum(my_loss), wv = warp_sum(my_valid);
    if (tx == 0) {
      s_loss[0][ty] = wl;
      s_loss[1][ty] = wv;
    }
  }
  __syncthreads();
  if (loss_acc != nullptr && threadIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (int i = 0; i < TH; ++i) {
      a += s_loss[0][i];
      b += s_loss[1][i];
    }
    if (b > 0.0) {
      atomicAdd(&loss_acc[0], a);
      atomicAdd(&loss_acc[1], b);
    }
  }
  // Separable transposed interpolation.  Source indices are non-decreasing along a row / column,
  // so each (row, class) thread streams over the 32 columns keeping two running sums (for the
  // current low-resolution column and the next one) and flushes when the source index advances.
  const int j_min = s_iw[0].i0;
  for (int t = threadIdx.x; t < TH * NC; t += TH * TW) {
    const int r = t / NC, c = t - r * NC;
    float acc0 = 0.f, acc1 = 0.f;
    int j_cur = j_min;
    for (int x = 0; x < TW; ++x) {
      const Interp iw = s_iw[x];
      while (iw.i0 != j_cur) {
        s_a[r][j_cur - j_min][c] = acc0;
        acc0 = acc1;
        acc1 = 0.f;
        ++j_cur;
      }
      const float gv = s_g[r][x][c];
      acc0 += iw.l0 * gv;
      if (iw.i1 != iw.i0) acc1 += iw.l1 * gv;
      else acc0 += iw.l1 * gv;
    }
    s_a[r][j_cur - j_min][c] = acc0;
    if (j_cur + 1 - j_min < MAXJ) s_a[r][j_cur + 1 - j_min][c] = acc1;
    for (int jj = j_cur + 2 - j_min; jj < MAXJ; ++jj) s_a[r][jj][c] = 0.f;
  }
  __syncthreads();
  const int i_min = s_ih[0].i0;
  for (int t = threadIdx.x; t < MAXJ * NC; t += TH * TW) {
    const int jj = t / NC, c = t - jj * NC;
    const int j = j_min + jj;
    if (j >= w_lr) continue;
    float acc0 = 0.f, acc1 = 0.f;
    int i_cur = i_min;
    float* dst = d_lr + ((int64_t)n * h_lr * w_lr + j) * lr_ld + c;
    for (int y = 0; y < TH; ++y) {
      const Interp ih = s_ih[y];
      while (ih.i0 != i_cur) {
        if (acc0 != 0.f) atomicAdd(dst + (int64_t)i_cur * w_lr * lr_ld, acc0);
        acc0 = acc1;
        acc1 = 0.f;
        ++i_cur;
      }
      const float av = s_a[y][jj][c];
      acc0 += ih.l0 * av;
      if (ih.i1 != ih.i0) acc1 += ih.l1 * av;
      else acc0 += ih.l1 * av;
    }
    if (acc0 != 0.f) atomicAdd(dst + (int64_t)i_cur * w_lr * lr_ld, acc0);
    if (acc1 != 0.f && i_cur + 1 < h_lr) atomicAdd(dst + (int64_t)(i_cur + 1) * w_lr * lr_ld, acc1);
  }
}

// Fast backward (up-sampling factor >= 7): one CTA = a strip of SH_ROWS x TW pixels; warp w owns
// rows 8w .. 8w+7 and a lane owns one column.  A thread walks its 8 pixels and folds their class
// gradients, weighted by the vertical interpolation weights, into <= 3 low-resolution rows held in
// registers (the transposed interpolation along h costs 2 FMAs per class and pixel, no shared
// memory).  The per-column partials are added into a CTA-wide shared buffer, reduced along w with
// a precomputed weight table, and one atomicAdd per touched low-resolution value leaves the CTA:
// ~1/6 of the global atomics and ~1/5 of the instructions of the generic tile kernel.
// The staged pixels and the vertical partials live in dynamic shared memory (strip_smem_bytes: 31 KB at
// 19 classes, 54 KB at 32, above the 48 KB of static shared memory a kernel may declare).
template <int NC>
constexpr int strip_smem_bytes() {
  return (LI * LJ * staged_width<NC>() + LI * TW * strip_class_stride<NC>()) * (int)sizeof(float);
}
template <int NC>
__global__ void __launch_bounds__(256)
upsample_bwd_strip_kernel(const float* __restrict__ lr, int lr_ld, int N, int h_lr, int w_lr, int H, int W,
                          int mode, const void* __restrict__ grad_in, int grad_is_bf16, int p_ld,
                          const int64_t* __restrict__ labels, int ignore_index,
                          const float* __restrict__ pixel_weight, const float* __restrict__ coef_num,
                          const double* __restrict__ coef_den, float coef_scale, float* __restrict__ d_lr,
                          double* __restrict__ loss_acc) {
  extern __shared__ __align__(16) float s_dyn[];
  float* s_lr = s_dyn;                                   // staged low-res pixels
  constexpr int SV = strip_class_stride<NC>();
  float (*s_v)[TW][SV] = reinterpret_cast<float (*)[TW][SV]>(s_dyn + LI * LJ * staged_width<NC>());
                                                         // vertical partials: [low-res row][column][class]
  __shared__ float s_wx[LJ][TW];      // weight of column x on low-res column jj
  __shared__ int s_xlo[LJ], s_xhi[LJ];
  __shared__ Interp s_iw[TW], s_ih[SH_ROWS];
  __shared__ float s_loss[2][8];
  const float sh = H > 1 ? (float)(h_lr - 1) / (float)(H - 1) : 0.f;
  const float sw = W > 1 ? (float)(w_lr - 1) / (float)(W - 1) : 0.f;
  const int tiles_w = (W + TW - 1) / TW, tiles_h = (H + SH_ROWS - 1) / SH_ROWS;
  const int n = blockIdx.x / (tiles_w * tiles_h);
  const int t_in = blockIdx.x - n * tiles_w * tiles_h;
  const int h_base = (t_in / tiles_w) * SH_ROWS, w_base = (t_in % tiles_w) * TW;
  const int tx = threadIdx.x % TW, wp = threadIdx.x / TW;
  if (threadIdx.x < TW) s_iw[threadIdx.x] = interp_at(min(w_base + threadIdx.x, W - 1), sw, w_lr);
  if (threadIdx.x >= TW && threadIdx.x < TW + SH_ROWS)
    s_ih[threadIdx.x - TW] = interp_at(min(h_base + threadIdx.x - TW, H - 1), sh, h_lr);
  for (int i = threadIdx.x; i < LI * TW * SV; i += 256) (&s_v[0][0][0])[i] = 0.f;
  __syncthreads();
  const int i_min = s_ih[0].i0, j_min = s_iw[0].i0;
  if (mode != 0) stage_lowres<LI, NC>(lr, lr_ld, h_lr, w_lr, n, i_min, j_min, s_lr);
  if (threadIdx.x < LJ * TW) {  // weight table of the transposed interpolation along w
    const int jj = threadIdx.x / TW, x = threadIdx.x % TW;
    const Interp iw = s_iw[x];
    float wgt = 0.f;
    if (w_base + x < W) wgt = (iw.i0 - j_min == jj ? iw.l0 : 0.f) + (iw.i1 - j_min == jj ? iw.l1 : 0.f);
    s_wx[jj][x] = wgt;
    const unsigned nz = __ballot_sync(0xffffffffu, wgt != 0.f);
    if (x == 0) {
      s_xlo[jj] = nz ? __ffs(nz) - 1 : 0;
      s_xhi[jj] = nz ? 32 - __clz(nz) : 0;
    }
  }
  __syncthreads();

  const Interp iw = s_iw[tx];
  const int w = w_base + tx;
  const int i_w = s_ih[wp * 8].i0;  // first low-resolution row this warp touches
  float acc0[NC], acc1[NC], acc2[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) acc0[c] = acc1[c] = acc2[c] = 0.f;
  float my_loss = 0.f, my_valid = 0.f;
  float cf0 = coef_scale * (coef_num != nullptr ? *coef_num : 1.f);
  if (coef_den != nullptr) cf0 /= (float)fmax(*coef_den, 1e-30);
  const int64_t plane = (int64_t)H * W;
#pragma unroll 1
  for (int r = 0; r < 8; ++r) {
    const int h = h_base + wp * 8 + r;
    if (h >= H) break;
    const Interp ih = s_ih[wp * 8 + r];
    float g[NC];
    bool live = w < W;
    if (live) {
      const int64_t p = ((int64_t)n * H + h) * W + w;
      if (mode == 0) {
        const int64_t o = (int64_t)n * NC * plane + (int64_t)h * W + w;
        if (grad_is_bf16) {
          const __nv_bfloat16* q = static_cast<const __nv_bfloat16*>(grad_in);
#pragma unroll
          for (int c = 0; c < NC; ++c) g[c] = __bfloat162float(q[o + c * plane]);
        } else {
          const float* q = static_cast<const float*>(grad_in);
#pragma unroll
          for (int c = 0; c < NC; ++c) g[c] = q[o + c * plane];
        }
      } else {
        sample_smem<NC>(s_lr, ih, iw, i_min, j_min, g);
        if (mode == 1) {
          const int64_t lab = labels[p];
          if (lab != ignore_index && (unsigned long long)lab < (unsigned long long)NC) {
            float tgt = 0.f;
#pragma unroll
            for (int c = 0; c < NC; ++c) tgt = (c == lab) ? g[c] : tgt;
            float lse;
            softmax_inplace<NC>(g, &lse);
            my_loss += fmaxf(lse - tgt, 0.f);
            my_valid += 1.f;
            const float cf = pixel_weight != nullptr ? cf0 * pixel_weight[p] : cf0;
#pragma unroll
            for (int c = 0; c < NC; ++c) g[c] = (g[c] - (c == lab ? 1.f : 0.f)) * cf;
          } else {
            live = false;
          }
        } else {
          float lse;
          softmax_inplace<NC>(g, &lse);
          float dp[NC];
          const __nv_bfloat16* q = static_cast<const __nv_bfloat16*>(grad_in) +
                                   (grad_is_bf16 == 2 ? padded_pixel(n, h, w, H, W) : p) * p_ld;
          if ((p_ld & 7) == 0) {  // 16-byte aligned pixel rows: one vector load per 8 classes
            uint32_t raw[(NC + 7) / 8 * 4];
#pragma unroll
            for (int k = 0; k < (NC + 7) / 8; ++k) {
              const uint4 u = __ldg(reinterpret_cast<const uint4*>(q) + k);
              raw[4 * k] = u.x; raw[4 * k + 1] = u.y; raw[4 * k + 2] = u.z; raw[4 * k + 3] = u.w;
            }
#pragma unroll
            for (int c = 0; c < NC; ++c) {
              const float2 f = unpack_bf16(raw[c >> 1]);
              dp[c] = (c & 1) ? f.y : f.x;
            }
          } else {
#pragma unroll
            for (int c = 0; c < NC; ++c) dp[c] = __bfloat162float(q[c]);
          }
          float dot = 0.f;
#pragma unroll
          for (int c = 0; c < NC; ++c) dot += dp[c] * g[c];
#pragma unroll
          for (int c = 0; c < NC; ++c) g[c] = g[c] * (dp[c] - dot) * cf0;
        }
      }
    }
    if (live) {
      const bool same = ih.i1 == ih.i0;  // clamped at the bottom edge
      const float le0 = same ? ih.l0 + ih.l1 : ih.l0, le1 = same ? 0.f : ih.l1;
      if (ih.i0 == i_w) {                // warp-uniform: the whole warp is on one row
#pragma unroll
        for (int c = 0; c < NC; ++c) {
          acc0[c] += le0 * g[c];
          acc1[c] += le1 * g[c];
        }
      } else {
#pragma unroll
        for (int c = 0; c < NC; ++c) {
          acc1[c] += le0 * g[c];
          acc2[c] += le1 * g[c];
        }
      }
    }
  }
  {
    const int row = i_w - i_min;
#pragma unroll
    for (int c = 0; c < NC; ++c) atomicAdd(&s_v[row][tx][c], acc0[c]);
    if (row + 1 < LI) {
#pragma unroll
      for (int c = 0; c < NC; ++c) atomicAdd(&s_v[row + 1][tx][c], acc1[c]);
    }
    if (row + 2 < LI) {
#pragma unroll
      for (int c = 0; c < NC; ++c) atomicAdd(&s_v[row + 2][tx][c], acc2[c]);
    }
  }
  if (loss_acc != nullptr) {
    const float wl = warp_sum(my_loss), wv = warp_sum(my_valid);
    if (tx == 0) {
      s_loss[0][wp] = wl;
      s_loss[1][wp] = wv;
    }
  }
  __syncthreads();
  if (loss_acc != nullptr && threadIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (int i = 0; i < 8; ++i) {
      a += s_loss[0][i];
      b += s_loss[1][i];
    }
    if (b > 0.0) {
      atomicAdd(&loss_acc[0], a);
      atomicAdd(&loss_acc[1], b);
    }
  }
  // transposed interpolation along w + the CTA's contribution to d_lr
  for (int t = threadIdx.x; t < LI * LJ * NC; t += 256) {
    const int c = t % NC, jj = (t / NC) % LJ, ii = t / (NC * LJ);
    const int i = i_min + ii, j = j_min + jj;
    if (i >= h_lr || j >= w_lr) continue;
    const int x0 = s_xlo[jj], x1 = s_xhi[jj];
    float sum = 0.f;
    for (int x = x0; x < x1; ++x) sum += s_wx[jj][x] * s_v[ii][x][c];
    if (sum != 0.f) atomicAdd(d_lr + (((int64_t)n * h_lr + i) * w_lr + j) * lr_ld + c, sum);
  }
}

// ----------------------------------------------------- radix select (OHEM)
// k-th largest of non-negative fp32 values: for x >= 0 the IEEE bit pattern orders like the value,
// so four 8-bit passes over the bit patterns find it without sorting.
// state[0] = prefix bits found so far, state[1] = remaining rank (0-based, descending)
__global__ void __launch_bounds__(256)
radix_hist_kernel(const float* __restrict__ x, int64_t count, int pass, const uint32_t* __restrict__ state,
                  uint32_t* __restrict__ hist /* [256] */) {
  __shared__ uint32_t s_h[256];
  s_h[threadIdx.x] = 0;
  __syncthreads();
  const int shift = 24 - 8 * pass;
  const uint32_t prefix = state[0];
  const uint32_t mask = pass == 0 ? 0u : (0xFFFFFFFFu << (shift + 8));
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count;
       i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t u = __float_as_uint(x[i]);
    if ((u & mask) == (prefix & mask)) atomicAdd(&s_h[(u >> shift) & 0xFF], 1u);
  }
  __syncthreads();
  if (s_h[threadIdx.x]) atomicAdd(&hist[threadIdx.x], s_h[threadIdx.x]);
}
__global__ void radix_init_kernel(uint32_t* __restrict__ state, uint32_t* __restrict__ hist, uint32_t rank) {
  if (threadIdx.x == 0) {
    state[0] = 0u;
    state[1] = rank;
  }
  hist[threadIdx.x] = 0u;
}
__global__ void radix_pick_kernel(uint32_t* __restrict__ state, uint32_t* __restrict__ hist, int pass) {
  if (threadIdx.x != 0) return;
  const int shift = 24 - 8 * pass;
  uint32_t rank = state[1];
  int d = 255;
  for (; d > 0; --d) {
    const uint32_t c = hist[d];
    if (rank < c) break;
    rank -= c;
  }
  state[0] |= ((uint32_t)d) << shift;
  state[1] = rank;
  for (int i = 0; i < 256; ++i) hist[i] = 0;
}

// OHEM reduction (utils.py:263-271).  t = sorted_desc[keep_num] (bit pattern in state[0]).
//   t > threshold : mean of the losses > threshold
//   else          : mean of the keep_num largest = (sum_{x>v} x + (keep - cnt_{x>v}) * v) / keep
//                   with v = t  (every element above t is among the top keep_num)
// pass 1 accumulates the sums, pass 2 (ohem_finalize) writes the loss and the per-pixel weights'
// parameters: out[0] = loss, out[1] = cut value, out[2] = weight above the cut, out[3] = weight at the cut.
__global__ void __launch_bounds__(256)
ohem_sums_kernel(const float* __restrict__ x, int64_t count, const uint32_t* __restrict__ state,
                 float threshold, double* __restrict__ sums /* [5] */) {
  const float t = __uint_as_float(state[0]);
  double s_thr = 0.0, n_thr = 0.0, s_t = 0.0, n_t = 0.0, n_eq = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count;
       i += (int64_t)gridDim.x * blockDim.x) {
    const float v = x[i];
    if (v > threshold) { s_thr += v; n_thr += 1.0; }
    if (v > t) { s_t += v; n_t += 1.0; }
    if (v == t) n_eq += 1.0;
  }
  double vals[5] = {s_thr, n_thr, s_t, n_t, n_eq};
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    double v = vals[k];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v != 0.0) atomicAdd(&sums[k], v);
  }
}
__global__ void ohem_finalize_kernel(const uint32_t* __restrict__ state, const double* __restrict__ sums,
                                     float threshold, int64_t keep_num, float* __restrict__ out) {
  if (threadIdx.x != 0) return;
  const float t = __uint_as_float(state[0]);
  if (t > threshold) {
    out[0] = (float)(sums[0] / sums[1]);
    out[1] = threshold;
    out[2] = (float)(1.0 / sums[1]);
    out[3] = 0.f;
  } else {
    const double rest = (double)keep_num - sums[3];
    out[0] = (float)((sums[2] + rest * (double)t) / (double)keep_num);
    out[1] = t;
    out[2] = (float)(1.0 / (double)keep_num);
    out[3] = sums[4] > 0.0 ? (float)(rest / (sums[4] * (double)keep_num)) : 0.f;
  }
}
// per-pixel gradient weight of the OHEM mean: w = out[2] above the cut, out[3] at the cut, else 0
__global__ void __launch_bounds__(256)
ohem_weights_kernel(const float* __restrict__ x, int64_t count, const float* __restrict__ sel,
                    float* __restrict__ wout) {
  const float cut = sel[1], wa = sel[2], we = sel[3];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count;
       i += (int64_t)gridDim.x * blockDim.x) {
    const float v = x[i];
    wout[i] = v > cut ? wa : (v == cut ? we : 0.f);
  }
}

// mean BCE-with-logits against a constant target (0 or 1): loss = mean(softplus(x) - t*x)
//   forward: out[0] += sum / count ; backward: dx = (sigmoid(x) - t) * (*gscale) * gmul / count
__global__ void __launch_bounds__(256)
bce_const_fwd_kernel(const float* __restrict__ x, int count, float target, float* __restrict__ out) {
  float acc = 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    const float v = x[i];
    acc += fmaxf(v, 0.f) - v * target + log1pf(__expf(-fabsf(v)));
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) atomicAdd(out, acc / count);
}
__global__ void __launch_bounds__(256)
bce_const_bwd_kernel(const float* __restrict__ x, int count, float target,
                     const float* __restrict__ gscale, float gmul, float* __restrict__ dx) {
  const float gs = (gscale != nullptr ? *gscale : 1.f) * gmul / count;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    const float v = x[i];
    dx[i] = (1.f / (1.f + __expf(-v)) - target) * gs;
  }
}

// y = x * (*num) * mul / (*den)      (applies the upstream gradient and 1/#valid to a fused CE gradient)
__global__ void __launch_bounds__(256)
scale_f32_kernel(const float* __restrict__ x, int64_t count4, const float* __restrict__ num,
                 const double* __restrict__ den, float mul, float* __restrict__ y) {
  float cf = mul * (num != nullptr ? *num : 1.f);
  if (den != nullptr) cf /= (float)fmax(*den, 1e-30);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count4;
       i += (int64_t)gridDim.x * blockDim.x) {
    float4 v = reinterpret_cast<const float4*>(x)[i];
    v.x *= cf; v.y *= cf; v.z *= cf; v.w *= cf;
    reinterpret_cast<float4*>(y)[i] = v;
  }
}

static int grid1d(int64_t total, int cap) {
  int64_t b = (total + 255) / 256;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

static int round_up4(int v) { return (v + 3) / 4 * 4; }

// Every class count with a compiled instance (kMaxCls = 32 is the widest padded logit map).
#define B200_FOR_EACH_CLASS_COUNT(X)                                                                       \
  X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15) X(16) X(17) X(18) X(19)      \
  X(20) X(21) X(22) X(23) X(24) X(25) X(26) X(27) X(28) X(29) X(30) X(31) X(32)

struct FwdArgs {
  const float* lr; int lr_ld, N, h_lr, w_lr, H, W, mode; void* out; int out_flag, p_ld;
  const int64_t* labels; int ignore_index; double* acc; float* loss_map;
};
struct BwdArgs {
  const float* lr; int lr_ld, N, h_lr, w_lr, H, W, mode; const void* grad_in; int grad_is_bf16, p_ld;
  const int64_t* labels; int ignore_index; const float* pixel_weight; const float* coef_num;
  const double* coef_den; float coef_scale; float* d_lr; double* loss_acc;
};

template <int NC>
static int launch_fwd(const FwdArgs& a, cudaStream_t stream) {
  const int64_t total = (int64_t)a.N * a.H * a.W;
  const float sh = a.H > 1 ? (float)(a.h_lr - 1) / (float)(a.H - 1) : 0.f;
  const float sw = a.W > 1 ? (float)(a.w_lr - 1) / (float)(a.W - 1) : 0.f;
  if (sw * (TW - 1) + 2.f <= (float)LJ && sh * (TH - 1) + 2.f <= (float)LI_ROW) {
    const int tiles = ((a.W + TW - 1) / TW) * ((a.H + TH - 1) / TH) * a.N;
    upsample_fwd_tiled_kernel<NC><<<tiles, TH * TW, 0, stream>>>(
        a.lr, a.lr_ld, a.N, a.h_lr, a.w_lr, a.H, a.W, a.mode, a.out, a.out_flag, a.p_ld, a.labels, a.ignore_index,
        a.acc, a.loss_map);
    return check_launch("upsample_fwd(tiled)");
  }
  upsample_fwd_kernel<NC><<<grid1d(total, 148 * 16), 256, 0, stream>>>(
      a.lr, a.lr_ld, a.N, a.h_lr, a.w_lr, a.H, a.W, a.mode, a.out, a.out_flag, a.p_ld, a.labels, a.ignore_index,
      a.acc, a.loss_map);
  return check_launch("upsample_fwd");
}

// The strip kernel's dynamic shared memory exceeds the default 48 KB limit from 28 classes on; the
// opt-in is a per-device function attribute, set once per instance and device.
template <int NC>
static cudaError_t strip_smem_optin() {
  static std::atomic<unsigned long long> done{0};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const unsigned long long bit = 1ull << (dev & 63);
  if (done.load(std::memory_order_acquire) & bit) return cudaSuccess;
  e = cudaFuncSetAttribute(upsample_bwd_strip_kernel<NC>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           strip_smem_bytes<NC>());
  if (e == cudaSuccess) done.fetch_or(bit, std::memory_order_release);
  return e;
}

template <int NC>
static int launch_bwd(const BwdArgs& a, bool strip, cudaStream_t stream) {
  if (strip) {
    const cudaError_t e = strip_smem_optin<NC>();
    if (e != cudaSuccess) return set_error(B200_ECUDA, "upsample_bwd(strip) shared memory: %s", cudaGetErrorString(e));
    const int strips = ((a.W + TW - 1) / TW) * ((a.H + SH_ROWS - 1) / SH_ROWS) * a.N;
    upsample_bwd_strip_kernel<NC><<<strips, 256, strip_smem_bytes<NC>(), stream>>>(
        a.lr, a.lr_ld, a.N, a.h_lr, a.w_lr, a.H, a.W, a.mode, a.grad_in, a.grad_is_bf16, a.p_ld, a.labels,
        a.ignore_index, a.pixel_weight, a.coef_num, a.coef_den, a.coef_scale, a.d_lr, a.loss_acc);
    return check_launch("upsample_bwd(strip)");
  }
  const int tiles = ((a.W + TW - 1) / TW) * ((a.H + TH - 1) / TH) * a.N;
  upsample_bwd_kernel<NC><<<tiles, TH * TW, 0, stream>>>(
      a.lr, a.lr_ld, a.N, a.h_lr, a.w_lr, a.H, a.W, a.mode, a.grad_in, a.grad_is_bf16, a.p_ld, a.labels,
      a.ignore_index, a.pixel_weight, a.coef_num, a.coef_den, a.coef_scale, a.d_lr, a.loss_acc);
  return check_launch("upsample_bwd");
}

}  // namespace b200

using namespace b200;

extern "C" {

int b200_upsample_fwd(const float* lr, int lr_ld, int N, int h_lr, int w_lr, int H, int W,
                      int n_classes, int mode, void* out, int out_flag, int p_ld,
                      const int64_t* labels, int ignore_index, double* acc, float* loss_map,
                      cudaStream_t stream) {
  if (n_classes < 2 || n_classes > kMaxCls)
    return set_error(B200_EINVAL, "upsample_fwd: %d classes unsupported (2..%d are compiled)", n_classes, kMaxCls);
  if (lr_ld % 4 || lr_ld < round_up4(n_classes))
    return set_error(B200_EINVAL, "upsample_fwd: logits pixel stride %d must be a multiple of 4, >= %d for %d classes",
                     lr_ld, round_up4(n_classes), n_classes);
  if (mode == 2 && (p_ld % 8 || p_ld > kMaxCls || p_ld < n_classes))
    return set_error(B200_EINVAL, "upsample_fwd: probability stride %d unsupported", p_ld);
  const FwdArgs a{lr, lr_ld, N, h_lr, w_lr, H, W, mode, out, out_flag, p_ld, labels, ignore_index, acc, loss_map};
  switch (n_classes) {
#define B200_FWD_CASE(nc) case nc: return launch_fwd<nc>(a, stream);
    B200_FOR_EACH_CLASS_COUNT(B200_FWD_CASE)
#undef B200_FWD_CASE
  }
  return set_error(B200_EINVAL, "upsample_fwd: %d classes unsupported", n_classes);
}

int b200_upsample_bwd(const float* lr, int lr_ld, int N, int h_lr, int w_lr, int H, int W,
                      int n_classes, int mode, const void* grad_in, int grad_is_bf16, int p_ld,
                      const int64_t* labels, int ignore_index, const float* pixel_weight,
                      const float* coef_num, const double* coef_den, float coef_scale, float* d_lr,
                      double* loss_acc, cudaStream_t stream) {
  if (n_classes < 2 || n_classes > kMaxCls)
    return set_error(B200_EINVAL, "upsample_bwd: %d classes unsupported (2..%d are compiled)", n_classes, kMaxCls);
  if (lr_ld % 4 || lr_ld < round_up4(n_classes))
    return set_error(B200_EINVAL, "upsample_bwd: logits pixel stride %d must be a multiple of 4, >= %d for %d classes",
                     lr_ld, round_up4(n_classes), n_classes);
  if (mode == 2 && p_ld < n_classes)
    return set_error(B200_EINVAL, "upsample_bwd: probability-gradient stride %d < %d classes", p_ld, n_classes);
  const float sh = H > 1 ? (float)(h_lr - 1) / (float)(H - 1) : 0.f;
  const float sw = W > 1 ? (float)(w_lr - 1) / (float)(W - 1) : 0.f;
  const bool strip = sw * (TW - 1) + 2.f <= (float)LJ && sh * 7.f + 2.f <= (float)LI_ROW && sh * (SH_ROWS - 1) + 2.f <= (float)LI;
  if (!strip && (sw * (TW - 1) + 2.f > (float)MAXJ || sh * (TH - 1) + 2.f > (float)MAXI))
    return set_error(B200_EINVAL, "upsample_bwd: scale %dx%d -> %dx%d is below the supported up-sampling factor (>= 5.2 along w, >= 3.5 along h)", h_lr, w_lr, H, W);
  const BwdArgs a{lr, lr_ld, N, h_lr, w_lr, H, W, mode, grad_in, grad_is_bf16, p_ld, labels, ignore_index,
                  pixel_weight, coef_num, coef_den, coef_scale, d_lr, loss_acc};
  switch (n_classes) {
#define B200_BWD_CASE(nc) case nc: return launch_bwd<nc>(a, strip, stream);
    B200_FOR_EACH_CLASS_COUNT(B200_BWD_CASE)
#undef B200_BWD_CASE
  }
  return set_error(B200_EINVAL, "upsample_bwd: %d classes unsupported", n_classes);
}

// k-th largest (0-based rank in descending order) of `count` non-negative floats.
// state: uint32[2] scratch, hist: uint32[256] scratch (zeroed here).  Result bits in state[0].
int b200_radix_select_desc(const float* x, int64_t count, int64_t rank, uint32_t* state,
                           uint32_t* hist, cudaStream_t stream) {
  if (rank < 0 || rank >= count) return set_error(B200_EINVAL, "radix_select: rank %lld out of range", (long long)rank);
  if (count >= (1ll << 32)) return set_error(B200_EINVAL, "radix_select: count too large");
  radix_init_kernel<<<1, 256, 0, stream>>>(state, hist, (uint32_t)rank);
  for (int pass = 0; pass < 4; ++pass) {
    radix_hist_kernel<<<grid1d(count, 148 * 8), 256, 0, stream>>>(x, count, pass, state, hist);
    radix_pick_kernel<<<1, 32, 0, stream>>>(state, hist, pass);
  }
  return check_launch("radix_select");
}

// sums: double[5] scratch (zeroed here); out: float[4] = loss, cut, weight above, weight at cut
int b200_ohem_reduce(const float* x, int64_t count, const uint32_t* state, float threshold,
                     int64_t keep_num, double* sums, float* out, cudaStream_t stream) {
  cudaError_t e = cudaMemsetAsync(sums, 0, 5 * sizeof(double), stream);
  if (e != cudaSuccess) return set_error(B200_ECUDA, "ohem_reduce setup: %s", cudaGetErrorString(e));
  ohem_sums_kernel<<<grid1d(count, 148 * 8), 256, 0, stream>>>(x, count, state, threshold, sums);
  ohem_finalize_kernel<<<1, 32, 0, stream>>>(state, sums, threshold, keep_num, out);
  return check_launch("ohem_reduce");
}

int b200_ohem_weights(const float* x, int64_t count, const float* sel, float* wout, cudaStream_t stream) {
  ohem_weights_kernel<<<grid1d(count, 148 * 8), 256, 0, stream>>>(x, count, sel, wout);
  return check_launch("ohem_weights");
}

int b200_scale_f32(const float* x, int64_t count, const float* num, const double* den, float mul,
                   float* y, cudaStream_t stream) {
  if (count % 4) return set_error(B200_EINVAL, "scale_f32: count must be a multiple of 4");
  scale_f32_kernel<<<grid1d(count / 4, 148 * 8), 256, 0, stream>>>(x, count / 4, num, den, mul, y);
  return check_launch("scale_f32");
}

int b200_bce_const_fwd(const float* x, int count, float target, float* out, cudaStream_t stream) {
  bce_const_fwd_kernel<<<grid1d(count, 64), 256, 0, stream>>>(x, count, target, out);
  return check_launch("bce_const_fwd");
}

int b200_bce_const_bwd(const float* x, int count, float target, const float* gscale, float gmul,
                       float* dx, cudaStream_t stream) {
  bce_const_bwd_kernel<<<grid1d(count, 64), 256, 0, stream>>>(x, count, target, gscale, gmul, dx);
  return check_launch("bce_const_bwd");
}

}  // extern "C"
