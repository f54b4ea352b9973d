// Multi-scale + flip evaluation (BiSeNet's MscEval(scales, flip)):
//   image_rescale_kernel   F.interpolate(x, (h, w), mode='bilinear', align_corners=True) of the fp32 NCHW
//                          images, optionally followed by their horizontal mirrors (torch.flip(x, dims=[3]))
//                          in the same output, so that one forward runs both halves;
//   msc_argmax_kernel<NC>  for every full-resolution pixel: bilinear (align_corners=True) sample of every
//                          low-resolution logit map (a mirrored map at column W-1-x), softmax over the NC
//                          classes, fp32 sum over the maps, first maximum.  Only the class map is written;
//   msc_confidence_kernel<NC>  the same combine, writing the class map (uint8) and the confidence of each pixel,
//                          the mean probability of its class over the maps (pseudo-labels for self-training).
// Compiled without --use_fast_math so that the rescale's source index and weights are PyTorch's fp32
// arithmetic; the combine's softmax uses the __expf / __fdividef intrinsics explicitly.
#include <stdint.h>

#include "status.h"
#include "b200seg.h"
#include "upsample.cuh"

namespace b200 {

constexpr int kMscMaxMaps = 16;   // low-resolution maps one combine launch takes
constexpr int kMscMaxCls = 32;    // widest padded logit map (the compiled class counts are 2..32)
constexpr int kMaxDenseRows = 64; // batch limit of the network's [N, C] dense layers (b200_fc_small_fwd)
// Pixels one launch covers: the grid-stride loops index them in 32 bits (a 64-bit division is a
// subroutine call that needs a stack frame), with room for the last stride.
constexpr int64_t kMaxPixels = 1ll << 30;

// One output pixel (all three channels) per thread; the mirrored copy is written from the same value.
__global__ void __launch_bounds__(256)
image_rescale_kernel(const float* __restrict__ src, int N, int H, int W, float* __restrict__ dst, int h, int w,
                     int mirror) {
  const float sh = h > 1 ? (float)(H - 1) / (float)(h - 1) : 0.f;
  const float sw = w > 1 ? (float)(W - 1) / (float)(w - 1) : 0.f;
  const int total = N * h * w;  // <= kMaxPixels (host-checked)
  const int64_t plane_in = (int64_t)H * W, plane_out = (int64_t)h * w;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < total; p += gridDim.x * blockDim.x) {
    const int x = p % w;
    const int y = (p / w) % h;
    const int n = p / (w * h);
    const Interp iy = interp_at(y, sh, H), ix = interp_at(x, sw, W);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float* s = src + ((int64_t)n * 3 + c) * plane_in;
      const float a = __ldg(s + (int64_t)iy.i0 * W + ix.i0), b = __ldg(s + (int64_t)iy.i0 * W + ix.i1);
      const float d = __ldg(s + (int64_t)iy.i1 * W + ix.i0), e = __ldg(s + (int64_t)iy.i1 * W + ix.i1);
      // the order of upsample_bilinear2d_out_frame (ATen's CUDA kernel)
      const float v = iy.l0 * (ix.l0 * a + ix.l1 * b) + iy.l1 * (ix.l0 * d + ix.l1 * e);
      float* o = dst + ((int64_t)n * 3 + c) * plane_out + (int64_t)y * w;
      o[x] = v;
      if (mirror) dst[((int64_t)(N + n) * 3 + c) * plane_out + (int64_t)y * w + (w - 1 - x)] = v;
    }
  }
}

struct MscMap {
  const float* lr;  // fp32 NHWC [N, h, w, lr_ld]
  int lr_ld, h, w, mirrored;
};
struct MscTable {
  MscMap map[kMscMaxMaps];
  int n_maps;
};

// The map table arrives by value in the parameter block and is copied to shared memory once: indexed
// loads from the parameter block inside the pixel loop would cost hundreds of cycles each.
__device__ __forceinline__ void msc_stage_table(const MscTable& tab, int H, int W, MscMap* s_map, float* s_sh,
                                                float* s_sw) {
  if ((int)threadIdx.x < tab.n_maps) {
    const MscMap m = tab.map[threadIdx.x];
    s_map[threadIdx.x] = m;
    s_sh[threadIdx.x] = H > 1 ? (float)(m.h - 1) / (float)(H - 1) : 0.f;
    s_sw[threadIdx.x] = W > 1 ? (float)(m.w - 1) / (float)(W - 1) : 0.f;
  }
  __syncthreads();
}

// The per-pixel work of msc_argmax_kernel (whose own copy is kept as it was compiled before this helper
// existed): the sum over the maps of softmax(bilinear sample at (n, y, x)) in fp32 registers, and its first
// maximum (best, its sum bv).
template <int NC>
__device__ __forceinline__ void msc_accumulate(const MscMap* s_map, const float* s_sh, const float* s_sw,
                                               int n_maps, int n, int y, int x, int W, int& best, float& bv) {
  float acc[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) acc[c] = 0.f;
  for (int k = 0; k < n_maps; ++k) {
    const MscMap m = s_map[k];
    const Interp ih = interp_at(y, s_sh[k], m.h), iw = interp_at(m.mirrored ? W - 1 - x : x, s_sw[k], m.w);
    float v[NC];
    sample_logits<NC>(m.lr, m.lr_ld, m.h, m.w, n, ih, iw, v);
    float mx = v[0];
#pragma unroll
    for (int c = 1; c < NC; ++c) mx = fmaxf(mx, v[c]);
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      v[c] = __expf(v[c] - mx);
      s += v[c];
    }
    const float inv = __fdividef(1.f, s);
#pragma unroll
    for (int c = 0; c < NC; ++c) acc[c] += v[c] * inv;
  }
  best = 0;
  bv = acc[0];
#pragma unroll
  for (int c = 1; c < NC; ++c)
    if (acc[c] > bv) {
      bv = acc[c];
      best = c;
    }
}

template <int NC>
__global__ void __launch_bounds__(256)
msc_argmax_kernel(const __grid_constant__ MscTable tab, int N, int H, int W, void* __restrict__ pred,
                  int pred_is_u8) {
  __shared__ MscMap s_map[kMscMaxMaps];
  __shared__ float s_sh[kMscMaxMaps], s_sw[kMscMaxMaps];
  const int n_maps = tab.n_maps;
  if ((int)threadIdx.x < n_maps) {
    const MscMap m = tab.map[threadIdx.x];
    s_map[threadIdx.x] = m;
    s_sh[threadIdx.x] = H > 1 ? (float)(m.h - 1) / (float)(H - 1) : 0.f;
    s_sw[threadIdx.x] = W > 1 ? (float)(m.w - 1) / (float)(W - 1) : 0.f;
  }
  __syncthreads();
  const int total = N * H * W;  // <= kMaxPixels (host-checked)
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < total; p += gridDim.x * blockDim.x) {
    const int x = p % W;
    const int y = (p / W) % H;
    const int n = p / (W * H);
    float acc[NC];
#pragma unroll
    for (int c = 0; c < NC; ++c) acc[c] = 0.f;
    for (int k = 0; k < n_maps; ++k) {
      const MscMap m = s_map[k];
      const Interp ih = interp_at(y, s_sh[k], m.h), iw = interp_at(m.mirrored ? W - 1 - x : x, s_sw[k], m.w);
      float v[NC];
      sample_logits<NC>(m.lr, m.lr_ld, m.h, m.w, n, ih, iw, v);
      float mx = v[0];
#pragma unroll
      for (int c = 1; c < NC; ++c) mx = fmaxf(mx, v[c]);
      float s = 0.f;
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        v[c] = __expf(v[c] - mx);
        s += v[c];
      }
      const float inv = __fdividef(1.f, s);
#pragma unroll
      for (int c = 0; c < NC; ++c) acc[c] += v[c] * inv;
    }
    int best = 0;
    float bv = acc[0];
#pragma unroll
    for (int c = 1; c < NC; ++c)
      if (acc[c] > bv) {
        bv = acc[c];
        best = c;
      }
    if (pred_is_u8)
      static_cast<uint8_t*>(pred)[p] = (uint8_t)best;
    else
      static_cast<int64_t*>(pred)[p] = best;
  }
}

// The same combine, keeping the confidence of the prediction: conf = S[pred] / n_maps, the mean softmax
// probability of the first maximum (IEEE division: msc.cu is built without --use_fast_math).
template <int NC>
__global__ void __launch_bounds__(256)
msc_confidence_kernel(const __grid_constant__ MscTable tab, int N, int H, int W, uint8_t* __restrict__ pred,
                      float* __restrict__ conf) {
  __shared__ MscMap s_map[kMscMaxMaps];
  __shared__ float s_sh[kMscMaxMaps], s_sw[kMscMaxMaps];
  msc_stage_table(tab, H, W, s_map, s_sh, s_sw);
  const int n_maps = tab.n_maps;
  const float maps_f = (float)n_maps;
  const int total = N * H * W;  // <= kMaxPixels (host-checked)
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < total; p += gridDim.x * blockDim.x) {
    const int x = p % W;
    const int y = (p / W) % H;
    const int n = p / (W * H);
    int best;
    float bv;
    msc_accumulate<NC>(s_map, s_sh, s_sw, n_maps, n, y, x, W, best, bv);
    pred[p] = (uint8_t)best;
    conf[p] = bv / maps_f;
  }
}

static int msc_grid(int64_t total) {
  int64_t b = (total + 255) / 256;
  if (b > 148 * 16) b = 148 * 16;
  return (int)(b < 1 ? 1 : b);
}

#define B200_MSC_CLASS_COUNTS(X)                                                                           \
  X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15) X(16) X(17) X(18) X(19)      \
  X(20) X(21) X(22) X(23) X(24) X(25) X(26) X(27) X(28) X(29) X(30) X(31) X(32)

// The checks and the map table shared by b200_msc_argmax and b200_msc_confidence.
static int msc_table(const char* what, int n_maps, const float* const* maps, const int* lr_ld, const int* h_lr,
                     const int* w_lr, const int* mirrored, int N, int H, int W, int n_classes, MscTable& tab) {
  if (n_maps < 1 || n_maps > kMscMaxMaps)
    return set_error(B200_EINVAL, "%s: %d maps unsupported (1..%d)", what, n_maps, kMscMaxMaps);
  if (n_classes < 2 || n_classes > kMscMaxCls)
    return set_error(B200_EINVAL, "%s: %d classes unsupported (2..%d are compiled)", what, n_classes, kMscMaxCls);
  if (maps == nullptr || lr_ld == nullptr || h_lr == nullptr || w_lr == nullptr || mirrored == nullptr)
    return set_error(B200_EINVAL, "%s: NULL argument", what);
  if (N < 1 || H < 1 || W < 1) return set_error(B200_EINVAL, "%s: sizes N=%d %dx%d must be positive", what, N, H, W);
  const int width = (n_classes + 3) / 4 * 4;
  tab.n_maps = n_maps;
  for (int k = 0; k < n_maps; ++k) {
    if (maps[k] == nullptr) return set_error(B200_EINVAL, "%s: map %d is NULL", what, k);
    if (lr_ld[k] % 4 || lr_ld[k] < width)
      return set_error(B200_EINVAL, "%s: map %d pixel stride %d must be a multiple of 4, >= %d for %d classes",
                       what, k, lr_ld[k], width, n_classes);
    if (h_lr[k] < 1 || w_lr[k] < 1)
      return set_error(B200_EINVAL, "%s: map %d size %dx%d must be positive", what, k, h_lr[k], w_lr[k]);
    if (mirrored[k] != 0 && mirrored[k] != 1)
      return set_error(B200_EINVAL, "%s: map %d mirrored flag must be 0 or 1, got %d", what, k, mirrored[k]);
    tab.map[k] = MscMap{maps[k], lr_ld[k], h_lr[k], w_lr[k], mirrored[k]};
  }
  if ((int64_t)N * H * W > kMaxPixels)
    return set_error(B200_EINVAL, "%s: %d images of %dx%d exceed 2^30 pixels per launch", what, N, H, W);
  return B200_OK;
}

}  // namespace b200

using namespace b200;

extern "C" {

int b200_image_rescale(const float* src, int N, int H, int W, float* dst, int h, int w, int mirror,
                       cudaStream_t stream) {
  if (N < 1 || H < 1 || W < 1 || h < 1 || w < 1)
    return set_error(B200_EINVAL, "image_rescale: sizes N=%d %dx%d -> %dx%d must be positive", N, H, W, h, w);
  if (src == nullptr || dst == nullptr) return set_error(B200_EINVAL, "image_rescale: NULL image");
  if (mirror != 0 && mirror != 1) return set_error(B200_EINVAL, "image_rescale: mirror must be 0 or 1, got %d", mirror);
  if (mirror && 2 * N > kMaxDenseRows)
    return set_error(B200_EINVAL, "image_rescale: %d images and their mirrors exceed the network's batch limit of %d",
                     N, kMaxDenseRows);
  const int64_t total = (int64_t)N * h * w;
  if (total > kMaxPixels)
    return set_error(B200_EINVAL, "image_rescale: %d output images of %dx%d exceed 2^30 pixels per launch", N, h, w);
  image_rescale_kernel<<<msc_grid(total), 256, 0, stream>>>(src, N, H, W, dst, h, w, mirror);
  return check_launch("image_rescale");
}

int b200_msc_argmax(int n_maps, const float* const* maps, const int* lr_ld, const int* h_lr, const int* w_lr,
                    const int* mirrored, int N, int H, int W, int n_classes, void* pred, int pred_is_u8,
                    cudaStream_t stream) {
  if (pred == nullptr) return set_error(B200_EINVAL, "msc_argmax: NULL argument");
  if (pred_is_u8 != 0 && pred_is_u8 != 1)
    return set_error(B200_EINVAL, "msc_argmax: pred_is_u8 must be 0 or 1, got %d", pred_is_u8);
  MscTable tab{};
  const int rc = msc_table("msc_argmax", n_maps, maps, lr_ld, h_lr, w_lr, mirrored, N, H, W, n_classes, tab);
  if (rc != B200_OK) return rc;
  const int grid = msc_grid((int64_t)N * H * W);
  switch (n_classes) {
#define B200_MSC_CASE(nc)                                                                  \
  case nc:                                                                                 \
    msc_argmax_kernel<nc><<<grid, 256, 0, stream>>>(tab, N, H, W, pred, pred_is_u8);       \
    return check_launch("msc_argmax");
    B200_MSC_CLASS_COUNTS(B200_MSC_CASE)
#undef B200_MSC_CASE
  }
  return set_error(B200_EINVAL, "msc_argmax: %d classes unsupported", n_classes);
}

int b200_msc_confidence(int n_maps, const float* const* maps, const int* lr_ld, const int* h_lr, const int* w_lr,
                        const int* mirrored, int N, int H, int W, int n_classes, uint8_t* pred, float* conf,
                        cudaStream_t stream) {
  if (pred == nullptr || conf == nullptr) return set_error(B200_EINVAL, "msc_confidence: NULL argument");
  MscTable tab{};
  const int rc = msc_table("msc_confidence", n_maps, maps, lr_ld, h_lr, w_lr, mirrored, N, H, W, n_classes, tab);
  if (rc != B200_OK) return rc;
  const int grid = msc_grid((int64_t)N * H * W);
  switch (n_classes) {
#define B200_MSC_CASE(nc)                                                                  \
  case nc:                                                                                 \
    msc_confidence_kernel<nc><<<grid, 256, 0, stream>>>(tab, N, H, W, pred, conf);         \
    return check_launch("msc_confidence");
    B200_MSC_CLASS_COUNTS(B200_MSC_CASE)
#undef B200_MSC_CASE
  }
  return set_error(B200_EINVAL, "msc_confidence: %d classes unsupported", n_classes);
}

}  // extern "C"
