// ADVENT (Vu et al., CVPR 2019) on the bilinearly up-sampled (align_corners=True) class logits, fused with
// the up-sampling so that nothing of size N x n x H x W is written unless the self-information map is asked for:
//   self-information map (ADVENT's prob_2_entropy):  I_c = -p_c * log(p_c) / log(n),  p = softmax(up(lr))
//   entropy loss (ADVENT's entropy_loss):             E = sum over pixels and classes of I_c / (N*H*W)
// p_c * log(p_c) is computed as p_c * ls_c with ls = log_softmax from the log-sum-exp, so a probability that
// underflows to 0 in fp32 contributes 0 instead of 0 * -inf.
//   entropy_fwd_kernel<NC>  one CTA = an 8 x 32 output tile over the staged low-resolution rows; accumulates
//                           sum I in float64 and optionally writes I (bf16 NHWC, 32 channels, padding zero,
//                           plain or zero-bordered [N][H+2][W+2][32]).
//   entropy_bwd_kernel<NC>  one CTA = a 64 x 32 strip; per pixel the entropy gradient (with the loss sum, one
//                           pass) or the self-information backward from a bf16 dI, then the transposed
//                           interpolation as a gather over each low-resolution pixel's footprint with one
//                           atomicAdd per touched low-resolution value (the structure of loss.cu's
//                           upsample_bwd_strip_kernel).
// Both need an up-sampling factor >= ~7.75 along w and >= 7 along h (the `out` head of BiSeNet is 1/8 of the
// image), checked on the host.  Compiled without --use_fast_math; the softmax uses __expf / __logf explicitly.
#include <stdint.h>

#include <atomic>

#include "ptx.cuh"
#include "status.h"
#include "b200seg.h"
#include "upsample.cuh"

namespace b200 {

namespace ent {

constexpr int kMaxCls = 32;
constexpr int kMapLd = 32;       // channels per pixel of the self-information map
constexpr int TW = 32, TH = 8;   // forward tile
constexpr int LJ = 6;            // low-res columns under 32 output columns: 31 * sw + 2 <= 6
constexpr int LI_ROW = 3;        // low-res rows under 8 output rows:         7 * sh + 2 <= 3
constexpr int SH_ROWS = 64;      // rows of a backward strip (8 warps x 8 rows)
constexpr int LI = 11;           // low-res rows under a strip:              63 * sh + 2 <= 11
constexpr int64_t kMaxPixels = (1ll << 31) - 1;   // N*H*W (and the bordered N*(H+2)*(W+2)) of one launch

// Private copies of loss.cu's staging helpers (loss.cu is left as it is).
template <int ROWS, int NC>
__device__ __forceinline__ void stage_rows(const float* __restrict__ lr, int lr_ld, int h_lr, int w_lr, int n,
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
__device__ __forceinline__ void sample_staged(const float* s_lr, const Interp& ih, const Interp& iw, int i_min,
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

// v: logits in, p out; ls: log_softmax out.  Returns h = -sum p * ls (natural-log entropy).
template <int NC>
__device__ __forceinline__ float softmax_logsoftmax(float (&v)[NC], float (&ls)[NC]) {
  float m = v[0];
#pragma unroll
  for (int c = 1; c < NC; ++c) m = fmaxf(m, v[c]);
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    ls[c] = v[c] - m;
    v[c] = __expf(ls[c]);
    s += v[c];
  }
  const float inv = 1.f / s, lse = __logf(s);
  float h = 0.f;
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    v[c] *= inv;
    ls[c] -= lse;
    h -= v[c] * ls[c];
  }
  return h;
}

__device__ __forceinline__ int64_t bordered_pixel(int n, int h, int w, int H, int W) {
  return ((int64_t)n * (H + 2) + (h + 1)) * (W + 2) + (w + 1);
}
__device__ __forceinline__ void zero_map_pixel(__nv_bfloat16* q) {
#pragma unroll
  for (int c = 0; c < kMapLd / 8; ++c) reinterpret_cast<uint4*>(q)[c] = make_uint4(0u, 0u, 0u, 0u);
}
// The border pixels next to output pixel (h, w) of the zero-bordered layout.
__device__ __forceinline__ void zero_border_of(__nv_bfloat16* base, int n, int h, int w, int H, int W) {
  const bool top = h == 0, bot = h == H - 1, left = w == 0, right = w == W - 1;
  if (!(top | bot | left | right)) return;
  if (top) zero_map_pixel(base + bordered_pixel(n, -1, w, H, W) * kMapLd);
  if (bot) zero_map_pixel(base + bordered_pixel(n, H, w, H, W) * kMapLd);
  if (left) zero_map_pixel(base + bordered_pixel(n, h, -1, H, W) * kMapLd);
  if (right) zero_map_pixel(base + bordered_pixel(n, h, W, H, W) * kMapLd);
  if (top && left) zero_map_pixel(base + bordered_pixel(n, -1, -1, H, W) * kMapLd);
  if (top && right) zero_map_pixel(base + bordered_pixel(n, -1, W, H, W) * kMapLd);
  if (bot && left) zero_map_pixel(base + bordered_pixel(n, H, -1, H, W) * kMapLd);
  if (bot && right) zero_map_pixel(base + bordered_pixel(n, H, W, H, W) * kMapLd);
}

// Odd per-pixel class stride of the strip's vertical partials (no bank conflicts across a warp's columns).
template <int NC>
__host__ __device__ constexpr int strip_stride() { return NC | 1; }
template <int NC>
constexpr int bwd_smem_bytes() {
  return (LI * LJ * staged_width<NC>() + LI * TW * strip_stride<NC>()) * (int)sizeof(float);
}

}  // namespace ent

// ------------------------------------------------------------------ forward
// map == nullptr: acc[0] += sum over the pixels of sum_c I_c only.
// map != nullptr: also I (bf16, 32 channels per pixel, channels >= NC zero); layout 1 = [N][H][W][32],
// layout 2 = [N][H+2][W+2][32] with the map in rows / cols 1..H / 1..W and the border written zero.
// acc may be nullptr when the map is written.
template <int NC>
__global__ void __launch_bounds__(ent::TH * ent::TW)
entropy_fwd_kernel(const float* __restrict__ lr, int lr_ld, int N, int h_lr, int w_lr, int H, int W,
                   float inv_ln_n, __nv_bfloat16* __restrict__ map, int layout, double* __restrict__ acc) {
  using namespace ent;
  __shared__ __align__(16) float s_lr[LI_ROW * LJ * staged_width<NC>()];
  __shared__ Interp s_iw[TW], s_ih[TH];
  __shared__ float s_part[TH];
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
  stage_rows<LI_ROW, NC>(lr, lr_ld, h_lr, w_lr, n, s_ih[0].i0, s_iw[0].i0, s_lr);
  __syncthreads();
  const int h = h_base + ty, w = w_base + tx;
  float ent_sum = 0.f;
  if (h < H && w < W) {
    float v[NC], ls[NC];
    sample_staged<NC>(s_lr, s_ih[ty], s_iw[tx], s_ih[0].i0, s_iw[0].i0, v);
    ent_sum = softmax_logsoftmax<NC>(v, ls) * inv_ln_n;
    if (map != nullptr) {
      int64_t pix = ((int64_t)n * H + h) * W + w;
      if (layout == 2) {
        pix = bordered_pixel(n, h, w, H, W);
        zero_border_of(map, n, h, w, H, W);
      }
      uint32_t pk[kMapLd / 2];
#pragma unroll
      for (int c = 0; c < kMapLd / 2; ++c) {
        const float a = (2 * c < NC) ? -v[2 * c < NC ? 2 * c : 0] * ls[2 * c < NC ? 2 * c : 0] * inv_ln_n : 0.f;
        const float b =
            (2 * c + 1 < NC) ? -v[2 * c + 1 < NC ? 2 * c + 1 : 0] * ls[2 * c + 1 < NC ? 2 * c + 1 : 0] * inv_ln_n : 0.f;
        pk[c] = pack_bf16(a, b);
      }
      uint4* q = reinterpret_cast<uint4*>(map + pix * kMapLd);
#pragma unroll
      for (int c = 0; c < kMapLd / 8; ++c) q[c] = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
    }
  }
  if (acc != nullptr) {
    const float ws = warp_sum(ent_sum);
    if (tx == 0) s_part[ty] = ws;
    __syncthreads();
    if (threadIdx.x == 0) {
      double a = 0.0;
      for (int i = 0; i < TH; ++i) a += s_part[i];
      atomicAdd(acc, a);
    }
  }
}

// ------------------------------------------------------------------ backward
// d_lr[n, i, j, c] += sum over output pixels of wh(h, i) * ww(w, j) * G[n, h, w, c] with
//   mode 0 (entropy training pass): G = d(sum_c I_c)/dz = -(p / ln n) * (ls + h), h = -sum p * ls;
//          acc[0] += sum over the pixels of sum_c I_c (acc may be nullptr)
//   mode 1 (self-information backward): dp = -dI * (ls + 1) / ln n, G = p * (dp - sum_k p_k dp_k), dI bf16 with
//          32 channels per pixel, layout 1 = [N][H][W][32], layout 2 = [N][H+2][W+2][32] read at the interior
// One CTA = a strip of SH_ROWS x TW pixels; warp wp owns rows 8wp .. 8wp+7 and a lane one column, folding its
// pixels' gradients into <= 3 low-resolution rows in registers; the per-column partials meet in shared memory
// and are reduced along w with a weight table, one atomicAdd per touched low-resolution value.
template <int NC>
__global__ void __launch_bounds__(256, 1)
entropy_bwd_kernel(const float* __restrict__ lr, int lr_ld, int N, int h_lr, int w_lr, int H, int W,
                   float inv_ln_n, int mode, const __nv_bfloat16* __restrict__ d_map, int layout,
                   float* __restrict__ d_lr, double* __restrict__ acc) {
  using namespace ent;
  extern __shared__ __align__(16) float s_dyn[];
  float* s_lr = s_dyn;
  constexpr int SV = strip_stride<NC>();
  float (*s_v)[TW][SV] = reinterpret_cast<float (*)[TW][SV]>(s_dyn + LI * LJ * staged_width<NC>());
  __shared__ float s_wx[LJ][TW];
  __shared__ int s_xlo[LJ], s_xhi[LJ];
  __shared__ Interp s_iw[TW], s_ih[SH_ROWS];
  __shared__ float s_part[8];
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
  stage_rows<LI, NC>(lr, lr_ld, h_lr, w_lr, n, i_min, j_min, s_lr);
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
  float my_ent = 0.f;
#pragma unroll 1
  for (int r = 0; r < 8; ++r) {
    const int h = h_base + wp * 8 + r;
    if (h >= H) break;
    if (w >= W) continue;
    const Interp ih = s_ih[wp * 8 + r];
    float g[NC], t[NC];
    sample_staged<NC>(s_lr, ih, iw, i_min, j_min, g);
    const float hn = softmax_logsoftmax<NC>(g, t);   // g = p, t = log p
    if (mode == 0) {
      my_ent += hn * inv_ln_n;
#pragma unroll
      for (int c = 0; c < NC; ++c) g[c] = -g[c] * inv_ln_n * (t[c] + hn);
    } else {
      const int64_t pix = layout == 2 ? bordered_pixel(n, h, w, H, W) : ((int64_t)n * H + h) * W + w;
      const uint4* q = reinterpret_cast<const uint4*>(d_map + pix * kMapLd);
#pragma unroll
      for (int k = 0; k < (NC + 7) / 8; ++k) {
        const uint4 u = __ldg(q + k);
        const uint32_t raw[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int c = 8 * k + e;
          if (c < NC) {
            const float2 f = unpack_bf16(raw[e >> 1]);
            t[c] = -((e & 1) ? f.y : f.x) * (t[c] + 1.f) * inv_ln_n;   // dp_c
          }
        }
      }
      float dot = 0.f;
#pragma unroll
      for (int c = 0; c < NC; ++c) dot += g[c] * t[c];
#pragma unroll
      for (int c = 0; c < NC; ++c) g[c] = g[c] * (t[c] - dot);
    }
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
  if (acc != nullptr) {
    const float ws = warp_sum(my_ent);
    if (tx == 0) s_part[wp] = ws;
  }
  __syncthreads();
  if (acc != nullptr && threadIdx.x == 0) {
    double a = 0.0;
    for (int i = 0; i < 8; ++i) a += s_part[i];
    atomicAdd(acc, a);
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

namespace ent {

struct Args {
  const float* lr; int lr_ld, N, h_lr, w_lr, H, W; float inv_ln_n; int mode;
  __nv_bfloat16* map; int layout; float* d_lr; double* acc;
};

// The backward's dynamic shared memory exceeds the default 48 KB limit from 28 classes on; the opt-in is a
// per-device function attribute, set once per instance and device.
template <int NC>
static cudaError_t bwd_smem_optin() {
  static std::atomic<unsigned long long> done{0};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const unsigned long long bit = 1ull << (dev & 63);
  if (done.load(std::memory_order_acquire) & bit) return cudaSuccess;
  e = cudaFuncSetAttribute(entropy_bwd_kernel<NC>, cudaFuncAttributeMaxDynamicSharedMemorySize, bwd_smem_bytes<NC>());
  if (e == cudaSuccess) done.fetch_or(bit, std::memory_order_release);
  return e;
}

template <int NC>
static int launch_fwd(const Args& a, cudaStream_t stream) {
  const int tiles = ((a.W + TW - 1) / TW) * ((a.H + TH - 1) / TH) * a.N;
  entropy_fwd_kernel<NC><<<tiles, TH * TW, 0, stream>>>(a.lr, a.lr_ld, a.N, a.h_lr, a.w_lr, a.H, a.W, a.inv_ln_n,
                                                        a.map, a.layout, a.acc);
  return check_launch("entropy_fwd");
}

template <int NC>
static int launch_bwd(const Args& a, cudaStream_t stream) {
  const cudaError_t e = bwd_smem_optin<NC>();
  if (e != cudaSuccess) return set_error(B200_ECUDA, "entropy_bwd shared memory: %s", cudaGetErrorString(e));
  const int strips = ((a.W + TW - 1) / TW) * ((a.H + SH_ROWS - 1) / SH_ROWS) * a.N;
  entropy_bwd_kernel<NC><<<strips, 256, bwd_smem_bytes<NC>(), stream>>>(
      a.lr, a.lr_ld, a.N, a.h_lr, a.w_lr, a.H, a.W, a.inv_ln_n, a.mode, a.map, a.layout, a.d_lr, a.acc);
  return check_launch("entropy_bwd");
}

#define B200_ENT_FOR_EACH_CLASS_COUNT(X)                                                                   \
  X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15) X(16) X(17) X(18) X(19)      \
  X(20) X(21) X(22) X(23) X(24) X(25) X(26) X(27) X(28) X(29) X(30) X(31) X(32)

// The checks both entry points share; `map_mode`: a map is read or written (p_ld and the layout matter).
static int check_args(const char* what, int N, int h_lr, int w_lr, int H, int W, int n_classes, int lr_ld,
                      bool map_mode, int p_ld, int layout) {
  if (n_classes < 2 || n_classes > kMaxCls)
    return set_error(B200_EINVAL, "%s: %d classes unsupported (2..%d are compiled)", what, n_classes, kMaxCls);
  const int ld4 = (n_classes + 3) / 4 * 4;
  if (lr_ld % 4 || lr_ld < ld4)
    return set_error(B200_EINVAL, "%s: logits pixel stride %d must be a multiple of 4, >= %d for %d classes", what,
                     lr_ld, ld4, n_classes);
  if (N < 1 || h_lr < 1 || w_lr < 1 || H < 1 || W < 1)
    return set_error(B200_EINVAL, "%s: empty size N=%d %dx%d -> %dx%d", what, N, h_lr, w_lr, H, W);
  if (map_mode) {
    if (p_ld != kMapLd) return set_error(B200_EINVAL, "%s: map pixel stride %d must be %d", what, p_ld, kMapLd);
    if (layout != 1 && layout != 2) return set_error(B200_EINVAL, "%s: map layout %d unknown (1 or 2)", what, layout);
    if (layout == 2 && (H % 2 || W % 2))
      return set_error(B200_EINVAL, "%s: the zero-bordered layout needs even H and W, got %dx%d", what, H, W);
  }
  const int64_t pixels = (int64_t)N * (H + 2) * (W + 2);
  if (pixels > kMaxPixels)
    return set_error(B200_EINVAL, "%s: N*(H+2)*(W+2) = %lld exceeds %lld", what, (long long)pixels,
                     (long long)kMaxPixels);
  const float sh = H > 1 ? (float)(h_lr - 1) / (float)(H - 1) : 0.f;
  const float sw = W > 1 ? (float)(w_lr - 1) / (float)(W - 1) : 0.f;
  if (!(sw * (TW - 1) + 2.f <= (float)LJ && sh * (TH - 1) + 2.f <= (float)LI_ROW &&
        sh * (SH_ROWS - 1) + 2.f <= (float)LI))
    return set_error(B200_EINVAL,
                     "%s: scale %dx%d -> %dx%d is below the supported up-sampling factor (>= 7.75 along w, >= 7 "
                     "along h)", what, h_lr, w_lr, H, W);
  return 0;
}

static float inv_ln(int n_classes) { return (float)(1.0 / __builtin_log((double)n_classes)); }

}  // namespace ent
}  // namespace b200

using namespace b200;

extern "C" {

int b200_entropy_fwd(const float* lr, int lr_ld, int N, int h_lr, int w_lr, int H, int W, int n_classes,
                     int mode, void* map, int p_ld, int layout, double* acc, cudaStream_t stream) {
  if (mode != 0 && mode != 1) return set_error(B200_EINVAL, "entropy_fwd: mode %d unknown (0 or 1)", mode);
  const int rc = ent::check_args("entropy_fwd", N, h_lr, w_lr, H, W, n_classes, lr_ld, mode == 1, p_ld, layout);
  if (rc) return rc;
  if (mode == 0 && acc == nullptr) return set_error(B200_EINVAL, "entropy_fwd: mode 0 needs the accumulator");
  if (mode == 1 && map == nullptr) return set_error(B200_EINVAL, "entropy_fwd: mode 1 needs the map");
  const ent::Args a{lr, lr_ld, N, h_lr, w_lr, H, W, ent::inv_ln(n_classes), mode,
                    mode == 1 ? static_cast<__nv_bfloat16*>(map) : nullptr, layout, nullptr, acc};
  switch (n_classes) {
#define B200_ENT_FWD_CASE(nc) case nc: return ent::launch_fwd<nc>(a, stream);
    B200_ENT_FOR_EACH_CLASS_COUNT(B200_ENT_FWD_CASE)
#undef B200_ENT_FWD_CASE
  }
  return set_error(B200_EINVAL, "entropy_fwd: %d classes unsupported", n_classes);
}

int b200_entropy_bwd(const float* lr, int lr_ld, int N, int h_lr, int w_lr, int H, int W, int n_classes,
                     int mode, const void* d_map, int p_ld, int layout, float* d_lr, double* acc,
                     cudaStream_t stream) {
  if (mode != 0 && mode != 1) return set_error(B200_EINVAL, "entropy_bwd: mode %d unknown (0 or 1)", mode);
  const int rc = ent::check_args("entropy_bwd", N, h_lr, w_lr, H, W, n_classes, lr_ld, mode == 1, p_ld, layout);
  if (rc) return rc;
  if (d_lr == nullptr) return set_error(B200_EINVAL, "entropy_bwd: d_lr is required");
  if (mode == 1 && d_map == nullptr) return set_error(B200_EINVAL, "entropy_bwd: mode 1 needs the map gradient");
  const ent::Args a{lr, lr_ld, N, h_lr, w_lr, H, W, ent::inv_ln(n_classes), mode,
                    mode == 1 ? const_cast<__nv_bfloat16*>(static_cast<const __nv_bfloat16*>(d_map)) : nullptr,
                    layout, d_lr, mode == 0 ? acc : nullptr};
  switch (n_classes) {
#define B200_ENT_BWD_CASE(nc) case nc: return ent::launch_bwd<nc>(a, stream);
    B200_ENT_FOR_EACH_CLASS_COUNT(B200_ENT_BWD_CASE)
#undef B200_ENT_BWD_CASE
  }
  return set_error(B200_EINVAL, "entropy_bwd: %d classes unsupported", n_classes);
}

}  // extern "C"
