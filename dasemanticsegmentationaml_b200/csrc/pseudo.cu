// Pseudo-labels for target-domain self-training (BDL's SSL stage, CBST, IAST):
//   class_select_hist_kernel   one 8-bit radix pass of an exact per-class k-th largest: for each pixel whose
//                              confidence key matches its class's prefix so far, hist[class][next 8 bits] += 1
//                              (shared-memory counters, flushed as uint64 to global memory);
//   class_select_pick_kernel   one warp per class walks its 256 bins from the top, fixes the next 8 bits of
//                              the class's key and the remaining rank; after the last pass, the thresholds;
//   pseudo_label_apply_kernel  label = pred where conf >= thr[pred], else 255.
// A selection is four hist / pick rounds over any number of batches; the 64-bit totals live in hist and
// state, so the counts of a whole target set (1.56 G pixels for Cityscapes train at 512x1024) are exact.
// Built without --use_fast_math: k_c = ceil(portion * count_c) must be Python's float64 arithmetic.
#include <math.h>
#include <stdint.h>

#include "status.h"
#include "b200seg.h"

namespace b200 {

constexpr int kSelMaxCls = 32;
constexpr int kSelBins = 256;
// Shared-memory row stride of a class's bins: odd, so that pixels of different classes in the same bin
// (confidences pile up near 1.0) fall on different banks.
constexpr int kSelStride = kSelBins + 1;
constexpr int kSelThreads = 512;
constexpr int64_t kSelMaxPixels = 1ll << 30;  // per call: the pixel loops index in 32 bits
constexpr uint32_t kNoSlot = 0xFFFFFFFFu;

// Order-preserving key of an fp32 bit pattern: unsigned comparison of keys orders the values, -0 below +0.
__device__ __forceinline__ uint32_t order_key(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_value(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}

// Counts one pixel per lane.  Lanes of a warp that hit the same (class, bin) counter are merged first
// (match.any), so a warp issues one shared atomic per distinct counter instead of serialising on one address.
// Every lane of the warp must call it (idle lanes with valid = false).
__device__ __forceinline__ void sel_count(uint32_t* s_h, const uint32_t* s_prefix, int c, float v, bool valid,
                                          int n, int shift, uint32_t mask) {
  uint32_t slot = kNoSlot;
  if (valid && c < n && !isnan(v)) {
    const uint32_t k = order_key(v);
    if ((k & mask) == (s_prefix[c] & mask)) slot = c * kSelStride + ((k >> shift) & 0xFFu);
  }
  const uint32_t peers = __match_any_sync(0xFFFFFFFFu, slot);
  if (slot != kNoSlot && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&s_h[slot], (uint32_t)__popc(peers));
}

// vec: pred is 8-byte and conf 32-byte aligned, so eight pixels load as one uint2 and two float4.  The loop
// trip counts are warp-uniform (q - lane is the warp's first pixel) because match.any needs the whole warp.
__global__ void __launch_bounds__(kSelThreads, 2)
class_select_hist_kernel(const uint8_t* __restrict__ pred, const float* __restrict__ conf, int count, int n,
                         int pass, const uint64_t* __restrict__ state, unsigned long long* __restrict__ hist,
                         int vec) {
  extern __shared__ uint32_t s_h[];  // [n][kSelStride]
  __shared__ uint32_t s_prefix[kSelMaxCls];
  for (int i = threadIdx.x; i < n * kSelStride; i += blockDim.x) s_h[i] = 0u;
  if ((int)threadIdx.x < n) s_prefix[threadIdx.x] = pass == 0 ? 0u : (uint32_t)state[3 * threadIdx.x];
  __syncthreads();
  const int shift = 24 - 8 * pass;
  const uint32_t mask = pass == 0 ? 0u : 0xFFFFFFFFu << (shift + 8);
  const int lane = threadIdx.x & 31;
  const int stride = gridDim.x * blockDim.x;
  const int first = blockIdx.x * blockDim.x + threadIdx.x;
  int done = 0;
  if (vec) {
    const int n8 = count >> 3;
    for (int q = first; q - lane < n8; q += stride) {
      const bool ok = q < n8;
      uint2 c8 = make_uint2(0u, 0u);
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
      if (ok) {
        c8 = __ldg(reinterpret_cast<const uint2*>(pred) + q);
        a = __ldg(reinterpret_cast<const float4*>(conf) + 2 * q);
        b = __ldg(reinterpret_cast<const float4*>(conf) + 2 * q + 1);
      }
      const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
      for (int j = 0; j < 8; ++j)
        sel_count(s_h, s_prefix, ((j < 4 ? c8.x : c8.y) >> (8 * (j & 3))) & 0xFFu, v[j], ok, n, shift, mask);
    }
    done = n8 << 3;
  }
  for (int i = done + first; i - lane < count; i += stride) {
    const bool ok = i < count;
    sel_count(s_h, s_prefix, ok ? (int)pred[i] : 0, ok ? conf[i] : 0.f, ok, n, shift, mask);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n * kSelBins; i += blockDim.x) {
    const uint32_t v = s_h[(i >> 8) * kSelStride + (i & 0xFF)];
    if (v) atomicAdd(hist + i, (unsigned long long)v);
  }
}

// state[c] = {key prefix found so far, remaining 0-based rank from the top, count_c}.  Lane l of class c's
// warp holds bins 8l..8l+7; the lane whose bins contain the rank walks them from the top.
__global__ void __launch_bounds__(kSelMaxCls * 32)
class_select_pick_kernel(int n, int pass, double portion, float cap, unsigned long long* __restrict__ state,
                         unsigned long long* __restrict__ hist, float* __restrict__ thr, int64_t* __restrict__ counts) {
  const int c = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (c >= n) return;
  unsigned long long* h = hist + c * kSelBins + 8 * lane;
  unsigned long long* st = state + 3 * c;
  unsigned long long b[8], s = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    b[j] = h[j];
    s += b[j];
    h[j] = 0ull;  // ready for the next pass (or the next selection)
  }
  unsigned long long incl = s;  // sum over lanes >= this one
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long t = __shfl_down_sync(0xFFFFFFFFu, incl, o);
    if (lane + o < 32) incl += t;
  }
  unsigned long long prefix, rank, cnt;
  if (pass == 0) {
    cnt = __shfl_sync(0xFFFFFFFFu, incl, 0);
    const double kd = ceil(portion * (double)cnt);
    const unsigned long long k = kd < 1.0 ? 1ull : (kd >= (double)cnt ? cnt : (unsigned long long)kd);
    prefix = 0ull;
    rank = cnt ? k - 1 : 0ull;
  } else {
    prefix = st[0];
    rank = st[1];
    cnt = st[2];
  }
  if (cnt) {
    const unsigned long long above = incl - s;
    const uint32_t sel = __ballot_sync(0xFFFFFFFFu, above <= rank && rank < incl);
    const int owner = sel ? __ffs(sel) - 1 : 0;
    int d = 0;
    unsigned long long r = rank - above;
    if (lane == owner) {
      for (int j = 7; j >= 0; --j) {
        if (r < b[j]) {
          d = 8 * lane + j;
          break;
        }
        r -= b[j];
      }
    }
    d = __shfl_sync(0xFFFFFFFFu, d, owner);
    r = __shfl_sync(0xFFFFFFFFu, r, owner);
    prefix |= (unsigned long long)d << (24 - 8 * pass);
    rank = r;
  }
  if (lane == 0) {
    st[0] = prefix;
    st[1] = rank;
    st[2] = cnt;
    if (pass == 3) {
      thr[c] = cnt ? fminf(key_value((uint32_t)prefix), cap) : cap;
      counts[c] = (int64_t)cnt;
    }
  }
}

// pred and out may be the same buffer (uint8 output in place): each pixel is read before it is written.
__global__ void __launch_bounds__(256)
pseudo_label_apply_kernel(const uint8_t* pred, const float* __restrict__ conf, int count, int n,
                          const float* __restrict__ thr, void* out, int out_is_u8) {
  __shared__ float s_thr[kSelMaxCls];
  if ((int)threadIdx.x < n) s_thr[threadIdx.x] = thr[threadIdx.x];
  __syncthreads();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    const int c = pred[i];
    const float v = conf[i];
    const int label = (c < n && v >= s_thr[c]) ? c : 255;
    if (out_is_u8)
      static_cast<uint8_t*>(out)[i] = (uint8_t)label;
    else
      static_cast<int64_t*>(out)[i] = label;
  }
}

static int sel_check(const char* what, int64_t count, int n_classes) {
  if (n_classes < 2 || n_classes > kSelMaxCls)
    return set_error(B200_EINVAL, "%s: %d classes unsupported (2..%d)", what, n_classes, kSelMaxCls);
  if (count < 0 || count > kSelMaxPixels)
    return set_error(B200_EINVAL, "%s: %lld pixels per call unsupported (0..2^30; split larger inputs)", what,
                     (long long)count);
  return B200_OK;
}

}  // namespace b200

using namespace b200;

extern "C" {

int b200_class_select_hist(const uint8_t* pred, const float* conf, int64_t count, int n_classes, int pass,
                           const uint64_t* state, uint64_t* hist, cudaStream_t stream) {
  const int rc = sel_check("class_select_hist", count, n_classes);
  if (rc != B200_OK) return rc;
  if (pred == nullptr || conf == nullptr || state == nullptr || hist == nullptr)
    return set_error(B200_EINVAL, "class_select_hist: NULL argument");
  if (pass < 0 || pass > 3) return set_error(B200_EINVAL, "class_select_hist: pass %d outside 0..3", pass);
  if (count == 0) return B200_OK;
  const int vec = ((uintptr_t)pred % 8 == 0 && (uintptr_t)conf % 32 == 0) ? 1 : 0;
  const int64_t work = vec ? count / 8 : count;
  int64_t grid = (work + kSelThreads - 1) / kSelThreads;
  if (grid > 148 * 2) grid = 148 * 2;
  if (grid < 1) grid = 1;
  const size_t smem = (size_t)n_classes * kSelStride * sizeof(uint32_t);
  class_select_hist_kernel<<<(int)grid, kSelThreads, smem, stream>>>(
      pred, conf, (int)count, n_classes, pass, state, reinterpret_cast<unsigned long long*>(hist), vec);
  return check_launch("class_select_hist");
}

int b200_class_select_pick(int n_classes, int pass, double portion, float cap, uint64_t* state, uint64_t* hist,
                           float* thr, int64_t* counts, cudaStream_t stream) {
  const int rc = sel_check("class_select_pick", 0, n_classes);
  if (rc != B200_OK) return rc;
  if (state == nullptr || hist == nullptr || thr == nullptr || counts == nullptr)
    return set_error(B200_EINVAL, "class_select_pick: NULL argument");
  if (pass < 0 || pass > 3) return set_error(B200_EINVAL, "class_select_pick: pass %d outside 0..3", pass);
  if (!(isfinite(portion) && portion > 0.0 && portion <= 1.0))
    return set_error(B200_EINVAL, "class_select_pick: portion %g must be finite and in (0, 1]", portion);
  if (!(isfinite(cap) && cap > 0.f && cap <= 1.f))
    return set_error(B200_EINVAL, "class_select_pick: cap %g must be finite and in (0, 1]", (double)cap);
  class_select_pick_kernel<<<1, 32 * n_classes, 0, stream>>>(n_classes, pass, portion, cap,
                                                              reinterpret_cast<unsigned long long*>(state),
                                                              reinterpret_cast<unsigned long long*>(hist), thr, counts);
  return check_launch("class_select_pick");
}

int b200_pseudo_label_apply(const uint8_t* pred, const float* conf, int64_t count, int n_classes, const float* thr,
                            void* out, int out_is_u8, cudaStream_t stream) {
  const int rc = sel_check("pseudo_label_apply", count, n_classes);
  if (rc != B200_OK) return rc;
  if (pred == nullptr || conf == nullptr || thr == nullptr || out == nullptr)
    return set_error(B200_EINVAL, "pseudo_label_apply: NULL argument");
  if (out_is_u8 != 0 && out_is_u8 != 1)
    return set_error(B200_EINVAL, "pseudo_label_apply: out_is_u8 must be 0 or 1, got %d", out_is_u8);
  if (count == 0) return B200_OK;
  int64_t grid = (count + 255) / 256;
  if (grid > 148 * 16) grid = 148 * 16;
  pseudo_label_apply_kernel<<<(int)grid, 256, 0, stream>>>(pred, conf, (int)count, n_classes, thr, out, out_is_u8);
  return check_launch("pseudo_label_apply");
}

}  // extern "C"
