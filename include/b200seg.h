/*
 * libb200seg.so — C ABI of the B200-native (sm_100a) STDC-BiSeNet / domain-discriminator hot path.
 *
 * This is the drop-in boundary: plain pointers, sizes and a CUDA stream; no C++ or torch types.
 * The reference (TiloccaS/DASemanticSegmentationAML) has no native interface of its own — all of
 * its GPU arithmetic goes through PyTorch's dispatcher into cuDNN/ATen — so each entry point cites
 * the reference call site (file:line, relative to the reference root) whose arithmetic it replaces.
 * The binding a maintainer adds on the reference side is a ctypes stub (see INTEGRATION.md).
 *
 * Conventions
 *   - Activations are bf16 NHWC.  A tensor argument is (base pointer, ld): `ld` is the distance in
 *     elements between consecutive pixels, so a channel slice of a wider buffer is passed by
 *     offsetting the base pointer (this is how torch.cat is avoided).  ld and channel offsets are
 *     multiples of 8 (16 bytes), channel counts C multiples of 8 unless stated.
 *   - Parameters (filters, BatchNorm vectors, biases) are the fp32 PyTorch tensors in PyTorch layout.
 *   - Every call is asynchronous on `stream`, never synchronises, never allocates, and keeps no
 *     pointer after returning (TMA descriptors are built per call from the arguments): all calls
 *     are re-entrant and CUDA-graph capturable.  The caller owns every buffer.
 *   - Return value: 0, or a negative B200_E* code; b200_last_error() gives the text of the last
 *     failure on the calling thread.  b200_check_device() refuses anything but compute capability
 *     10.x — there is no fallback path.
 *   - act codes: 0 none, 1 ReLU, 2 LeakyReLU(slope), 3 sigmoid (dense-vector layers only).
 */
#ifndef B200SEG_H_
#define B200SEG_H_

#include <stddef.h>
#include <stdint.h>

#ifndef __DRIVER_TYPES_H__
typedef struct CUstream_st* cudaStream_t;
#endif

#define B200_OK 0
#define B200_EINVAL (-1)  /* bad shape / alignment / argument */
#define B200_ECUDA (-2)   /* CUDA runtime error */
#define B200_EDRIVER (-3) /* driver entry point / tensor-map encoding failure */
#define B200_EARCH (-4)   /* device is not sm_100 */

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ library */
const char* b200_last_error(void);
int b200_version(void);
int b200_check_device(void);

/* ---------------------------------------------- dense convolutions (tcgen05) */
/* fp32 [Cout][Cin][RS] filter -> bf16 K-major GEMM operand [rows_pad][RS][inner_pad]
 * (rows, inner) = (Cout, Cin), or (Cin, Cout) when transpose != 0 (operand of the data gradient).
 * Replaces cuDNN's internal filter transforms for nn.Conv2d at model/stdcnet.py:9,
 * model/model_stages.py:14-19, model/discriminator.py:9-13. */
int b200_pack_filter(const float* w, void* out_bf16, int Cout, int Cin, int RS, int rows_pad,
                     int inner_pad, int transpose, cudaStream_t stream);
/* transpose | 2 ("pair view", RS = 8, inner/rows = 64): the 4x4 / stride-2 / pad-1 filter of
 * FCDiscriminator.conv1 (discriminator.py:9,18) re-expressed over COLUMN PAIRS of the zero-bordered
 * probability map [N][H+2][W+2][32] that b200_upsample_fwd(mode 2, out_flag 2) writes: pair channel
 * ci2 = s*32 + c, tap t = kh*2 + b  <->  w[co][c][kh][2b + s].  The layer then runs through b200_conv_igemm /
 * b200_conv_wgrad as a stride-1 filter of 8 taps with 128-byte input rows (tap (a, r, b): dh = a,
 * dw = r*(W+2)/2 + b over the [N][(H+2)/2][W+2][64] view, slab (2a + r)*2 + b). */

/* The same for many filters in one launch: table_dev = int64 [n][8] on the device =
 * {src, dst, Cout, Cin, RS, rows_pad, inner_pad, transpose} (repacking after an optimizer step). */
int b200_pack_filters_batched(const int64_t* table_dev, int n_filters, cudaStream_t stream);

/* Implicit-GEMM convolution on the 5th-gen tensor cores (TMA-fed, TMEM accumulators):
 *   out[n, (h*os+oa), (w*os+ob), co] = act(bias[co] + sum_{tap, ci} in[n, h*is+dh, w*is+dw, ci] * filt[co, slab, ci])
 * `taps` = [n_classes][taps_stride][3] = (dh, dw, slab).  One class with is = conv stride is the
 * forward pass of nn.Conv2d (stdcnet.py:13, model_stages.py:26,46-47, discriminator.py:18-25);
 * with the transposed filter and (for stride 2) the four output-parity classes it is the data
 * gradient autograd derives for the same layers.  Out-of-bounds input is read as zero (padding).
 * stats != NULL: adds per-channel sum / sum of squares of the stored values to stats[0][.] /
 * stats[1][.] (train-mode BatchNorm, stdcnet.py:10,14).  tune: 0 = automatic tile, else the packed word of the
 * tuned table: BN | (sub-tiles << 12) | (pipeline stages << 16) | bit 20 persistent one-CTA kernel | bit 21 resident
 * filter | bit 22 CTA-pair kernel (cta_group::2) | bit 23 input-halo reuse | bits 24-26 K-blocks per stage / taps per
 * filter-ring slot | bit 27 epilogue stores from registers | bit 28 epilogue TMA stores at any tile width.
 * mask (optional, bf16 NHWC view shaped like the output): the result is multiplied by
 * LeakyReLU'(mask) = (mask > 0 ? 1 : mask_slope) -- the backward of the discriminators' biased
 * conv + LeakyReLU layers (discriminator.py:17-26) folded into the data-gradient launch that produces
 * the layer's output gradient; with stats_sum_only = 1 the statistics path then returns only
 * stats[0][c] = sum over pixels = that layer's bias gradient (stats[1] is left untouched). */
int b200_conv_igemm(const void* in, int in_ld, int in_coff, int in_C, int N, int Hin, int Win,
                    const void* filt, int filt_rows, int cin_pad, int n_slabs, void* out, int out_ld,
                    int out_coff, int Hout, int Wout, int out_f32, int n_classes, const int* class_Ho,
                    const int* class_Wo, const int* class_oa, const int* class_ob,
                    const int* class_ntaps, const int* taps, int taps_stride, int in_stride,
                    int out_stride, const float* bias, int act, float slope, float* stats,
                    int stats_ld, const void* mask, int mask_ld, float mask_slope, int stats_sum_only,
                    int tune, cudaStream_t stream);

/* Diagnostic: buf != NULL (device int64 [8 + 4*30]) makes CTA pair 0 of every following CTA-pair conv launch
 * record %globaltimer at its phase boundaries (kernel entry, set-up done, first operands landed, exit; per
 * tile: MMAs start / committed / epilogue starts / done) -- scripts/pair_timeline.py prints them.  NULL
 * (the default) turns it off; never set on a production path. */
int b200_debug_timeline(int64_t* buf);
/* Diagnostic: switches parts of the CTA-pair kernel's epilogue off for timing experiments (bit 0: no global
 * stores, bit 1: no TMEM loads, bit 2: no BatchNorm statistics).  Results are WRONG while it is non-zero;
 * 0 (the default) is the only value a production path may see. */
int b200_debug_knob(int knob);

/* Weight gradient dW[Cout][Cin][RS] (fp32, PyTorch layout, accumulated) of the same convolutions:
 * dW[co][ci][rs] += sum_pixels dz[pixel, co] * x[pixel*stride + tap, ci]; taps = [n_taps][3] = (dh, dw, rs).
 * tune: 0 = automatic, else ci-tile | (stages << 12) | (pixel splits << 16) | (K pixels / 64 << 28). */
int b200_conv_wgrad(const void* dz, int dz_ld, int dz_coff, int Cout, int N, int Ho, int Wo,
                    const void* x, int x_ld, int x_coff, int Cin, int Hin, int Win, int n_taps,
                    const int* taps, int RS, int in_stride, float* dw, float* scratch, int ci_pad, int tune,
                    cudaStream_t stream);
/* scratch (optional, Cin > 32): zeroed fp32 [RS][Cout][ci_pad], ci_pad = round_up(Cin, 16).  The split-K
 * partial sums are then accumulated there with 16-byte vector reductions (tap-major layout: a
 * thread's 16 input channels are contiguous) and dw is NOT touched; b200_wgrad_unscratch afterwards
 * writes dw[co][ci][rs] = scratch[rs][co][ci] for all layers of a module backward in one launch
 * (table_dev: int64 [n_layers][6] = {scratch offset, dw offset in floats from the two base
 * pointers, Cout, Cin, RS, ci_pad}). */
int b200_wgrad_unscratch(const float* scratch_base, float* dw_base, const int64_t* table_dev, int n_layers,
                         cudaStream_t stream);
/* Pair-view weight gradient (see b200_pack_filter): dw[co][c][kh][2b+s] = scratch[kh*2+b][co][s*32+c],
 * scratch = fp32 [8][Cout][64] accumulated by b200_conv_wgrad over the pair view. */
int b200_wgrad_unscratch_pairview(const float* scratch, float* dw, int Cout, int Cin, cudaStream_t stream);

/* Stem ConvX(3, 32, 3, 2) (stdcnet.py:171, 6-15): K = 27 is too thin for a tap-by-tap implicit GEMM,
 * so the fp32 NCHW image is unfolded ONCE into bf16 rows col[n, ho, wo, k], k = ci*9 + r*3 + s
 * (k = 27..31 zero, 64-byte pixels), which fuses the layout and precision conversion; forward and
 * filter gradient are then 1x1 launches of b200_conv_igemm / b200_conv_wgrad on `col` against the
 * filter viewed as [32, 27, 1, 1] (same memory as [32, 3, 3, 3]). */
int b200_stem_im2col(const float* img, int N, int H, int W, void* col, int col_ld, cudaStream_t stream);

/* ------------------------------------------------ BatchNorm / activation passes */
/* nn.BatchNorm2d (+ ReLU / LeakyReLU) of ConvX (stdcnet.py:10-14), ConvBNReLU (model_stages.py:21-29),
 * DepthWiseSepBNFCDiscriminator (discriminator.py:103-131): statistics, finalisation (running-stat
 * update with momentum, unbiased variance), normalise+activate, and the train-mode backward
 * (two passes: reductions for dgamma/dbeta, then dz).  dy2 may be NULL; when given, dy = dy1 + dy2
 * (gradient joins of the bottleneck's concatenation, stdcnet.py:112). */
int b200_channel_stats(const void* x, int ld, int C, int64_t npix, float* stats, cudaStream_t stream);
int b200_bn_finalize(const float* stats, int C, float count, const float* gamma, const float* beta,
                     float* running_mean, float* running_var, float momentum, float eps,
                     int training, float* scale, float* shift, float* mean_out, float* rstd_out,
                     cudaStream_t stream);
int b200_bn_act_apply(const void* x, int x_ld, void* y, int y_ld, int C, int64_t npix,
                      const float* scale, const float* shift, int act, float slope,
                      cudaStream_t stream);
/* b200_bn_finalize + b200_bn_act_apply in one launch (coefficients derived in-kernel; block 0
 * publishes scale/shift/mean/rstd for the backward and updates the running statistics). */
int b200_bn_norm_act(const void* x, int x_ld, void* y, int y_ld, int C, int64_t npix,
                     const float* stats, float count, const float* gamma, const float* beta,
                     float* running_mean, float* running_var, float momentum, float eps,
                     int training, int act, float slope, float* scale, float* shift,
                     float* mean_out, float* rstd_out, cudaStream_t stream);
int b200_bn_act_bwd_reduce(const void* dy1, int dy1_ld, const void* dy2, int dy2_ld, const void* z,
                           int z_ld, int C, int64_t npix, const float* scale, const float* shift,
                           const float* mean, const float* rstd, int act, float slope, float* red,
                           cudaStream_t stream);
int b200_bn_act_bwd_apply(const void* dy1, int dy1_ld, const void* dy2, int dy2_ld, const void* z,
                          int z_ld, void* dz, int dz_ld, int C, int64_t npix, const float* scale,
                          const float* shift, const float* mean, const float* rstd,
                          const float* red, float inv_count, int act, float slope,
                          cudaStream_t stream);
/* reduce + apply in one cooperative launch (grid-wide barrier in between).  `red` is float
 * [1 + 8][2][C], zeroed by the caller: [0] receives the totals (dbeta = red[0][0][c], dgamma =
 * red[0][1][c]), [1..8] are partial-sum replicas (same-address atomics serialise in L2). */
int b200_bn_act_bwd_fused(const void* dy1, int dy1_ld, const void* dy2, int dy2_ld, const void* z,
                          int z_ld, void* dz, int dz_ld, int C, int64_t npix, const float* scale,
                          const float* shift, const float* mean, const float* rstd, float* red,
                          float inv_count, int act, float slope, cudaStream_t stream);
/* LeakyReLU backward + bias gradient of the biased discriminator convs (discriminator.py:18-25). */
int b200_act_bwd_bias(const void* dy1, int dy1_ld, const void* dy2, int dy2_ld, const void* a,
                      int a_ld, void* dz, int dz_ld, int C, int64_t npix, int act, float slope,
                      float* dbias, cudaStream_t stream);
int b200_cast_f32_bf16(const float* x, void* y, int64_t count, cudaStream_t stream);

/* ---------------------------------------------------- depthwise convolutions */
/* Depthwise K x K (K = 3 or 4), stride 2, pad 1: avd_layer of the bottlenecks (stdcnet.py:24-28,73-77,
 * bias-free, optionally fused with the AvgPool2d(3,2,1) skip of stdcnet.py:78,108-109) and conv*_d of
 * the depthwise-separable discriminators (discriminator.py:35-45, with bias).  w: [C][K*K]. */
int b200_dwconv_s2_fwd(const void* x, int x_ld, int N, int H, int W, int C, int K, const float* w,
                       const float* bias, void* z, int z_ld, void* pool, int pool_ld, int act,
                       float slope, float* stats, cudaStream_t stream);
int b200_dwconv_s2_dgrad(const void* dz, int dz_ld, const void* dpool, int dpool_ld, int N, int H,
                         int W, int C, int K, const float* w, void* dx, int dx_ld,
                         cudaStream_t stream);
int b200_dwconv_s2_wgrad(const void* dz, int dz_ld, const void* x, int x_ld, int N, int H, int W,
                         int C, int K, float* dw, float* dbias, cudaStream_t stream);

/* ------------------------------------------------------ global-pool attention */
/* F.avg_pool2d(feat, feat.size()[2:]) numerator (model_stages.py:79,120,178): out[n][c] += sum_hw x. */
int b200_pool_sum(const void* x, int ld, int N, int HW, int C, float* out, cudaStream_t stream);
/* 1x1 conv on the pooled [N, C] vector (+BatchNorm over the batch) + activation: conv_atten+bn_atten+
 * sigmoid (model_stages.py:80-82), conv_avg (120-122), FFM conv1/relu/conv2/sigmoid (179-182). */
int b200_fc_small_fwd(const float* in, float in_scale, int N, int Cin, int Co, const float* W,
                      int has_bn, const float* gamma, const float* beta, float* running_mean,
                      float* running_var, float momentum, float eps, int training, int act,
                      float* pre, float* out, float* mean_out, float* rstd_out, cudaStream_t stream);
int b200_fc_small_bwd(const float* dout, const float* out, const float* pre, const float* in,
                      float in_scale, int N, int Cin, int Co, const float* W, int has_bn,
                      int training, const float* gamma, const float* mean, const float* rstd,
                      int act, float* dpre_scratch, float* dW, float* dgamma, float* dbeta,
                      float* din, int accumulate_din, cudaStream_t stream);
/* out[n,ho,wo,c] = a[n,hs,ws,c] * (s[n,c] + s_plus) + v[n,c]*v_scale + t[n,hs,ws,c], (hs,ws) = nearest
 * source of (ho,wo): torch.mul(feat, atten) (model_stages.py:84), "+ avg_up" / "+ feat32_up" and the
 * nearest F.interpolate (123,126-127,131-132), feat*atten + feat (183-184).  s, v, t may be NULL. */
int b200_scale_add_bcast(const void* a, int a_ld, int Hs, int Ws, const float* s, float s_plus,
                         const float* v, float v_scale, const void* t, int t_ld, void* out,
                         int out_ld, int N, int Ho, int Wo, int C, cudaStream_t stream);
/* backward of the above: footprint sum of dout per source pixel (dsum), dot[n][c] += sum dsum*b,
 * vsum[n][c] += sum dsum. */
int b200_upsum_dot_reduce(const void* dout, int dout_ld, int Ho, int Wo, const void* b, int b_ld,
                          void* dsum, int dsum_ld, int N, int Hs, int Ws, int C, float* dot,
                          float* vsum, cudaStream_t stream);

/* ------------------------------------ bilinear up-sampling fused with its users */
/* F.interpolate(x, (H, W), mode='bilinear', align_corners=True) of the class logits
 * (model_stages.py:240-242) fused with: mode 0 nothing (NCHW logits out), mode 1
 * CrossEntropyLoss(ignore_index=255) (train.py:66,86-89,214-217; acc[0] += sum, acc[1] += #valid;
 * optional per-pixel loss map for OHEM), mode 2 F.softmax(dim=1) (train.py:230,248,257; bf16 NHWC out),
 * mode 3 argmax (utils.py:120-121).  lr: fp32 NHWC low-resolution logits, pixel stride lr_ld.
 * n_classes: 2..32, each count its own compiled instance (B200_EINVAL otherwise).  lr_ld must be a
 * multiple of 4 and >= round_up(n_classes, 4); no float of a pixel beyond round_up(n_classes, 4) is read.
 * mode 2 with out_flag == 2 (forward) / grad_is_bf16 == 2 (backward): the probability map (its gradient) is
 * the zero-bordered [N][H+2][W+2][p_ld] layout -- Conv2d's padding=1 materialised -- that the dense
 * discriminator's first layer reads as 128-byte column pairs (discriminator.py:9,18); the forward writes
 * the border zeros, the backward ignores the border. */
int b200_upsample_fwd(const float* lr, int lr_ld, int N, int h_lr, int w_lr, int H, int W,
                      int n_classes, int mode, void* out, int out_flag, int p_ld,
                      const int64_t* labels, int ignore_index, double* acc, float* loss_map,
                      cudaStream_t stream);
int b200_upsample_bwd(const float* lr, int lr_ld, int N, int h_lr, int w_lr, int H, int W,
                      int n_classes, int mode, const void* grad_in, int grad_is_bf16, int p_ld,
                      const int64_t* labels, int ignore_index, const float* pixel_weight,
                      const float* coef_num, const double* coef_den, float coef_scale, float* d_lr,
                      double* loss_acc, cudaStream_t stream);
/* loss_acc != NULL (mode 1): the same pass also accumulates the forward loss sum / valid count, so a
 * training step needs no separate forward kernel; b200_scale_f32 then applies grad_out / #valid. */
int b200_scale_f32(const float* x, int64_t count, const float* num, const double* den, float mul,
                   float* y, cudaStream_t stream);
/* OHEM_CrossEntroy_Loss (utils.py:263-271) without torch.sort: k-th largest by radix select over the
 * fp32 bit patterns, then the thresholded / top-k mean and the per-pixel gradient weights. */
int b200_radix_select_desc(const float* x, int64_t count, int64_t rank, uint32_t* state,
                           uint32_t* hist, cudaStream_t stream);
int b200_ohem_reduce(const float* x, int64_t count, const uint32_t* state, float threshold,
                     int64_t keep_num, double* sums, float* out, cudaStream_t stream);
int b200_ohem_weights(const float* x, int64_t count, const float* sel, float* wout,
                      cudaStream_t stream);
/* BCEWithLogitsLoss against torch.zeros / torch.ones (train.py:173,231-232,249-250,258). */
int b200_bce_const_fwd(const float* x, int count, float target, float* out, cudaStream_t stream);
int b200_bce_const_bwd(const float* x, int count, float target, const float* gscale, float gmul,
                       float* dx, cudaStream_t stream);

/* ------------------------------------------------- discriminator classifier */
/* Conv2d(512, 1, 4, 2, 1) (discriminator.py:13,26,47,72,97,132): forward, data and filter gradients. */
int b200_classifier_fwd(const void* x, int x_ld, int N, int H, int W, int C, const float* w,
                        const float* bias, float* out, cudaStream_t stream);
int b200_classifier_dgrad(const float* dout, int N, int H, int W, int C, const float* w, void* dx,
                          int dx_ld, cudaStream_t stream);
int b200_classifier_wgrad(const float* dout, const void* x, int x_ld, int N, int H, int W, int C,
                          float* dw, float* dbias, cudaStream_t stream);

/* ------------------------------------------------------------------ metrics */
/* fast_hist(a = label, b = pred, n) (utils.py:161-167, called at train.py:47): hist[n*a+b] += 1 for
 * 0 <= a < n, int64, accumulated.  *_bytes: element size of the arrays (8 = int64 as in the reference,
 * 4, 1).  *bad is set to 1 if an index falls outside [0, n*n) (numpy would fail the reshape). */
int b200_fast_hist(const void* label, int label_bytes, const void* pred, int pred_bytes,
                   int64_t count, int n, int64_t* hist, int* bad, cudaStream_t stream);
/* compute_global_accuracy numerator (utils.py:151-159): *out += #(pred == label). */
int b200_count_equal(const void* label, int label_bytes, const void* pred, int pred_bytes,
                     int64_t count, int64_t* out, cudaStream_t stream);
/* The same per image, for the evaluation loop (train.py:50,56: precision = mean of the per-image
 * ratios): out[i] += #(pred == label) over image i's `per_image` positions; label/pred hold n_images
 * images back to back.  Element sizes 8/8, 8/1 or 1/1. */
int b200_count_equal_batched(const void* label, int label_bytes, const void* pred, int pred_bytes,
                             int n_images, int64_t per_image, int64_t* out, cudaStream_t stream);

/* ------------------------------------------------------------------ collectives (NCCL) */
/* The two exchange steps of the data-parallel path for callers that do not use torch.distributed
 * (the Python host of this repository does, and never calls these): one process per GPU, NCCL over
 * NVLink.  NCCL is dlopen'ed ("libnccl.so.2") at the first call; B200_EDRIVER when it is absent.
 *   unique_id : rank 0 creates the 128-byte id and hands it to the other ranks out of band
 *   init      : ncclCommInitRank on the calling thread's current device -> opaque communicator
 *   allreduce_grads : in-place sum (average != 0: mean) of a flat fp32 gradient bucket over the ranks
 *                     (the reference's nn.DataParallel gradient reduce, train.py:145-152,497)
 *   allreduce_hist  : in-place int64 sum of the n*n confusion matrix (train.py:47 over a sharded loader;
 *                     exact, so the result is bit-identical to a single-process evaluation) */
int b200_nccl_unique_id(void* id128);
int b200_nccl_init(const void* id128, int world, int rank, void** comm_out);
int b200_nccl_allreduce_grads(void* comm, float* flat, int64_t count, int average, cudaStream_t stream);
int b200_nccl_allreduce_hist(void* comm, int64_t* hist, int count, cudaStream_t stream);
int b200_nccl_destroy(void* comm);

/* ------------------------------------------------------------------ input pipeline */
/* pil_loader(path).resize(size, Image.BILINEAR) -> ToTensor() -> Normalize(mean, std)
 * (dataset/cityscapes.py:65,67 and dataset/GTAV.py:85,87; Pillow Resample.c two-pass 8-bit resample).
 * src: decoded uint8 RGB [N, H0, W0, 3].  xb / yb: int32 [W or H][2] = (first source index, tap count)
 * per output column / row; xk / yk: int32 fixed-point (22 fractional bits) coefficients [W][kx] /
 * [H][ky] (the host restates Pillow's precompute_coeffs in float64).  The horizontal pass rounds to
 * uint8 before the vertical pass exactly as Pillow does.  lut: float [3][256] = ((v/255) - mean_c) /
 * std_c in fp32.  dst: fp32 NCHW [N, 3, H, W].  max_rows: the largest number of source rows one band
 * of 8 output rows touches (sizes the shared-memory staging).  Bit-exact with the reference. */
int b200_image_resize_normalize(const uint8_t* src, int N, int H0, int W0, const int32_t* xb,
                                const int32_t* xk, int kx, const int32_t* yb, const int32_t* yk, int ky,
                                int H, int W, const float* lut, float* dst, int max_rows,
                                cudaStream_t stream);
/* Image.open(path).resize(size, Image.NEAREST) -> PILToTensor() [-> GtaV.convert_labels]
 * (cityscapes.py:66,68; GTAV.py:86,88-89,97-100; Pillow Geometry.c ImagingScaleAffine).
 * src: uint8 [N, H0, W0]; ix / iy: int32 source column / row per output column / row; lut: uint8[256]
 * label remap (identity for Cityscapes); dst: uint8 or int64 [N, H, W]. */
int b200_label_resize_remap(const uint8_t* src, int N, int H0, int W0, const int32_t* ix, const int32_t* iy,
                            int H, int W, const uint8_t* lut, void* dst, int dst_is_i64,
                            cudaStream_t stream);

/* ------------------------------------------------------------------ optimizers */
/* One launch = one optimizer.step() over every parameter tensor (train.py:170-172, 219-221, 235-237,
 * 252-254, 260-262): torch.optim.SGD (momentum, dampening, L2 weight decay, nesterov) and
 * torch.optim.Adam (bias-corrected, L2 weight decay, no amsgrad).
 * table_dev: int64 [n_tensors][8] = {param*, grad*, state1* (momentum buffer / exp_avg, 0 = none),
 *   state2* (exp_avg_sq), numel, first chunk (prefix sum of ceil(numel / b200_optim_chunk())),
 *   hyper-parameter group, flags (bit 0: momentum buffer already initialised)}; all fp32.
 * hyper_dev: float [n_groups][8] = {lr, momentum, dampening, weight_decay, nesterov, beta1, beta2, eps}.
 * counters_dev (Adam): int64[2] = {step count, 0}; the kernel advances the step itself, so a captured
 * graph replays correctly. */
int b200_sgd_step(const int64_t* table_dev, int n_tensors, int total_chunks, const float* hyper_dev,
                  cudaStream_t stream);
int b200_adam_step(const int64_t* table_dev, int n_tensors, int total_chunks, const float* hyper_dev,
                   int64_t* counters_dev, cudaStream_t stream);
int b200_optim_chunk(void);

#ifdef __cplusplus
}
#endif
#endif /* B200SEG_H_ */
