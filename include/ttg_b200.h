/* ttg_b200.h — C ABI of libttg_b200.so: the hand-written sm_100a kernels behind
 * tartangan's GAN training step (SA-GAN / SA-GAN-IQN generator + discriminator,
 * forward, backward and the double-backward the R1 penalty needs).
 *
 * tartangan has no FFI of its own: every arithmetic op on its hot path is an ATen
 * library call made from Python (SURVEY.md §2.2).  Each entry point below therefore
 * cites the reference call site (file:line under /root/reference/tartangan) whose
 * ATen op(s) it replaces.  INTEGRATION.md shows the ctypes binding a maintainer of
 * the reference would add.
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer owned by the caller
 *     (PyTorch allocates inputs, outputs and workspaces; kernels never allocate,
 *     never retain pointers past return);
 *   - activations are NHWC ("channels last"), element type given by a dtype code:
 *     TTG_F32 = 0, TTG_BF16 = 1; parameters, statistics and losses are fp32;
 *   - `stream` is a cudaStream_t passed as void*; every launch goes to it, nothing
 *     synchronises, so all entry points are CUDA-graph capturable and re-entrant;
 *   - return 0 on success, non-zero on error; ttg_last_error() gives the
 *     thread-local message.  Unsupported shapes are errors, never fallbacks.
 */
#ifndef TTG_B200_H
#define TTG_B200_H
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

const char* ttg_last_error(void);
int ttg_version(void);
int ttg_device_arch(void);

/* ---- convolution: nn.Conv2d k in {1,3}, stride 1, pad k/2
 * (models/blocks/generator.py:41,44,52,124; discriminator.py:17,63,66,78; attention.py:14-17)
 * ttg_pack_weight_direct: OIHW fp32 -> [tap][Cin][Cout] (mode 0, fprop) or the flipped,
 * transposed filter [tap][Cout][Cin] (mode 1, dgrad = fprop with swapped channel roles).
 * ttg_conv2d_direct: exact fp32-accumulate CUDA-core path (fp32 parity mode, RGB layers).
 * `up`=1 folds F.interpolate(scale_factor=2, mode='nearest') (generator.py:58) into the
 * input addressing: x is [N, H/2, W/2, Cin]. */
int ttg_pack_weight_direct(const float* w, float* wp, int Cout, int Cin, int ksize, int mode, void* stream);
int ttg_conv2d_direct(const void* x, const float* wp, const float* bias, void* y, int N, int H, int W, int Cin,
                      int Cout, int ksize, int up, int dtype_in, int dtype_out, void* stream);
int ttg_conv2d_wgrad_direct(const void* x, const void* gy, float* gw, int N, int H, int W, int Cin, int Cout,
                            int ksize, int up, int dtype_x, int dtype_gy, void* stream);
/* same, bitwise repeatable: every split of the pixel range writes its partial sums to its own slab of `workspace`
 * (ttg_conv2d_wgrad_direct_workspace_bytes) and the slabs are added in a fixed order — the reference's CPU
 * convolution_backward is run-to-run deterministic (SURVEY 8c) and so is the fp32 parity path. */
size_t ttg_conv2d_wgrad_direct_workspace_bytes(int N, int H, int W, int Cin, int Cout, int ksize);
int ttg_conv2d_wgrad_direct_det(const void* x, const void* gy, float* gw, int N, int H, int W, int Cin, int Cout,
                                int ksize, int up, int dtype_x, int dtype_gy, void* workspace, void* stream);

/* ---- tensor-core convolution (bf16 operands, fp32 accumulate in TMEM, tcgen05.mma)
 * same reference call sites as above; Cin, Cout multiples of 16, stride 1, no fused upsample: the
 * generator's nearest x2 upsample (generator.py:58) is materialised by ttg_upsample2 first, so that the
 * activation tiles of fprop, dgrad and wgrad are all fetched with tensor-map (TMA) loads.  The CUDA driver must
 * provide cuTensorMapEncodeTiled; otherwise these entry points return an error.
 * ttg_pack_weight_tc: OIHW fp32 -> bf16 UMMA B-operand image, mode 0 fprop / 1 dgrad.
 * ttg_conv2d_tc: y = conv(x) (+bias), y bf16 or fp32 (dtype_out).
 * ttg_conv2d_wgrad_tc: gw (fp32 OIHW) = sum_pixels gy x shifted(x). */
size_t ttg_pack_weight_tc_bytes(int Cout, int Cin, int ksize);
int ttg_pack_weight_tc(const float* w, void* wp, int Cout, int Cin, int ksize, int mode, void* stream);
int ttg_conv2d_tc(const void* x, const void* wp, const float* bias, void* y, int N, int H, int W, int Cin, int Cout,
                  int ksize, int dtype_out, void* stream);
/* channel-padded variants: Cin/Cout are the padded GEMM sizes (16), cin_real/cout_real the channel counts in memory
 * (RGB layers: Cin == 3 first D conv discriminator.py:63, Cout == 3 image gradient / generator.py:124).
 * ttg_conv2d_tc_ex also accepts other narrow tensors (<= 8 input channels; <= 16 output channels when Cout == 16),
 * read / written with scalar accesses; the wgrad entry points accept only the 8-channel staging tensors below. */
int ttg_pack_weight_tc_pad(const float* w, void* wp, int Cout, int Cin, int CoutP, int CinP, int ksize, int mode,
                           void* stream);
int ttg_conv2d_tc_ex(const void* x, const void* wp, const float* bias, void* y, int N, int H, int W, int Cin, int Cout,
                     int cin_real, int cout_real, int ksize, int dtype_out, void* stream);
int ttg_conv2d_wgrad_tc_ex(const void* x, const void* gy, float* gw, int N, int H, int W, int Cin, int Cout,
                           int cin_real, int cout_real, int ksize, void* workspace, void* stream);
/* 8-channel staging copies of the <= 8-channel (RGB) bf16 tensors: y8[p][0..7] = x[p][0..c_real-1], 0...  With
 * cin_real / cout_real == 8 (Cin / Cout == 16) the _ex entry points above read / write such tensors through the
 * same TMA tiles and 16-byte stores as the wide layers (missing channel groups are zero-filled by the TMA engine). */
/* conv (bf16 NHWC, channels multiples of 16) that also returns the BatchNorm statistics of its output:
 * sums[0..Cout) = sum over pixels, sums[Cout..2Cout) = sum of squares (fp64; of the bf16 values written).  Replaces the
 * first pass of native_batch_norm over the conv output (conv -> BatchNorm2d pairs: generator.py:41-43,
 * discriminator.py:63-65).  ttg_bn_finalize turns the sums into mean / invstd / running statistics. */
int ttg_conv2d_tc_stats_supported(int Cin, int Cout, int ksize);
int ttg_conv2d_tc_stats(const void* x, const void* wp, const float* bias, void* y, int N, int H, int W, int Cin, int Cout,
                        int ksize, double* sums, void* stream);
/* every conv filter of a model (views of one flat fp32 parameter buffer) packed in one launch; table rows of 9
 * int64 {src offset (floats), dst offset (bytes), Cout, Cin, CoutP, CinP, ksize, mode, first block}, 256 threads per
 * block, one element per thread; padded destination images must have been zeroed once. */
int ttg_pack_weights_multi(const float* flat, void* packed, const long long* table, int n_entries, int total_blocks,
                           void* stream);
int ttg_pad_channels8(const void* x, void* y8, long long npix, int c_real, void* stream);
int ttg_unpad_channels8(const void* y8, void* y, long long npix, int c_real, void* stream);
/* wgrad + bias gradient gbias[co] = sum_pixels gy (fp32) in ONE pass over gy (both halves of convolution_backward's
 * parameter gradients, nn.Conv2d(bias=True): generator.py:41,44, discriminator.py:63,66) */
int ttg_conv2d_wgrad_bias_tc_ex(const void* x, const void* gy, float* gw, float* gbias, int N, int H, int W, int Cin,
                                int Cout, int cin_real, int cout_real, int ksize, void* workspace, void* stream);
int ttg_conv2d_wgrad_tc(const void* x, const void* gy, float* gw, int N, int H, int W, int Cin, int Cout, int ksize,
                        void* workspace, void* stream);
size_t ttg_conv2d_wgrad_tc_workspace_bytes(int Cin, int Cout, int ksize);

/* ---- train-mode BatchNorm2d fused with LeakyReLU
 * (nn.BatchNorm2d + nn.LeakyReLU(0.2) pairs: generator.py:38-43,120-122;
 *  discriminator.py:60-65,132-135,153-156; eps 1e-5, momentum 0.1, unbiased running var)
 * workspace: ttg_bn_workspace_bytes(C) bytes. */
size_t ttg_bn_workspace_bytes(int C);
int ttg_bn_stats(const void* x, long long M, int C, float eps, float momentum, float* mean, float* invstd,
                 float* running_mean, float* running_var, long long* num_batches, void* workspace,
                 long long count_mult, int dtype, void* stream);
int ttg_bn_finalize(const double* sums, long long M, int C, float eps, float momentum, float* mean, float* invstd,
                    float* running_mean, float* running_var, long long* num_batches, long long count_mult, void* stream);
int ttg_bn_eval_stats(const float* running_mean, const float* running_var, float eps, int C, float* mean,
                      float* invstd, void* stream);
int ttg_bn_act_fwd(const void* x, void* y, long long M, int C, const float* mean, const float* invstd,
                   const float* gamma, const float* beta, float slope, int dtype, void* stream);
/* statistics finalisation + apply in one launch: sums = {sum x, sum x^2} (fp64 [2C]) from the kernel that produced x
 * (ttg_conv2d_tc_stats, ttg_add_up2_stats, ...) or NULL (then they are reduced into `workspace` first); writes y,
 * mean / invstd (for backward) and updates running_mean / running_var / num_batches like ttg_bn_stats. */
int ttg_bn_act_fwd_stats(const void* x, void* y, long long M, int C, const double* sums, const float* gamma,
                         const float* beta, float eps, float momentum, float slope, float* mean, float* invstd,
                         float* running_mean, float* running_var, long long* num_batches, long long count_mult,
                         void* workspace, int dtype, void* stream);
int ttg_bn_act_bwd(const void* x, const void* ga, void* gx, long long M, int C, const float* mean,
                   const float* invstd, const float* gamma, const float* beta, float slope, float* ggamma,
                   float* gbeta, void* workspace, int dtype, void* stream);
/* backward of ttg_bn_act_bwd w.r.t. (ga, x, gamma) given u = cotangent of gx: the
 * NativeBatchNormBackwardBackward0 nodes created by models/losses.py:23-26. */
int ttg_bn_act_bwd2(const void* x, const void* ga, const void* u, void* g_ga, void* g_x, long long M, int C,
                    const float* mean, const float* invstd, const float* gamma, const float* beta, float slope,
                    float* ggamma, void* workspace, int dtype, void* stream);
int ttg_lrelu_fwd(const void* x, void* y, long long n, float slope, int dtype, void* stream);
int ttg_lrelu_bwd(const void* x, const void* g, void* gx, long long n, float slope, int dtype, void* stream);
/* nn.ELU / nn.SELU (--activation elu|selu: trainers/cnn.py:41-45, trainers/iqn.py:42-45):
 * f(x) = scale * (x > 0 ? x : alpha * (exp(x) - 1)).  _bwd: gx = g * f'(x);  _bwd2: out = g * u * f''(x), the cotangent
 * of x through _bwd that the R1 penalty (models/losses.py:23-26) needs. */
int ttg_elu_fwd(const void* x, void* y, long long n, float alpha, float scale, int dtype, void* stream);
int ttg_elu_bwd(const void* x, const void* g, void* gx, long long n, float alpha, float scale, int dtype, void* stream);
int ttg_elu_bwd2(const void* x, const void* g, const void* u, void* out, long long n, float alpha, float scale, int dtype,
                 void* stream);
/* conv bias gradient: out[c] = sum over rows of x[M,C] */
int ttg_channel_sum(const void* x, long long M, int C, float* out, void* workspace, int dtype, void* stream);

/* ---- parameter gradients accumulated in place (torch::autograd::AccumulateGrad, i.e. `param.grad += g` after
 * loss.backward() in trainers/cnn.py:134,150 and iqn.py:128,139): the `_acc` variants ADD the parameter gradient to the
 * caller's buffer (a view of the model's flat .grad buffer) instead of returning a fresh tensor that autograd then adds
 * with one more kernel per parameter.  `accumulate` / `flags`: bit 0 = add to the gradient buffers (0 gives the plain
 * behaviour of the entry point without suffix; ttg_conv2d_wgrad_tc_acc always accumulates), bit 1 = the caller
 * guarantees that `workspace` is all zero already (one clear per training step instead of one memset per call). */
int ttg_conv2d_wgrad_tc_acc(const void* x, const void* gy, float* gw, float* gbias, int N, int H, int W, int Cin, int Cout,
                            int cin_real, int cout_real, int ksize, int flags, void* workspace, void* stream);
int ttg_bn_act_bwd_acc(const void* x, const void* ga, void* gx, long long M, int C, const float* mean,
                       const float* invstd, const float* gamma, const float* beta, float slope, float* ggamma,
                       float* gbeta, int accumulate, void* workspace, int dtype, void* stream);
int ttg_bn_act_bwd2_acc(const void* x, const void* ga, const void* u, void* g_ga, void* g_x, long long M, int C,
                        const float* mean, const float* invstd, const float* gamma, const float* beta, float slope,
                        float* ggamma, int accumulate, void* workspace, int dtype, void* stream);
int ttg_channel_sum_acc(const void* x, long long M, int C, float* out, int accumulate, void* workspace, int dtype,
                        void* stream);

/* ---- train-mode BatchNorm + LeakyReLU with the fp64 channel sums exposed between the reduce and the apply pass, so
 * that a caller can all-reduce them over the ranks of a data-parallel job (synchronised BatchNorm, --sync-bn).
 * M: rows this call walks; count: pixel count the sums were taken over (world * M for equal shards; count == M is
 * what the combined entry points above compute, bit for bit).  flags / accumulate as above.  param_scale multiplies the
 * gamma / beta gradients (1 / world: the gradient all-reduce adds every rank's copy of the global value).
 *   ttg_bn_sums: sums[2C] = {sum x, sum x^2}
 *   ttg_bn_act_fwd_stats_n: ttg_bn_act_fwd_stats with statistics and running-variance correction over count
 *   ttg_bn_act_bwd_reduce / _apply: ttg_bn_act_bwd_acc, sums[2C]; _apply with gx NULL writes the parameter gradients only
 *   ttg_bn_act_bwd2_reduce / _apply: ttg_bn_act_bwd2_acc, sums[5C] */
int ttg_bn_sums(const void* x, long long M, int C, double* sums, int flags, int dtype, void* stream);
int ttg_bn_act_fwd_stats_n(const void* x, void* y, long long M, int C, long long count, const double* sums,
                           const float* gamma, const float* beta, float eps, float momentum, float slope, float* mean,
                           float* invstd, float* running_mean, float* running_var, long long* num_batches,
                           long long count_mult, void* workspace, int dtype, void* stream);
int ttg_bn_act_bwd_reduce(const void* x, const void* ga, long long M, int C, const float* mean, const float* invstd,
                          const float* gamma, const float* beta, float slope, double* sums, int flags, int dtype,
                          void* stream);
int ttg_bn_act_bwd_apply(const void* x, const void* ga, void* gx, long long M, int C, long long count, const double* sums,
                         const float* mean, const float* invstd, const float* gamma, const float* beta, float slope,
                         float* ggamma, float* gbeta, float param_scale, int accumulate, int dtype, void* stream);
int ttg_bn_act_bwd2_reduce(const void* x, const void* ga, const void* u, long long M, int C, const float* mean,
                           const float* invstd, const float* gamma, const float* beta, float slope, double* sums,
                           int flags, int dtype, void* stream);
int ttg_bn_act_bwd2_apply(const void* x, const void* ga, const void* u, void* g_ga, void* g_x, long long M, int C,
                          long long count, const double* sums, const float* mean, const float* invstd,
                          const float* gamma, const float* beta, float slope, float* ggamma, float param_scale,
                          int accumulate, int dtype, void* stream);

/* ---- resampling / glue
 * pool2_sum: nn.AvgPool2d(2) with scale 0.25 (discriminator.py:67); adjoint of upsample2.
 * upsample2: F.interpolate nearest x2 (generator.py:58); adjoint of pool2_sum.
 * bilinear_down_*: F.interpolate(scale_factor=0.5, mode='bilinear', align_corners=True)
 *   (discriminator.py:55-57,92) and its transpose.
 * axpby: residual add x + h (generator.py:62, discriminator.py:95) and gradient accumulation.
 * spatial_sum/bcast: torch.sum(feats, [2,3]) (discriminator.py:143,166) and its adjoint. */
int ttg_pool2_sum(const void* x, void* y, int N, int Ho, int Wo, int C, float scale, int dtype, void* stream);
int ttg_upsample2(const void* x, void* y, int N, int Hi, int Wi, int C, float scale, int dtype, void* stream);
int ttg_bilinear_down_fwd(const void* x, void* y, int N, int Hi, int Wi, int C, int dtype, void* stream);
int ttg_bilinear_down_bwd(const void* gy, void* gx, int N, int Hi, int Wi, int C, int dtype, void* stream);
/* gx = add + B^T gy: the gradient fan-in at the input of a residual D block (bilinear skip + conv branch,
 * discriminator.py:90-95) in one pass instead of a transposed-bilinear pass plus an add pass */
int ttg_bilinear_down_bwd_add(const void* gy, const void* add, void* gx, int N, int Hi, int Wi, int C, int dtype,
                              void* stream);
/* fused residual joins: h + nearest_up2(skip) (generator.py:58-62) and avg_pool2(h) + skip (discriminator.py:67,95) */
int ttg_add_up2(const void* h, const void* s, void* y, int N, int Ho, int Wo, int C, int dtype, void* stream);
int ttg_pool2_add(const void* h, const void* s, void* y, int N, int Ho, int Wo, int C, float scale, int dtype, void* stream);
/* residual joins that also return the BatchNorm statistics of the tensor they write (sums: double[2C] = sum, sum of
 * squares of the rounded outputs; bf16, C % 8 == 0); the next block starts with nn.BatchNorm2d (generator.py:38,
 * discriminator.py:60, 132, 153) */
int ttg_join_stats_supported(int C);
int ttg_add_up2_stats(const void* h, const void* s, void* y, int N, int Ho, int Wo, int C, double* sums, int dtype, void* stream);
int ttg_pool2_add_stats(const void* h, const void* s, void* y, int N, int Ho, int Wo, int C, float scale, double* sums,
                        int dtype, void* stream);
int ttg_axpby(const void* a, const void* b, void* out, long long n, float alpha, float beta, int dtype, void* stream);
int ttg_scale_f32(const float* x, float* out, long long n, float host_scale, const float* dev_scale, void* stream);
int ttg_spatial_sum(const void* x, float* out, int N, int HW, int C, int dtype, void* stream);
int ttg_spatial_bcast(const float* g, void* gx, int N, int HW, int C, int dtype, void* stream);
/* module boundary: reference tensors are fp32 NCHW (trainers/trainer.py:57-61,69-74) */
int ttg_nchw_to_nhwc(const float* x, void* y, int N, int C, int HW, int dtype, void* stream);
int ttg_nhwc_to_nchw(const void* x, float* y, int N, int C, int HW, int dtype, void* stream);
/* Device-side input pipeline (datasets/image_bytes_dataset.py:44-49 + trainers/trainer.py:69-74: random crop of a
 * uint8 HWC image, ToTensor, Normalize(0.5, 0.5)): stack [M][H][W][C] uint8 resident in device memory;
 * out[b][c][y][x] = stack[index[b]][oy[b] + y][ox[b] + x][c] / 127.5 - 1 as fp32 NCHW (nchw_out = 1) or as the
 * NHWC activation tensor (nchw_out = 0, dtype_out).  index / oy / ox: int32 device arrays of length B. */
int ttg_u8_crop_normalize(const unsigned char* stack, const int* index, const int* oy, const int* ox, void* out, int B,
                          int H, int W, int C, int size, int dtype_out, int nchw_out, void* stream);
int ttg_cast(const void* x, int src_dtype, void* y, int dst_dtype, long long n, void* stream);
/* nn.Tanh at the generator output (generator.py:126) */
/* generator head (GeneratorOutput, generator.py:115-129): y = tanh(conv1x1(a, w) + bias) for C -> 3, a bf16 NHWC, y fp32
 * NCHW (the module boundary's layout): one streaming CUDA-core kernel instead of an N = 3 GEMM + tanh + layout pass;
 * _bwd: input gradient (bf16 NHWC), weight and bias gradients (fp32; added to gw / gb when accumulate) in one pass */
int ttg_rgb_head_supported(int Cin, int Cout);
size_t ttg_rgb_head_workspace_bytes(int Cin);
int ttg_rgb_head_fwd(const void* a, const float* w, const float* bias, float* y, int N, int HW, int Cin, void* stream);
int ttg_rgb_head_bwd(const void* a, const float* w, const float* y, const float* g, void* ga, float* gw, float* gb, int N,
                     int HW, int Cin, int accumulate, void* workspace, void* stream);
int ttg_tanh_fwd(const float* x, float* y, long long n, void* stream);
int ttg_tanh_bwd(const float* y, const float* g, float* gx, long long n, void* stream);

/* ---- IQN head + losses
 * ttg_iqn_head_fwd: IQN.forward + CosineQuantileEmbedding.forward + Linear(C->1) + mean over
 *   quantiles (models/iqn.py:41-46,91-103; blocks/discriminator.py:164-175).  rows r = q*B + b.
 * ttg_iqn_head_bwd: gradient of p_tau w.r.t. feats, We, be, wo, bo given g[r].
 * ttg_quantile_huber_*: iqn_loss (models/iqn.py:111-130).
 * ttg_bce_logits_*: nn.BCEWithLogitsLoss (trainers/cnn.py:88,131,147).
 * ttg_sqsum_f32: grad_dout.pow(2).view(B,-1).sum(1).mean() (models/losses.py:27-29), scale=1/B. */
int ttg_iqn_head_fwd(const float* feats, const float* taus, const float* We, const float* be, const float* wo,
                     const float* bo, float* p_tau, float* p_mean, int B, int nq, int C, int E, void* stream);
int ttg_iqn_head_bwd(const float* g, const float* feats, const float* taus, const float* We, const float* be,
                     const float* wo, float* gf, float* gWe, float* gbe, float* gwo, float* gbo, int B, int nq,
                     int C, int E, void* stream);
/* The whole IQN head in ONE forward and ONE backward kernel (blocks/discriminator.py:164-178): embedding + mix +
 * Linear(C->1) (p_tau, rows r = q*B + b), the mean over quantiles p_mean [B] (:174-175) and iqn_loss (:111-130) against
 * target [B] (NULL: no loss).  Backward: cotangents of p_mean and of the loss (either may be NULL) -> gradients of
 * feats, We, be, wo, bo.  C <= 256, E <= 32. */
int ttg_iqn_head_loss_fwd(const float* feats, const float* taus, const float* We, const float* be, const float* wo,
                          const float* bo, const float* target, float* p_tau, float* p_mean, float* loss, int B, int nq,
                          int C, int E, float k, void* stream);
int ttg_iqn_head_loss_bwd(const float* g_pmean, const float* gloss, const float* p_tau, const float* target,
                          const float* feats, const float* taus, const float* We, const float* be, const float* wo,
                          float* gf, float* gWe, float* gbe, float* gwo, float* gbo, int B, int nq, int C, int E, float k,
                          void* stream);
int ttg_quantile_huber_fwd(const float* p_tau, const float* target, const float* taus, float* loss, int B, int nq,
                           float k, void* stream);
int ttg_quantile_huber_bwd(const float* p_tau, const float* target, const float* taus, const float* gloss,
                           float* gp, int B, int nq, float k, void* stream);
int ttg_bce_logits_fwd(const float* x, const float* y, float* loss, int n, void* stream);
int ttg_bce_logits_bwd(const float* x, const float* y, const float* gloss, float* gx, int n, void* stream);
int ttg_sqsum_f32(const float* x, long long n, float scale, float* out, void* workspace, void* stream);
/* nn.Linear (generator.py:71 input MLP, discriminator.py:137 SA-GAN head) and its gradients */
int ttg_matmul_f32(const float* A, const float* B, const float* bias, float* C, int M, int N, int K, int transA,
                   int transB, void* stream);
int ttg_colsum_f32(const float* x, float* out, int M, int N, float scale, void* stream);
int ttg_rowbcast_f32(const float* g, float* out, int M, int N, float scale, void* stream);

/* ---- optimiser
 * torch.optim.Adam(betas=(0,0.999)) (trainers/cnn.py:84-85, iqn.py:84-85) over a flat fp32
 * buffer, with update_target_generator's EMA (cnn.py:158-165) fused in when ema != NULL. */
int ttg_adam_flat(float* p, const float* g, float* m, float* v, float* ema, long long n, float lr, float beta1,
                  float beta2, float eps, float ema_lr, float* step, void* stream);
int ttg_ema_flat(float* target, const float* src, long long n, float lr, void* stream);

/* ---- 2-D self-attention (models/blocks/attention.py:21-35)
 * maxpool2: F.max_pool2d(.,[2,2]) with argmax bookkeeping; attn_*: softmax(theta^T phi) g. */
int ttg_maxpool2_fwd(const void* x, void* y, unsigned char* idx, int N, int Ho, int Wo, int C, int dtype, void* stream);
int ttg_maxpool2_scatter(const void* gy, const unsigned char* idx, void* gx, int N, int Ho, int Wo, int C, int dtype,
                         void* stream);
int ttg_maxpool2_gather(const void* x, const unsigned char* idx, void* y, int N, int Ho, int Wo, int C, int dtype,
                        void* stream);
int ttg_bmm(const void* A, const void* B, void* C, int batch, int M, int N, int K, int transA, int transB, int dtype,
            void* stream);
int ttg_softmax_fwd(const void* x, void* y, long long rows, int cols, int dtype, void* stream);
int ttg_softmax_bwd(const void* y, const void* gy, void* gx, long long rows, int cols, int dtype, void* stream);
/* backward of ttg_softmax_bwd given w = cotangent of gx: cot_gy, cot_y (D-side attention under R1) */
int ttg_softmax_bwd2(const void* y, const void* gy, const void* w, void* cot_gy, void* cot_y, long long rows, int cols,
                     int dtype, void* stream);
/* Fused attention core (attention.py:25-34: beta = softmax(bmm(theta^T, phi), -1); o = bmm(g, beta^T)) on the
 * tensor cores, beta never written to memory.  Per image: q = theta [Nq][dk], k = max-pooled phi [Nk][dk],
 * v = max-pooled g [Nk][dv] (rows = positions, bf16), o [Nq][dv] bf16, lse [Nq] fp32 (row max + log row sum).
 * Supported: Nq % 128 == 0, Nk % 128 == 0, dk in {8, 16}, dv in {32, 64} (C = 64 / 128 of the '256', '512thin'
 * and '512' configs, models/pluggan.py:252-325); ttg_attn_supported() tells, other shapes return an error.
 * ttg_attn_bwd: first-order backward (dq, dk, dv from dout, recomputing beta tile by tile); workspace of
 * ttg_attn_bwd_workspace_bytes() bytes, no initialisation needed. */
int ttg_attn_supported(int Nq, int Nk, int dk, int dv);
int ttg_attn_fwd(const void* q, const void* k, const void* v, void* o, float* lse, int batch, int Nq, int Nk, int dk,
                 int dv, void* stream);
size_t ttg_attn_bwd_workspace_bytes(int batch, int Nq, int dk);
int ttg_attn_bwd(const void* q, const void* k, const void* v, const void* o, const void* dout, const float* lse,
                 void* dq, void* dk_out, void* dv_out, int batch, int Nq, int Nk, int dk, int dv, void* workspace,
                 void* stream);
/* gamma * o (attention.py:35): out = x * (*dev_scale); and the dot product giving d/dgamma */
int ttg_scale_dev(const void* x, void* out, long long n, const float* dev_scale, int dtype, void* stream);
int ttg_dot_f32out(const void* a, const void* b, float* out, long long n, void* workspace, int dtype, void* stream);

/* ---- spectral norm power iteration (torch.nn.utils.spectral_norm semantics; the seam is the
 * conv_factory kwarg of the blocks: generator.py:34, discriminator.py:28,52) */
/* one launch each: a cluster of 8 CTAs, phases separated by cluster barriers, fixed-order sums (bitwise repeatable);
 * workspace: ttg_spectral_norm_workspace_floats(rows, cols) floats (also enough for _sigma and _bwd) */
size_t ttg_spectral_norm_workspace_floats(int rows, int cols);
int ttg_spectral_norm(const float* w, float* u, float* v, float* w_out, float* sigma, int rows, int cols,
                      int n_iter, float eps, void* workspace, void* stream);
int ttg_spectral_norm_sigma(const float* w, const float* u, const float* v, float* w_out, float* sigma, int rows,
                            int cols, void* workspace, void* stream);
/* g_w = (g - dot(g, w_out) * u v^T) / sigma */
int ttg_spectral_norm_bwd(const float* g, const float* w_out, const float* u, const float* v, const float* sigma,
                          float* gw, int rows, int cols, void* workspace, void* stream);

#ifdef __cplusplus
}
#endif
#endif
