/*
 * hpfg_b200 -- C ABI of the B200-native (sm_100a) semi-supervised U-Net training hot path.
 *
 * This is the drop-in boundary for the path the reference reaches through PyTorch:
 *   model/builder.py:29-30 build_model -> model/unet.py:155-175 UNet.forward   (hpfg_unet_forward)
 *   loss.backward() through that module (2017_03_NIPS_Mean-Teacher_ACDC.py:108)  (hpfg_unet_backward)
 *   utils/loss/medloss.py:44-56 Med_Sup_Loss, utils/loss/diceloss.py:155-191 DiceLoss,
 *   the inline consistency / pseudo-label terms of the MT / CPS / UAMT trainers    (hpfg_ssl_loss_*)
 *   utils/utils.py:82-86 update_ema_variables                                      (hpfg_ema_update)
 *   torch.optim.SGD as built by utils/__init__.py:14-16                            (hpfg_sgd_momentum*)
 *   torch.optim.Adam / AdamW as built by utils/__init__.py:13-49 (+ update_ema_variables) (hpfg_adam*)
 *
 * Conventions: plain pointers and sizes only.  Every pointer is a DEVICE pointer unless its name ends in
 * _host.  All work is enqueued on the caller's stream (passed as void* == cudaStream_t); no call
 * synchronises the host except plan create/destroy.  Return value: 0 = ok, non-zero = error code; the
 * message is available from hpfg_last_error() (thread-local).  The caller owns every buffer it passes; a
 * plan owns only its internal workspace.  A plan is re-entrant per handle but not thread-safe per handle.
 * There is NO CPU fallback: on a machine without an sm_100 device every compute entry point fails.
 */
#ifndef HPFG_B200_H
#define HPFG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HPFG_OK 0
#define HPFG_ERR_INVALID 1     /* bad argument                                   */
#define HPFG_ERR_CUDA 2        /* a CUDA runtime / driver call failed            */
#define HPFG_ERR_UNSUPPORTED 3 /* shape / device not supported by this build     */

#define HPFG_PREC_FP32 0 /* fp32 NHWC activations, CUDA-core FMA convs: the 1e-5 check path            */
#define HPFG_PREC_BF16 1 /* bf16 NHWC activations, tcgen05/TMEM implicit-GEMM convs, fp32 accumulation */

#define HPFG_LOSS_SUP 0  /* Med_Sup_Loss on the labeled slices only                                   */
#define HPFG_LOSS_MT 1   /* + w * mean((softmax(s_u)-softmax(t_u))^2)        (Mean-Teacher)           */
#define HPFG_LOSS_CPS 2  /* two nets, cross pseudo supervision                (CPS)                    */
#define HPFG_LOSS_UAMT 3 /* + w * uncertainty-masked softmax-MSE              (UAMT)                   */
#define HPFG_LOSS_ICT 4  /* + w * MSE against a per-sample mix of two teacher softmaxes (hpfg_ict_loss)  */
#define HPFG_LOSS_S4CV 5 /* two nets: Dice-only cross pseudo supervision + teacher MSE (hpfg_s4cv_loss)  */
#define HPFG_LOSS_CUTMIX 6 /* + w * Dice against CutMix-pasted teacher pseudo-labels (HPFG model1, hpfg_cutmix_loss) */

#define HPFG_NUM_BN 18
#define HPFG_NUM_DROPOUT 5

typedef struct hpfg_unet_plan *hpfg_unet_plan_t;

const char *hpfg_last_error(void);
int hpfg_version(void);
/* Number of CUDA kernels this library has launched since load (bench.py's gpu_launches). */
int64_t hpfg_launch_count(void);

/* Optional device timing per kernel category (bench.py's roofline leg): between begin and end every host-side
 * launcher brackets its kernels with CUDA events on the caller's stream; end synchronises and returns the summed
 * milliseconds and call counts for categories {0 tensor-core conv, 1 CUDA-core conv, 2 CUDA-core wgrad, 3 BN /
 * pool / upsample glue, 4 loss, 5 SGD/EMA, 6 weight packing, 7 tensor-core wgrad}: double[8], int64[8] on the host. */
int hpfg_profile_begin(void);
int hpfg_profile_end(double *ms_per_category_host, int64_t *calls_per_category_host);

/* ---- model layout (mirrors model/unet.py state_dict order) -------------------------------------------
 * Flat parameter buffer: the 82 tensors of UNet.named_parameters() in registration order, each in its
 * native PyTorch layout (conv weight OIHW), fp32, back to back.  offsets/sizes: int64[82] in elements.
 * bn_running: fp32 [running_mean(C) | running_var(C)] for each of the 18 BatchNorms in registration order;
 * bn_offsets: int64[18] element offset of each BN's running_mean (running_var follows at +C). */
int hpfg_unet_param_layout(int in_channels, int num_classes, int64_t *offsets_host, int64_t *sizes_host,
                           int64_t *total_host);
int hpfg_unet_bn_layout(int in_channels, int num_classes, int64_t *bn_offsets_host, int64_t *bn_channels_host,
                        int64_t *total_host);

/* ---- plan ------------------------------------------------------------------------------------------- */
int hpfg_unet_plan_create(int batch, int in_channels, int num_classes, int height, int width, int precision,
                          hpfg_unet_plan_t *plan_out);
int hpfg_unet_plan_destroy(hpfg_unet_plan_t plan);
int64_t hpfg_unet_plan_workspace_bytes(hpfg_unet_plan_t plan);
/* ---- exact-global data-parallel mode (SURVEY 8e caveats 1-3) -------------------------------------------------------------
 * Default data parallelism has DDP semantics: every rank normalises BatchNorm, Dice, CE and the consistency mean over ITS shard.
 * In exact-global mode an N-rank step computes what the single-GPU reference computes on the concatenated batch: the library
 * calls `fn(ctx, device_ptr, count, is_double, stream)` -- a SUM all-reduce over the ranks, enqueued in stream order by the host
 * (NCCL through torch.distributed in hpfg_b200/_lib.py) -- on the 2*C BatchNorm sums of every BatchNorm forward and backward
 * (plans with hpfg_unet_plan_set_sync_bn) and on the 128 loss accumulators between the loss reduce and gradient launches
 * (hpfg_ssl_loss_set_global_sums).  Parameter gradients are then SUMMED over the ranks (grad_scale 1, not 1/world). */
int hpfg_set_allreduce_hook(void (*fn)(void *ctx, void *device_ptr, int64_t count, int is_double, void *stream), void *ctx,
                            int world_size);
int hpfg_unet_plan_set_sync_bn(hpfg_unet_plan_t plan, int enabled);
int hpfg_ssl_loss_set_global_sums(int enabled);

/* Cap on the persistent CTAs of this plan's forward convolutions (0 = none: one CTA per SM on all 148 SMs).  A tensor-core
 * convolution CTA owns a whole SM (~200 KB of shared memory, the full register file), so two forwards enqueued on two streams
 * (student | teacher, the two CPS networks) take turns kernel by kernel; with 74 CTAs each they run side by side on disjoint SMs
 * and the latency-bound deep layers overlap (measured +1.8 % Mean-Teacher step throughput, profiles/README.md). */
int hpfg_unet_plan_set_forward_ctas(hpfg_unet_plan_t plan, int ctas);
/* bf16 plans: select the backward schedule.  0 (default; env HPFG_BWD_FUSE=1 flips the default): BatchNorm backward as streaming
 * kernels (two passes + finalize) that materialise the raw gradient; 1: folded into the tensor-core kernels -- the producing
 * data-gradient epilogue stores g = dact*leaky'*dropout' with the two BatchNorm sums, the consuming dgrad / wgrad loaders build
 * draw = scale*g + kb*raw + kd on the fly.  Same results to bf16 rounding; measured slower on B200 (profiles/README.md). */
int hpfg_unet_plan_set_bwd_fusion(hpfg_unet_plan_t plan, int enabled);

/* UNet.forward.  x: fp32 NCHW [batch,in_channels,H,W]; logits: fp32 NCHW [batch,num_classes,H,W].
 * training != 0: BatchNorm uses batch statistics and updates bn_running / bn_counters (+1 each), dropout is
 * active in the five encoder ConvBlocks (p = .05,.1,.2,.3,.5).  Dropout keep-masks come from
 * dropout_masks_host (host array of HPFG_NUM_DROPOUT device pointers to uint8 NCHW keep-masks; a NULL entry
 * or NULL array means "draw with the library's Philox stream keyed by dropout_seed/dropout_offset"; pass
 * no_dropout != 0 to disable dropout entirely while keeping batch-statistics BN).
 * save_for_backward != 0 keeps the activations hpfg_unet_backward needs inside the plan; x itself is NOT copied
 * and must stay valid and unchanged until that backward has been enqueued (the first layer's weight gradient
 * re-reads it). */
int hpfg_unet_forward(hpfg_unet_plan_t plan, const float *params, float *bn_running, int64_t *bn_counters,
                      const float *x, float *logits, int training, int no_dropout, int save_for_backward,
                      uint64_t dropout_seed, uint64_t dropout_offset, const uint8_t *const *dropout_masks_host,
                      void *stream);

/* CUDA-graph friendly variants ("_dv": device values).  Scalars that change every iteration are read from device memory
 * at execution time instead of being baked into the launch, so a captured step can be replayed after updating a small
 * device block: the Philox offset of the dropout masks (hpfg_unet_forward_dv), the consistency weight
 * (hpfg_ssl_loss_dv: utils/utils.py:67-79 ramp-up), {lr, ema_alpha, 1-ema_alpha} (hpfg_sgd_momentum_ema_dv:
 * utils/scheduler/medical_lr.py:13-17, utils/utils.py:84) and the per-step Adam scalars (hpfg_adam_dv). */
int hpfg_unet_forward_dv(hpfg_unet_plan_t plan, const float *params, float *bn_running, int64_t *bn_counters,
                         const float *x, float *logits, int training, int no_dropout, int save_for_backward,
                         uint64_t dropout_seed, const uint64_t *dropout_offset_dev,
                         const uint8_t *const *dropout_masks_host, void *stream);

/* Backward of the last save_for_backward forward on this plan.  dlogits: fp32 NCHW.  grads: flat fp32
 * buffer with the parameter layout; overwritten (accumulate == 0) or added to (accumulate != 0). */
int hpfg_unet_backward(hpfg_unet_plan_t plan, const float *params, const float *dlogits, float *grads,
                       int accumulate, void *stream);

/* UNet_Plus (model/unet.py:178-206, SURVEY 8f.2) needs one tensor from inside the network and sends one gradient back:
 * hpfg_unet_bottleneck copies feature[-1] of the last forward on this plan -- the activated output of the down4 ConvBlock,
 * fp32 NCHW [batch, 256, H/16, W/16] -- for the dense_projection_high neck; hpfg_unet_backward_ex is hpfg_unet_backward
 * with an optional gradient wrt that tensor (same layout, NULL = none) added where the decoder's gradient arrives. */
int hpfg_unet_bottleneck(hpfg_unet_plan_t plan, float *feature_nchw, void *stream);
int hpfg_unet_backward_ex(hpfg_unet_plan_t plan, const float *params, const float *dlogits, const float *dbottleneck,
                          float *grads, int accumulate, void *stream);

/* Data-parallel hook: gradients complete back-to-front.  The flat gradient buffer is cut into
 * hpfg_unet_num_buckets() contiguous ranges (bucket 0 = the tail: out_conv, up4, ...).  After
 * hpfg_unet_backward has been enqueued, hpfg_unet_bucket_wait makes comm_stream wait until bucket i is
 * final, so an NCCL all-reduce of that range can be enqueued on comm_stream and overlap the rest of backward. */
int hpfg_unet_num_buckets(hpfg_unet_plan_t plan);
int hpfg_unet_bucket_range(hpfg_unet_plan_t plan, int bucket, int64_t *offset_host, int64_t *count_host);
int hpfg_unet_bucket_wait(hpfg_unet_plan_t plan, int bucket, void *comm_stream);
/* The same ranges without a plan (host only): int64[4] offsets / counts, bucket 0 first. */
int hpfg_unet_bucket_layout(int in_channels, int num_classes, int64_t *offsets_host, int64_t *counts_host);

/* Debug / parity taps: copy an internal activation of the last forward as fp32 NCHW.  name is one of the
 * conv names ("encoder.in_conv.conv_conv.0", ..., raw conv outputs incl. bias) . */
int hpfg_unet_debug_tap(hpfg_unet_plan_t plan, const char *name, float *out_nchw, int64_t capacity, void *stream);

/* Layer-isolated test hook for the bf16 tensor-core convolution kernels: runs ONE convolution on caller
 * tensors (bf16 NHWC activations, fp32 OIHW weights) and synchronises.  op 0 = fprop (in has cin channels, out
 * cout; optional per-input-channel scale/shift = the fused BN+LeakyReLU loader; optional bias[cout]);
 * op 1 = dgrad (in = dout with cout channels, out = din with cin channels).  stats_out (optional):
 * float[2*C_out_of_the_op] = per-channel sum | sum of squares of the fp32 accumulators. */
int hpfg_conv_tc_debug(int op, int batch, int height, int width, int cin, int cout, int ksize,
                       const void *in_bf16_nhwc, const float *w_oihw, const float *bias, const float *scale,
                       const float *shift, void *out_bf16_nhwc, float *stats_out, void *stream);

/* Same for the tensor-core weight-gradient kernel: dw_oihw[cout,cin,k,k] = sum_pixels act(x)[pixel+tap] * dy[pixel],
 * dbias[cout] = sum_pixels dy; x is transformed on load by scale/shift (+LeakyReLU) when given. */
int hpfg_wgrad_tc_debug(int batch, int height, int width, int cin, int cout, int ksize, const void *x_bf16_nhwc,
                        const void *dy_bf16_nhwc, const float *scale, const float *shift, float *dw_oihw, float *dbias,
                        void *stream);

/* Layer-isolated hooks for the BatchNorm-backward fusions (bf16 plans; DESIGN.md section 3.2).
 * hpfg_dgrad_tc_fused_debug: din = conv_transpose(draw, w) with
 *   raw_in  != NULL: draw = sc*g_in + kb*raw_in + kd built in the loader (g_in / raw_in bf16 NHWC [N,H,W,cout], constants float[cout]),
 *                    else draw = g_in;
 *   raw_out != NULL: the output is turned into g = din * leaky'(raw_out*gs_scale + gs_shift) * keep/(1-p) in the epilogue
 *                    (raw_out bf16 NHWC [N,H,W,cin]; gs_keep_mask_nchw uint8 [N,cin,H,W] or NULL) and stats_out (float[2*cin]) receives
 *                    sum g | sum g*raw_out per channel.
 * hpfg_wgrad_tc_fused_debug: dw = sum_pixels act(x)[pixel+tap] * draw[pixel] with draw = sc*g + kb*raw + kd built inside the kernel.
 * hpfg_glue_debug: one bf16 glue kernel on caller tensors; op 0 pool_act, 1 upcat, 2 bn_bwd (out_f32 = dgamma|dbeta), 3 skip_pool_bwd,
 *   4 up_bwd, 5 skip_pool_bwd fused with BatchNorm-backward pass 0 (out = g, out_f32 = dgamma|dbeta|kb|kd); shapes in csrc/glue.cu. */
int hpfg_dgrad_tc_fused_debug(int batch, int height, int width, int cin, int cout, int ksize, const void *g_in, const void *raw_in,
                              const float *sc, const float *kb, const float *kd, const float *w_oihw, const void *raw_out,
                              const float *gs_scale, const float *gs_shift, const uint8_t *gs_keep_mask_nchw, float gs_p_drop,
                              void *out_bf16_nhwc, float *stats_out, void *stream);
int hpfg_wgrad_tc_fused_debug(int batch, int height, int width, int cin, int cout, int ksize, const void *x_bf16_nhwc,
                              const void *g_bf16_nhwc, const void *raw_bf16_nhwc, const float *sc, const float *kb, const float *kd,
                              const float *scale, const float *shift, float *dw_oihw, float *dbias, void *stream);
int hpfg_glue_debug(int op, int batch, int height, int width, int channels, const void *a, const void *b, const void *c,
                    const float *scale, const float *shift, const float *mean, const float *invstd, const uint8_t *keep_mask_nchw,
                    float p_drop, void *out_bf16, float *out_f32, void *stream);

/* Layer micro-benchmark: average milliseconds of `iters` back-to-back launches of one tensor-core convolution
 * (op 0 fprop incl. fused loader and BN-stat epilogue, 1 dgrad, 2 wgrad) on internally allocated buffers. */
int hpfg_conv_tc_bench(int op, int batch, int height, int width, int cin, int cout, int ksize, int iters,
                       float *ms_out_host, void *stream);

/* ---- fused SSL loss (forward value + d loss / d logits) ---------------------------------------------
 * student: fp32 NCHW [n_l+n_u, C, H, W] logits.  labels: int64 [n_l, H, W] (255 = ignored by CE only).
 * other: MT/UAMT -> teacher logits for the UNLABELED slices [n_u, C, H, W];
 *        CPS     -> the peer network's logits [n_l+n_u, C, H, W];  SUP -> NULL.
 * mc_logits (UAMT only): [T*n_u, C, H, W] logits of the T stochastic teacher passes (pass-major).
 * dstudent / dother: gradients (dother only for CPS, else NULL).  class_weights: HOST array of C floats or NULL (=1).
 * scalars_out: float[8] device: {loss, loss_sup, loss_cons_or_semi, ce, dice, n_valid, mask_sum, 0}.
 * pseudo1/pseudo2 (CPS, optional): int64 [n_u,H,W] argmax pseudo-labels of net1 / net2.
 * workspace: at least hpfg_ssl_loss_workspace_bytes(...) bytes of device scratch. */
int64_t hpfg_ssl_loss_workspace_bytes(int mode, int n_l, int n_u, int num_classes, int height, int width);
int hpfg_ssl_loss(int mode, const float *student, const float *other, const float *mc_logits, int mc_passes,
                  const int64_t *labels, int n_l, int n_u, int num_classes, int height, int width,
                  float cons_weight, float uamt_threshold, const float *class_weights, float ce_coef,
                  float dice_coef, float *dstudent, float *dother, float *scalars_out, int64_t *pseudo1,
                  int64_t *pseudo2, void *workspace, void *stream);

/* hpfg_ssl_loss with the consistency weight read from device memory (cons_weight_dev, required) and, when
 * uamt_threshold_dev is not NULL, the UAMT threshold too (2019_07...:150, it ramps with the iteration count); with
 * uamt_threshold_dev NULL the by-value uamt_threshold is used. */
int hpfg_ssl_loss_dv(int mode, const float *student, const float *other, const float *mc_logits, int mc_passes,
                     const int64_t *labels, int n_l, int n_u, int num_classes, int height, int width,
                     const float *cons_weight_dev, float uamt_threshold, const float *uamt_threshold_dev,
                     const float *class_weights, float ce_coef, float dice_coef, float *dstudent, float *dother,
                     float *scalars_out, int64_t *pseudo1, int64_t *pseudo2, void *workspace, void *stream);

/* ---- "next" rows of SURVEY 8f.4: the ICT-MedSeg and S4CVNet step losses on the same two kernels ------------------
 * ICT (2022_02_ISBI_ICT-MedSeg_ACDC.py:111-137): student = logits of cat([labeled, mixed unlabeled]) [n_l+n_mixed,C,H,W];
 * teacher_u = teacher logits of the 2*n_mixed un-mixed unlabeled slices (first half ux0, second half ux1);
 * mix_factors = device float[n_mixed] (the Beta(alpha,alpha) draws).  loss = 0.5*(CE+Dice) on the labeled slices +
 * w * mean((softmax(student_mixed) - ((1-l)*softmax(t(ux0)) + l*softmax(t(ux1))))^2).  cons_weight_dev (optional device
 * scalar) overrides cons_weight (graph replay).  scalars_out as hpfg_ssl_loss ([2] = the unweighted consistency term).
 * Workspace: hpfg_ssl_loss_workspace_bytes(HPFG_LOSS_ICT, n_l, n_mixed, ...). */
int hpfg_ict_loss(const float *student, const float *teacher_u, const float *mix_factors, const int64_t *labels,
                  int n_l, int n_mixed, int num_classes, int height, int width, float cons_weight,
                  const float *cons_weight_dev, const float *class_weights, float ce_coef, float dice_coef,
                  float *dstudent, float *scalars_out, void *workspace, void *stream);
/* The ICT input mix out[u] = a[u]*(1-l_u) + b[u]*l_u over n images of per_image floats (2022_02...:115-117). */
int hpfg_ict_mix(const float *a, const float *b, const float *mix_factors, int n, int64_t per_image, float *out,
                 void *stream);
/* S4CVNet (2022_08_CVPR_S4CVNet_ACDC.py:124-156): logits1/logits2 [n_l+n_u,C,H,W] of the two students, teacher_u
 * [n_u,C,H,W] EMA-teacher logits (NULL = no Mean-Teacher term, the reference's cur_itrs < 1000 branch).
 * loss = sup1 + sup2 + cps_weight*(Dice(softmax1_u, argmax2) + Dice(softmax2_u, argmax1))
 *        + mt_weight*(mean((softmax1_u-softmax_t)^2) + mean((softmax2_u-softmax_t)^2));
 * the caller passes cps_weight = 7*consistency*linear_rampup(...) (:148-149).  weights_dev: optional device float[2]
 * {cps_weight, mt_weight} overriding the by-value weights.  scalars_out: {loss, loss_sup, loss_semi, ce1, dice1, n_valid,
 * ps1+ps2, cl1+cl2}.  Workspace: hpfg_ssl_loss_workspace_bytes(HPFG_LOSS_S4CV, ...). */
int hpfg_s4cv_loss(const float *logits1, const float *logits2, const float *teacher_u, const int64_t *labels, int n_l,
                   int n_u, int num_classes, int height, int width, float cps_weight, float mt_weight,
                   const float *weights_dev, const float *class_weights, float ce_coef, float dice_coef,
                   float *dlogits1, float *dlogits2, float *scalars_out, int64_t *pseudo1, int64_t *pseudo2,
                   void *workspace, void *stream);

/* ---- HPFG model1 (main.py:125-134,143; replaces Med_Sup_Loss on outputs1[:n_l] plus the pseudo_supervision1 DiceLoss):
 *   loss = ce_coef*CE(s[:n_l], labels) + dice_coef*Dice(softmax(s[:n_l]), labels) + pseudo_weight*Dice(softmax(s[n_l:]), pseudo)
 *   pseudo[u,p] = labels1[u % n_l1, p]*(1 - m[u,p]) + argmax_c softmax(teacher_u[u])[c,p]*m[u,p]   in fp32 as torch rounds it;
 * a pixel is class c for the Dice term iff that float equals c (the reference's one-hot; for a 0/1 mask: a torch.where).  The
 * argmax is the first maximum of the accurate softmax, the labels of hpfg_argmax_labels.  student [n_l+n_u,C,H,W], teacher_u
 * [n_u,C,H,W] fp32; labels [n_l,H,W], labels1 [n_l1,H,W] int64 (never repeated: image u reads u % n_l1, main.py:139-140);
 * cutmix_mask [n_u,1,H,W] fp32.  n_u must be a multiple of n_l1 (HPFG_ERR_INVALID otherwise).  pseudo_weight_dev (optional
 * device scalar) overrides pseudo_weight (graph replay).  dstudent: the gradient for all n_l+n_u images.  scalars_out: {loss,
 * loss_sup, pseudo Dice (unweighted), ce, dice, n_valid, 0, 0}.  pseudo_out (optional): int64 [n_u,H,W], the class each pixel
 * took in the Dice term (255: none).  Workspace: hpfg_ssl_loss_workspace_bytes(HPFG_LOSS_CUTMIX, n_l, n_u, ...). */
int hpfg_cutmix_loss(const float *student, const float *teacher_u, const int64_t *labels, const int64_t *labels1,
                     const float *cutmix_mask, int n_l, int n_u, int n_l1, int num_classes, int height, int width,
                     float pseudo_weight, const float *pseudo_weight_dev, const float *class_weights, float ce_coef,
                     float dice_coef, float *dstudent, float *scalars_out, int64_t *pseudo_out, void *workspace, void *stream);
/* The CutMix input mix (main.py:139,145): out[u] = a[u % n_a]*(1 - m[u]) + b[u]*m[u] over n images of `channels` planes of
 * H*W floats, the [n,1,H,W] mask broadcast over the channels; separate fp32 roundings (bit-identical to torch's expression on
 * the repeated draw).  n must be a multiple of n_a. */
int hpfg_cutmix_mix(const float *a, const float *b, const float *cutmix_mask, int n, int n_a, int channels, int height,
                    int width, float *out, void *stream);

/* ---- inference side (SURVEY 8f.3; val.py:268-281 test_single_volume): argmax(softmax(logits), dim=1), first maximum
 * wins, for a whole batch of eval-mode logits in one launch.  Either output may be NULL. */
int hpfg_argmax_labels(const float *logits, int n, int num_classes, int height, int width, int64_t *labels_i64,
                       uint8_t *labels_u8, void *stream);

/* softmax_mse_loss (utils/loss/diceloss.py:64-81): the UNREDUCED map (softmax(input) - softmax(target))^2 over dim 1
 * (sigmoid != 0: element-wise sigmoids instead), all tensors fp32 NCHW [n,C,H,W].  grad_out == NULL: out = the map;
 * grad_out != NULL: out = d(sum(grad_out * map)) / d input_logits (the target carries no gradient, as in the trainers,
 * where it is the no_grad teacher output: 2019_07...:134-143,148). */
int hpfg_softmax_mse(const float *input_logits, const float *target_logits, const float *grad_out, int n, int num_classes,
                     int height, int width, int sigmoid, float *out, void *stream);

/* DiceLoss.forward (utils/loss/diceloss.py:178-191) alone: inputs are probabilities (softmax == 0) or
 * logits (softmax != 0); target int64 [n,H,W]; dinputs optional. scalars_out: float[1+C] = {loss, dice_c..}. */
int hpfg_dice_loss(const float *inputs, const int64_t *target, int n, int num_classes, int height, int width,
                   int softmax, const float *class_weights, float *dinputs, float *scalars_out, void *workspace,
                   void *stream);

/* ---- UNet_Plus projection necks and Dense_Loss (SURVEY 8f.2) ----------------------------------------------------
 * projection_conv.forward (model/unet.py:140-152) on x [n,channels,H,W] fp32 NCHW:
 *   out_global [n,out]     = mlp(AdaptiveAvgPool2d((1,1))(x))            (Linear -> ReLU -> Linear)
 *   out_dense  [n,out,s*s] = mlp_conv(AdaptiveAvgPool2d((s,s))(x))       (1x1 conv -> ReLU -> 1x1 conv), s >= 1.
 * params[8]: mlp.0.weight [hid,channels], mlp.0.bias, mlp.2.weight [out,hid], mlp.2.bias, mlp_conv.0.weight
 * [hid,channels(,1,1)], mlp_conv.0.bias, mlp_conv.2.weight [out,hid(,1,1)], mlp_conv.2.bias -- the module's registration
 * order.  pooled [n*(1+s*s), channels] and hidden [n*(1+s*s), hid] are written here and read by hpfg_neck_backward
 * (rows 0..n-1: the global branch; row n + image*s*s + i*s + j: bin (i,j)). */
int hpfg_neck_forward(const float *x, int n, int channels, int height, int width, int s, int hid, int out,
                      const float *const *params, float *pooled, float *hidden, float *out_global, float *out_dense,
                      void *stream);
/* Adjoint of hpfg_neck_forward: d_global [n,out], d_dense [n,out,s*s] -> grads[8] (same order and shapes as params,
 * overwritten) and, when dx != NULL, dx [n,channels,H,W] (overwritten).  scratch: n*s*s*out + n*(1+s*s)*(hid+channels)
 * floats. */
int hpfg_neck_backward(const float *d_global, const float *d_dense, int n, int channels, int height, int width, int s,
                       int hid, int out, const float *const *params, const float *pooled, const float *hidden,
                       float *const *grads, float *dx, float *scratch, void *stream);
/* Dense_Loss.contrastive_loss (utils/loss/dense_loss.py:18-34) with batch_size = batch: out1, out2 [batch,dim,positions]
 * fp32 (positions = 1 for the global vectors); loss[1]; d_out1 (optional) = d loss / d out1 (out2 is the detached teacher
 * side, :38-39).  workspace: hpfg_dense_contrastive_workspace_floats(batch, dim, positions) floats. */
int64_t hpfg_dense_contrastive_workspace_floats(int batch, int dim, int positions);
int hpfg_dense_contrastive(const float *out1, const float *out2, int batch, int dim, int positions, float temperature,
                           float *loss, float *d_out1, float *workspace, void *stream);
/* The same with d_out1 = scale * d loss / d out1 (a separate fp32 rounding: bit-identical to scaling the unscaled gradient);
 * the loss stays unscaled.  scale_dev (optional device scalar) overrides scale (graph replay).  HPFGStep passes the 0.5*w
 * that main.py:144,166 (w * (0.5*(contrast_global + contrast_dense)) per neck) puts in front of each term, which autograd
 * used to apply. */
int hpfg_dense_contrastive_scaled(const float *out1, const float *out2, int batch, int dim, int positions, float temperature,
                                  float scale, const float *scale_dev, float *loss, float *d_out1, float *workspace,
                                  void *stream);

/* ---- optimiser-side passes over the flat buffers --------------------------------------------------- */
/* update_ema_variables (utils/utils.py:82-86): ema <- alpha*ema + (1-alpha)*param, alpha already clamped. */
int hpfg_ema_update(float *ema, const float *param, int64_t n, float alpha, void *stream);
/* The same with alpha_dev: device float[2] = {alpha, 1 - alpha} (graph replay; the same arithmetic as hpfg_ema_update, whose
 * 1 - alpha is an fp32 subtraction).  HPFGStep: the backbone EMA model2 <- model1 (main.py:68-76) and the teacher EMA over the
 * flat buffer and each neck tensor (utils/utils.py:82-86). */
int hpfg_ema_update_dv(float *ema, const float *param, int64_t n, const float *alpha_dev, void *stream);
/* torch.optim.SGD step (momentum, weight decay, no nesterov/dampening): first_step != 0 initialises the
 * momentum buffer with the decayed gradient.  grad_scale multiplies the gradient first (1/world for DP). */
int hpfg_sgd_momentum(float *param, const float *grad, float *momentum_buf, int64_t n, float lr, float momentum,
                      float weight_decay, float grad_scale, int first_step, void *stream);
/* SGD step and EMA teacher update in one pass (the two calls above, fused). */
int hpfg_sgd_momentum_ema(float *param, const float *grad, float *momentum_buf, float *ema, int64_t n, float lr,
                          float momentum, float weight_decay, float grad_scale, int first_step, float ema_alpha,
                          void *stream);

/* lr_alpha_dev: device float[3] = {lr, ema_alpha, 1 - ema_alpha}. */
int hpfg_sgd_momentum_ema_dv(float *param, const float *grad, float *momentum_buf, float *ema, int64_t n,
                             float momentum, float weight_decay, float grad_scale, int first_step,
                             const float *lr_alpha_dev, void *stream);

/* lr_dev: device float[1] = {lr} (the CPS networks have no EMA teacher). */
int hpfg_sgd_momentum_dv(float *param, const float *grad, float *momentum_buf, int64_t n, float momentum,
                         float weight_decay, float grad_scale, int first_step, const float *lr_dev, void *stream);

/* torch.optim.Adam (decoupled == 0: L2 weight decay added to the gradient) or torch.optim.AdamW (decoupled != 0:
 * param *= decay_factor) step, foreach implementation, no amsgrad / maximize; with ema != NULL, followed in the same
 * pass by update_ema_variables (utils/utils.py:82-86) of the updated parameters into ema.  The scalars are what torch
 * computes in Python (double) and casts to fp32: one_minus_beta1 = 1 - beta1, one_minus_beta2 = 1 - beta2 (not
 * recomputed from the fp32 betas), and per step t: step_size = -lr / (1 - beta1^t), bc2_sqrt = sqrt(1 - beta2^t),
 * decay_factor = 1 - lr*weight_decay.  grad_scale multiplies the gradient first (1/world for DP).  The caller keeps
 * the step count. */
int hpfg_adam(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, float *ema, int64_t n,
              float one_minus_beta1, float beta2, float one_minus_beta2, float eps, float weight_decay, int decoupled,
              float grad_scale, float step_size, float bc2_sqrt, float decay_factor, float ema_alpha, void *stream);

/* dyn: device float[5] = {step_size, bc2_sqrt, decay_factor, ema_alpha, 1 - ema_alpha}. */
int hpfg_adam_dv(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, float *ema, int64_t n,
                 float one_minus_beta1, float beta2, float one_minus_beta2, float eps, float weight_decay, int decoupled,
                 float grad_scale, const float *dyn, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* HPFG_B200_H */
