/*
 * b200resnet.h — C ABI of libb200resnet.so: the sm_100a kernels behind the ResNet/WRN training step.
 *
 * This is the drop-in boundary for the hot path of lucaslingle/pytorch_ddp_resnet. The reference has
 * no native code of its own: every arithmetic op on its path is a torch (ATen/cuDNN/cuBLAS) call made
 * from Python. Each entry point below names the reference call site (file:line under the reference
 * repo) whose ATen dispatch it replaces. The host-side mirror in pytorch_ddp_resnet_b200/ binds these
 * through ctypes (see INTEGRATION.md for the stub a reference maintainer would add).
 *
 * Conventions
 *   - plain C linkage, POD arguments only (device pointers, ints, floats, a cudaStream_t as void*);
 *   - every call returns 0 on success, non-zero on error; b200_last_error() gives the message
 *     (thread-local). Nothing throws, nothing calls exit();
 *   - all launches are asynchronous on the given stream; no call synchronises the device;
 *   - no allocation inside: the caller owns every buffer, including workspaces whose size the
 *     matching *_workspace_bytes() query returns;
 *   - activations are NHWC bf16 ("channels_last" physical layout of an NCHW-shaped torch tensor);
 *     conv filters are KRSC (physical layout of an OIHW-shaped channels_last torch tensor):
 *     fp32 masters, bf16 working copies in KRSC and CRSK (transposed) order made by b200_weight_prep;
 *   - statistics, affine parameters, optimizer state and weight gradients are fp32.
 */
#ifndef B200RESNET_H_
#define B200RESNET_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* b200_stream_t; /* a cudaStream_t */

/* conv algorithm selector */
enum { B200_ALGO_AUTO = 0, B200_ALGO_DIRECT = 1, B200_ALGO_TC = 2 };
/* Flag, or-ed into any `algo` argument: DETERMINISTIC reductions (the analogue of cuDNN's deterministic algorithms
 * behind torch.use_deterministic_algorithms). b200_conv2d_wgrad then reduces its pixel-range splits (and the
 * blocks of the bias gradient) in a fixed order from partials kept in the workspace - pass the flag to
 * b200_conv2d_workspace_bytes too - instead of fp32 atomics in completion order; the conv epilogues with fused
 * statistics (b200_conv2d_fprop_stats, b200_conv2d_dgrad_bnbwd) sum their per-warp partials in a fixed order
 * instead of shared-memory atomics. Same inputs => bit-identical outputs, run after run. Without the flag the
 * last bits of weight gradients and batch statistics depend on the order in which CTAs finish. */
enum { B200_ALGO_DETERMINISTIC = 0x100 };
/* which conv pass a workspace query refers to */
enum { B200_PASS_FPROP = 0, B200_PASS_DGRAD = 1, B200_PASS_WGRAD = 2 };
/* skip-connection addressing for the fused BN kernels */
enum {
  B200_SKIP_NONE = 0,
  B200_SKIP_SAME = 1,       /* skip tensor has the output's shape                                  */
  B200_SKIP_SUBSAMPLE_PAD = 2 /* skip is [N,2H,2W,Cs]: read at (2h,2w), channels >= Cs read as zero */
};

/* ---- library ------------------------------------------------------------------------------- */
int b200_version(void);
const char* b200_last_error(void);
/* Number of kernels this library has launched in the calling process so far. */
long long b200_launch_count(void);
/* 0 iff the current CUDA device is compute capability 10.x (sm_100a code is the only code here). */
int b200_device_check(void);
/* Returns 1 when the tcgen05 path supports the shape, else 0. Never fails. */
int b200_conv2d_tc_supported(int pass, int N, int H, int W, int C, int K, int R, int S, int stride,
                             int pad);

/* ---- filters --------------------------------------------------------------------------------
 * fp32 KRSC master -> bf16 KRSC (fprop, wgrad layout) and bf16 CRSK (dgrad operand).
 * Replaces the per-call autocast weight cast of tc.nn.Conv2d (residual_block.py:34-57,129-159;
 * resnet.py:69-75). Either output may be NULL. */
int b200_weight_prep(const float* w_krsc, void* w_krsc_bf16, void* w_crsk_bf16, int K, int RS, int C,
                     b200_stream_t stream);

/* The same for n filters in one launch. `table` is a DEVICE array of n 40-byte records
 * { const float* w_krsc; void* w_krsc_bf16; void* w_crsk_bf16; int32 K, RS, C, pad; }. */
int b200_weight_prep_multi(const void* table, int n, b200_stream_t stream);

/* ---- convolution (aten::convolution / convolution_backward; call sites residual_block.py:73,78,
 * 81,86,179-203,92,208 and resnet.py:69-75). Shapes: x [N,H,W,C], w [K,R,S,C], y [N,P,Q,K] with
 * P = (H + 2*pad - R)/stride + 1. stride in {1,2}. --------------------------------------------- */
size_t b200_conv2d_workspace_bytes(int pass, int N, int H, int W, int C, int K, int R, int S,
                                   int stride, int pad, int algo);

/* y = bf16( conv(x, w) [+ bias] ) ; if residual: y = bf16(y + residual)  (residual add of
 * residual_block.py:96,212 fused into the epilogue); if relu: y = max(y, 0) last (evaluation with the
 * following batch norm folded into w / bias, see utils/fold_util.py). bias (fp32 [K]) and residual may be NULL. */
int b200_conv2d_fprop(const void* x, const void* w_krsc, const float* bias, const void* residual,
                      void* y, int N, int H, int W, int C, int K, int R, int S, int stride, int pad,
                      int relu, int algo, void* ws, size_t ws_bytes, b200_stream_t stream);

/* b200_conv2d_fprop that ALSO computes the batch statistics of its output for the batch norm that follows a
 * conv in the reference (residual_block.py:69-98), so that BN needs no pass of its own over y. Per output
 * channel k, sum(y[..,k]) and sum(y[..,k]^2) over all N*P*Q output pixels (of the bf16 values it stores) are
 * accumulated in the BN accumulator workspace `stats_ws` (b200_bn_workspace_bytes(rows, K) bytes, contract
 * below: zero on entry). With mean / invstd non-NULL (fp32 [K]) the CTA that finishes last turns the sums
 * into mean and invstd = rsqrt(biased var + eps) and clears the workspace: no further launch is needed (the
 * running statistics are then updated by b200_bn_act_fwd or b200_bn_running_update). With mean == invstd ==
 * NULL the sums stay in the workspace for b200_bn_stats_finalize. The tcgen05 SM-pair kernels do all of this
 * in their epilogue; other conv paths run one reduction pass over y, so the result is the same either way. */
int b200_conv2d_fprop_stats(const void* x, const void* w_krsc, const float* bias, const void* residual,
                            void* y, int N, int H, int W, int C, int K, int R, int S, int stride,
                            int pad, int algo, void* ws, size_t ws_bytes, void* stats_ws,
                            size_t stats_ws_bytes, float eps, float* mean, float* invstd,
                            b200_stream_t stream);

/* dx = bf16( conv_transpose(dy, w) ) ; if addend: dx = bf16(dx + addend) (skip-path gradient).
 * w_crsk is the transposed bf16 filter from b200_weight_prep. */
int b200_conv2d_dgrad(const void* dy, const void* w_crsk, const void* addend, void* dx, int N, int H,
                      int W, int C, int K, int R, int S, int stride, int pad, int algo, void* ws,
                      size_t ws_bytes, b200_stream_t stream);

/* b200_conv2d_dgrad whose output dx is the dy of a batch norm + ReLU + dropout backward (the layer in FRONT of the
 * convolution: reference resnet/architectures/residual_block.py:67-85, autograd of norm -> act -> dropout -> conv).
 * The tcgen05 epilogue also accumulates, per channel of dx, sum(g) and sum(g * x_bn) with g = dx where the mask bit
 * of b200_bn_act_fwd is set (scaled by 1/(1-p) and rounded to bf16 when dropout_p > 0), else 0, and the last CTA
 * writes dbeta = sum(g), dgamma = invstd * (sum(g x) - mean * sum(g)): the whole reduction pass of b200_bn_act_bwd.
 * x_bn: the batch norm's input [N,H,W,C] bf16; mask: uint8 [N,H,W,C/8]; stats_ws as for b200_conv2d_fprop_stats.
 * *fused = 1: dgamma / dbeta are final, continue with b200_bn_act_bwd_apply. *fused = 0: the shape ran on a
 * kernel without this epilogue (dx is still complete), continue with b200_bn_act_bwd. */
int b200_conv2d_dgrad_bnbwd(const void* dy, const void* w_crsk, void* dx, int N, int H, int W, int C, int K,
                            int R, int S, int stride, int pad, int algo, void* ws, size_t ws_bytes,
                            const void* x_bn, const void* mask, const float* mean, const float* invstd,
                            float dropout_p, float* dgamma, float* dbeta, void* stats_ws,
                            size_t stats_ws_bytes, int* fused, b200_stream_t stream);

/* dw[K,R,S,C] (fp32) = sum over pixels of dy (x) x. dbias (fp32 [K], may be NULL) = sum of dy.
 * dw may point into a flat gradient bucket. With B200_ALGO_DETERMINISTIC in `algo` the reduction over pixel
 * ranges is ordered (16-byte aligned workspace of b200_conv2d_workspace_bytes(B200_PASS_WGRAD, ..., same algo)). */
int b200_conv2d_wgrad(const void* dy, const void* x, float* dw_krsc, float* dbias, int N, int H, int W,
                      int C, int K, int R, int S, int stride, int pad, int algo, void* ws,
                      size_t ws_bytes, b200_stream_t stream);

/* ---- fp32 / TF32 precision mode ---------------------------------------------------------------------------
 * The reference evaluates WITHOUT autocast (evaluation.py:32-39) and trains without it when no GradScaler is
 * passed (training.py:101-102): fp32 tensors whose convolutions cuDNN runs on TF32 tensor cores (torch's
 * default allow_tf32 for cudnn). These entry points are that mode: fp32 NHWC activations, fp32 KRSC (fprop,
 * wgrad) / CRSK (dgrad) filters read directly by tcgen05 kind::tf32 MMAs (fp32 accumulate), fp32 outputs, no
 * intermediate rounding of bias / residual / addend. No workspace. Shapes the TF32 path does not cover are an
 * error (b200_conv2d_tf32_supported tells). */
int b200_conv2d_tf32_supported(int pass, int N, int H, int W, int C, int K, int R, int S, int stride, int pad);
/* fprop accepts EVERY shape: those outside the tensor path run as im2col + TF32 GEMM (few input channels: the
 * stems; needs the workspace) or as an exact fp32 CUDA-core convolution (channel counts below 32, odd tiles). */
size_t b200_conv2d_tf32_workspace_bytes(int N, int H, int W, int C, int K, int R, int S, int stride, int pad);
int b200_conv2d_fprop_tf32(const float* x, const float* w_krsc, const float* bias, const float* residual,
                           float* y, int N, int H, int W, int C, int K, int R, int S, int stride, int pad,
                           int relu, void* ws, size_t ws_bytes, b200_stream_t stream);
int b200_conv2d_dgrad_tf32(const float* dy, const float* w_crsk, const float* addend, float* dx, int N, int H,
                           int W, int C, int K, int R, int S, int stride, int pad, b200_stream_t stream);
int b200_conv2d_wgrad_tf32(const float* dy, const float* x, float* dw_krsc, int N, int H, int W, int C, int K,
                           int R, int S, int stride, int pad, b200_stream_t stream);

/* The fp32 activation kernels around the TF32 convolutions (forward pass of the un-autocast reference:
 * evaluation.py:32-39): same semantics as their bf16 namesakes, fp32 NHWC in and out, no intermediate rounding. */
int b200_nchw_to_nhwc_f32(const float* x, float* y, int N, int C, int H, int W, b200_stream_t stream);
int b200_bn_act_fwd_f32(const float* x, float* y, int N, int H, int W, int C, const float* mean,
                        const float* stat, int stat_is_var, float eps, const float* gamma, const float* beta,
                        const float* skip, int skip_mode, int skip_C, int relu, b200_stream_t stream);
int b200_subsample2_f32(const float* x, float* y, int N, int H, int W, int C, b200_stream_t stream);
int b200_pool_fwd_f32(const float* x, float* y, int N, int H, int W, int C, int k, int stride, int pad,
                      int is_max, b200_stream_t stream);
int b200_linear_fwd_f32(const float* x, const float* w, const float* b, float* logits, int B, int I, int O,
                        b200_stream_t stream);
/* out (fp32[3]) = {mean cross entropy, top-1 error, top-5 error} of fp32 logits */
int b200_ce_topk_f32(const float* logits, const int64_t* labels, float* out, int B, int O, b200_stream_t stream);

/* fp32 NCHW image batch -> bf16 NHWC (the x.to(device) + autocast input cast of training.py:94-96). */
int b200_nchw_f32_to_nhwc_bf16(const float* x, void* y, int N, int C, int H, int W,
                               b200_stream_t stream);

/* ---- batch norm + activation + dropout + skip (aten::native_batch_norm, relu, native_dropout, add,
 * constant_pad_nd, avg_pool2d(k=1,s=2); residual_block.py:58-65,69-98,175-214; resnet.py:111-115) -- */
/* Size of the ACCUMULATOR workspace of b200_bn_stats / b200_bn_act_bwd / b200_conv2d_fprop_stats:
 * several copies of fp64 [2][C] sums (spread over L2 slices) + a ticket counter. Contract: 8-byte aligned, zero-filled before its first use, not shared between streams that
 * run concurrently; every call leaves it zero-filled again (the block that finishes last folds the sums
 * into the outputs and clears them), so one cudaMemset when it is allocated is all a caller needs. */
size_t b200_bn_workspace_bytes(int64_t rows, int C);

/* Per-channel batch statistics of x [rows, C] (bf16): mean, invstd = rsqrt(biased var + eps).
 * If running_mean/running_var are non-NULL they are updated in place with `momentum` and the
 * unbiased variance; if num_batches_tracked (int64 scalar) is non-NULL it is incremented. */
int b200_bn_stats(const void* x, int64_t rows, int C, float eps, float momentum, float* mean,
                  float* invstd, float* running_mean, float* running_var,
                  int64_t* num_batches_tracked, void* ws, size_t ws_bytes, b200_stream_t stream);

/* Second half of b200_bn_stats for sums that b200_conv2d_fprop_stats left in `ws`: mean / invstd
 * (+ running statistics, num_batches_tracked) from the accumulated sums of `rows` values per channel;
 * clears the workspace. */
int b200_bn_stats_finalize(int64_t rows, int C, float eps, float momentum, float* mean, float* invstd,
                           float* running_mean, float* running_var, int64_t* num_batches_tracked,
                           void* ws, size_t ws_bytes, b200_stream_t stream);

/* running_mean / running_var (momentum, unbiased variance) and num_batches_tracked from a batch mean /
 * invstd pair that b200_conv2d_fprop_stats produced (aten::native_batch_norm's buffer update). */
int b200_bn_running_update(const float* mean, const float* invstd, int64_t rows, int C, float eps,
                           float momentum, float* running_mean, float* running_var,
                           int64_t* num_batches_tracked, b200_stream_t stream);

/* y = dropout( act( (x - mean) * invstd * gamma + beta [+ skip] ) ).
 * stat_is_var != 0: `invstd` holds a variance (eval mode, running stats) and rsqrt(var+eps) is applied.
 * gamma/beta/mean/invstd NULL  => the affine/normalise step is skipped (plain act/dropout/add).
 * relu: 0/1. dropout_p in [0,1): keep mask from the counter RNG keyed by (seed, element index);
 * seed_offset (device uint64 scalar, may be NULL) is a step counter folded into the seed on the
 * device, so a captured CUDA graph draws a fresh mask at every replay (see b200_tick).
 * x is [N,H,W,C]; skip addressing per skip_mode (skip_C = channel count of the skip tensor).
 * running_mean (may be NULL): also perform the running-statistics update of b200_bn_running_update with
 * these mean / invstd, eps, `momentum` and rows = N*H*W (training forward whose statistics came out of
 * b200_conv2d_fprop_stats: saves the separate launch).
 * mask_out (may be NULL): N*H*W*C/8 bytes, one per (pixel, 8-channel group); bit j set = channel 8g+j passed
 * the ReLU gate (if relu) and was kept by the dropout (if dropout_p > 0). b200_bn_act_bwd takes it instead of
 * y: 0.125 instead of 2 bytes per element of backward traffic in each of its two kernels. */
int b200_bn_act_fwd(const void* x, void* y, int N, int H, int W, int C, const float* mean,
                    const float* invstd, int stat_is_var, float eps, const float* gamma,
                    const float* beta, const void* skip, int skip_mode, int skip_C, int relu,
                    float dropout_p, uint64_t seed, const uint64_t* seed_offset, float* running_mean,
                    float* running_var, int64_t* num_batches_tracked, float momentum, void* mask_out,
                    b200_stream_t stream);

/* Backward of b200_bn_act_fwd. x is the forward input, dy the gradient w.r.t. the forward output y.
 * The combined ReLU + dropout mask comes from `mask` (the bytes b200_bn_act_fwd wrote to mask_out) when it is
 * non-NULL; else from the non-zero pattern of y when relu != 0 (y may then not be NULL); without ReLU and
 * without mask the dropout mask is regenerated from (seed, element index).
 * With g = dy * dropmask * 1/(1-p) * relumask this produces dbeta = sum(g), dgamma = sum(g * xhat), dx (bf16)
 * and, if dskip != NULL, g itself (the gradient flowing to the skip operand, output-shaped). If addend !=
 * NULL: dx = bf16(dx + addend) (same shape; the strided skip gradients use b200_upsample_add).
 * gamma NULL => no normalisation (dx = g). */
int b200_bn_act_bwd(const void* dy, const void* y, const void* mask, const void* x, void* dx, void* dskip,
                    const void* addend, int64_t rows, int C, const float* mean, const float* invstd,
                    const float* gamma, float* dgamma, float* dbeta, int relu, float dropout_p,
                    uint64_t seed, const uint64_t* seed_offset, void* ws, size_t ws_bytes,
                    b200_stream_t stream);

/* The second pass of b200_bn_act_bwd alone: dx (and dskip) from dy, the mask bytes, x and the per-channel sums
 * dgamma / dbeta, which are INPUTS here (b200_conv2d_dgrad_bnbwd with *fused = 1 produced them). Needs the mask
 * and the affine operands; no workspace, no random numbers. */
int b200_bn_act_bwd_apply(const void* dy, const void* mask, const void* x, void* dx, void* dskip,
                          const void* addend, int64_t rows, int C, const float* mean, const float* invstd,
                          const float* gamma, const float* dgamma, const float* dbeta, int relu,
                          float dropout_p, b200_stream_t stream);

/* y[n,h,w,c] = x[n,2h,2w,c] (AvgPool2d(kernel 1, stride 2), residual_block.py:49,90,151,206). */
int b200_subsample2(const void* x, void* y, int N, int H, int W, int C, b200_stream_t stream);
/* dx[n,2h,2w,c] += g[n,h,w,c] for c < Cg (backward of subsample (+ zero channel pad)); dx is
 * [N,2H,2W,C] with C >= Cg, g is [N,H,W,ldg] (channel pitch ldg >= Cg; only the first Cg are used). */
int b200_upsample_add(void* dx, const void* g, int N, int H, int W, int C, int Cg, int ldg,
                      b200_stream_t stream);

/* ---- pooling (resnet.py:77-87) ------------------------------------------------------------- */
int b200_avgpool_fwd(const void* x, void* y, int N, int H, int W, int C, int k, int stride, int pad,
                     b200_stream_t stream);
int b200_avgpool_bwd(const void* dy, void* dx, int N, int H, int W, int C, int k, int stride, int pad,
                     b200_stream_t stream);
/* argmax (may be NULL in eval): one byte per output element = window position r*k + s of the first maximum in
 * row-major scan order (torch's max_pool2d_with_indices rule); the backward pass needs only dy and argmax. */
int b200_maxpool_fwd(const void* x, void* y, void* argmax, int N, int H, int W, int C, int k, int stride,
                     int pad, b200_stream_t stream);
int b200_maxpool_bwd(const void* dy, const void* argmax, void* dx, int N, int H, int W, int C, int k,
                     int stride, int pad, b200_stream_t stream);

/* ---- classifier head (resnet.py:117-120; metrics.py:10-29) ---------------------------------- */
/* logits[B,O] (bf16) = bf16(x[B,I] (bf16) . bf16(w[O,I])^T + bf16(b[O])) */
int b200_linear_fwd(const void* x, const float* w, const float* b, void* logits, int B, int I, int O,
                    b200_stream_t stream);
/* dx (bf16 [B,I]), dw (fp32 [O,I]), db (fp32 [O]) from dlogits (bf16 [B,O]) */
int b200_linear_bwd(const void* dlogits, const void* x, const float* w, void* dx, float* dw,
                    float* db, int B, int I, int O, b200_stream_t stream);
/* Mean cross entropy over the batch + top-1 / top-5 error. out (fp32[3], may be NULL) =
 * {loss, top1_err, top5_err}; dlogits (bf16 [B,O], may be NULL) = (softmax - onehot) * s / B with
 * s = *grad_scale (device fp32 scalar, NULL => 1). labels int64. */
int b200_ce_topk(const void* logits, const int64_t* labels, float* out, void* dlogits,
                 const float* grad_scale, int B, int O, b200_stream_t stream);

/* ---- input pipeline (the step BEFORE the hot path: resnet/utils/transform_util.py:32-205 applied per sample
 * by the DataLoader, data_util.py:218-227, then x.to(device), training.py:94) --------------------------------
 * One launch builds a whole batch from a device-resident uint8 dataset data[M][H][W][C]:
 *   out[b] = crop( pad( flip( whiten( to_tensor( data[index[b]] ) ) ) ) )
 * to_tensor: x/255 (ToTensorTransform); whiten: (x - mean) / stddev with per-pixel-and-channel statistics
 * [C][H][W] (mean NULL: none; stddev NULL: zero-mean only); flip[b] != 0: horizontal flip (NULL: none);
 * pad / pad_mirror: PaddingTransform zero or 'reflect'; top[b], left[b]: RandomCropTransform offsets into the
 * padded image (NULL: no crop, the output is the whole padded image). The random draws are inputs.
 * Outputs (either may be NULL): fp32 [B][C][out_h][out_w] — bit-identical to the reference pipeline — and
 * bf16 [B][out_h][out_w][C], the NHWC tensor the stem convolution consumes. */
int b200_augment_batch(const void* data, const int64_t* index, const void* flip, const int32_t* top,
                       const int32_t* left, const float* mean, const float* stddev, int B, int H, int W,
                       int C, int pad, int pad_mirror, int out_h, int out_w, int to_tensor,
                       float* out_f32_nchw, void* out_bf16_nhwc, b200_stream_t stream);

/* ---- optimizer (torch.optim.SGD via optim_util.py:11-18, stepped at training.py:108-113) ------
 * One launch for `n` tensors. Per element: g = grad (* inv_scale); g += wd * p;
 * buf = first_step ? g : momentum*buf + (1-dampening)*g; g = nesterov ? g + momentum*buf : buf;
 * p -= lr * g. If found_inf != NULL and *found_inf != 0 the step is skipped (GradScaler contract).
 * lr_ptr (device fp32 scalar, may be NULL) overrides lr: schedulers can change it under a CUDA graph.
 * params/grads/bufs: device arrays of n device pointers; sizes: device array of n element counts. */
int b200_sgd_step(float* const* params, const float* const* grads, float* const* bufs,
                  const int64_t* sizes, int n, int64_t max_size, float lr, float momentum,
                  float dampening, float weight_decay, int nesterov, int first_step,
                  const float* inv_scale, const float* found_inf, const float* lr_ptr,
                  b200_stream_t stream);

/* ---- optimizer (torch.optim.Adam / AdamW via get_optimizer('Adam' | 'AdamW', ...)) ---------------------------
 * One launch for `n` tensors; torch's _single_tensor_adam per element, with t = *steps[i] + 1:
 * g = grad (* inv_scale); decoupled ? p *= 1 - lr*wd : g += wd * p (only when wd != 0);
 * m = m + (1-beta1)*(g - m); v = beta2*v + (1-beta2)*g*g; amsgrad: vmax = max(vmax, v), used for v below;
 * p -= (lr / (1 - beta1^t)) * m / (sqrt(v) / sqrt(1 - beta2^t) + eps), the bias corrections in fp64.
 * steps: device array of n pointers to fp32 step counters (torch's fused / capturable state['step']); the launch
 * advances each by one, so a captured graph does at every replay. If found_inf != NULL and *found_inf != 0
 * nothing is written: not parameters, not moments, not steps (GradScaler contract). lr_ptr (device fp32 scalar,
 * may be NULL) overrides lr. max_exp_avg_sqs may be NULL unless amsgrad. tickets: n device uint32 counters,
 * zero on entry and left zero on exit; launches that may run concurrently need separate tickets.
 * params/grads/exp_avgs/exp_avg_sqs/max_exp_avg_sqs/steps: device arrays of n device pointers; sizes: device
 * array of n element counts; max_size: the largest of them. 28 B of HBM traffic per element (36 B with amsgrad). */
int b200_adam_step(float* const* params, const float* const* grads, float* const* exp_avgs,
                   float* const* exp_avg_sqs, float* const* max_exp_avg_sqs, float* const* steps,
                   const int64_t* sizes, int n, int64_t max_size, double lr, double beta1, double beta2,
                   double eps, double weight_decay, int decoupled, int amsgrad, const float* inv_scale,
                   const float* found_inf, const float* lr_ptr, unsigned* tickets, b200_stream_t stream);

/* *counter += 1 on the device (one launch): the per-step tick of the dropout seed offset. */
int b200_tick(uint64_t* counter, b200_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* B200RESNET_H_ */
