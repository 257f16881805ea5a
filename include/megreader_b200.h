/*
 * megreader_b200 — C-ABI of the B200-native OCR hot path (drop-in for MegReader's native ops).
 *
 * Plain pointers and sizes only: no torch / ATen types.  Every pointer is a DEVICE pointer unless
 * the name ends in `_host`.  `stream` is a cudaStream_t passed as void* (NULL = legacy default
 * stream, which is what the reference launches on).  Every entry point returns an mr_status
 * (0 = OK); mr_status_string() gives the reference's error text for it.  Nothing here allocates
 * device memory unless stated; outputs are caller-allocated exactly like the reference's ATen
 * tensors (shapes in each comment).  Functions are asynchronous with respect to the host.
 *
 * The reference interface each entry replaces is cited as file:line under /root/reference.
 */
#ifndef MEGREADER_B200_H
#define MEGREADER_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    MR_OK = 0,
    MR_ERR_NULL_POINTER = 1,
    MR_ERR_BLANK_RANGE = 2,       /* "blank must be in label range"      ctc2d_cuda.cu:40 */
    MR_ERR_TARGET_TOO_LONG = 3,   /* "max target length out of range"    ctc2d_cuda_kernel.cu:220 */
    MR_ERR_BAD_SHAPE = 4,
    MR_ERR_UNSUPPORTED = 5,       /* shape does not fit the on-chip staging of this build */
    MR_ERR_CUDA = 6,              /* a CUDA runtime call failed; see mr_last_cuda_error() */
    MR_ERR_NO_DEVICE = 7
} mr_status;

const char *mr_status_string(int status);
const char *mr_last_cuda_error(void);
/* library/ABI version, bumped when a signature changes */
int mr_abi_version(void);
/* number of kernels this library has launched since load / since the last reset (bench.py's gpu_launches) */
int64_t mr_launch_count(void);
void mr_launch_count_reset(void);

/* ------------------------------------------------------------------------------------------------
 * 2D-CTC  (replaces pybind module ops.ctc_2d.ctc_2d_csrc: ops/ctc_2d/csrc/ctc2d.cpp:3-6)
 *
 * log_probs [T,H,N,C] contiguous; targets [N,S] int64 with element strides (tg_stride_n, tg_stride_s);
 * input_lengths, target_lengths [N] int64; blank in [0,C); 2S+1 <= 1024.
 * ---------------------------------------------------------------------------------------------- */

/* ctc2d_forward: ops/ctc_2d/csrc/ctc2d.h:7-21 -> ctc2d_cuda.cu:30-45 -> ctc2d_cuda_kernel.cu:54-251 (K1).
 * Writes nll [N] and log_alpha [N,T,H,2S+1] (every element is written; no pre-zeroing needed).
 * `fast_math` != 0 uses ex2/lg2.approx (f32 only); 0 uses expf/logf. */
int mr_ctc2d_forward_f32(const float *log_probs, const int64_t *targets, const int64_t *input_lengths,
                         const int64_t *target_lengths, int64_t T, int64_t H, int64_t N, int64_t C, int64_t S,
                         int64_t tg_stride_n, int64_t tg_stride_s, int64_t blank, int fast_math,
                         float *nll, float *log_alpha, void *stream);
int mr_ctc2d_forward_f64(const double *log_probs, const int64_t *targets, const int64_t *input_lengths,
                         const int64_t *target_lengths, int64_t T, int64_t H, int64_t N, int64_t C, int64_t S,
                         int64_t tg_stride_n, int64_t tg_stride_s, int64_t blank, int fast_math,
                         double *nll, double *log_alpha, void *stream);

/* ctc2d_backward: ops/ctc_2d/csrc/ctc2d.h:24-43 -> ctc2d_cuda_kernel.cu:520-629 (K2 + K3, is_large = 0).
 * Writes grad [T,H,N,C] (every element).  grad_out [N] with element stride grad_out_stride.
 * `log_alpha` and `nll` are accepted for signature parity; this implementation re-derives both from
 * log_probs on chip (cheaper than re-reading 2S+1 states per pixel from HBM) and ignores them (may be NULL). */
int mr_ctc2d_backward_f32(const float *grad_out, int64_t grad_out_stride, const float *log_probs,
                          const int64_t *targets, const int64_t *input_lengths, const int64_t *target_lengths,
                          const float *nll, const float *log_alpha,
                          int64_t T, int64_t H, int64_t N, int64_t C, int64_t S,
                          int64_t tg_stride_n, int64_t tg_stride_s, int64_t blank, int fast_math,
                          float *grad, void *stream);
int mr_ctc2d_backward_f64(const double *grad_out, int64_t grad_out_stride, const double *log_probs,
                          const int64_t *targets, const int64_t *input_lengths, const int64_t *target_lengths,
                          const double *nll, const double *log_alpha,
                          int64_t T, int64_t H, int64_t N, int64_t C, int64_t S,
                          int64_t tg_stride_n, int64_t tg_stride_s, int64_t blank, int fast_math,
                          double *grad, void *stream);

/* Training pair used by CTCLoss2DFunction (ops/ctc_2d/ctc_loss_2d.py:7-37) when log_probs.requires_grad:
 * the forward keeps no log_alpha; it writes nll [N] and a per-(t,class) factor `gfac` [T,N,C] such that
 *   grad[t,h,b,c] = exp(log_probs[t,h,b,c]) * gfac[t,b,c] * grad_out[b]        (same values as K3),
 * which mr_ctc2d_backward_apply streams out.  Total HBM traffic 3*|log_probs| instead of
 * 3*|log_probs| + 2*|log_alpha| (SURVEY.md §8d). */
int mr_ctc2d_forward_train_f32(const float *log_probs, const int64_t *targets, const int64_t *input_lengths,
                               const int64_t *target_lengths, int64_t T, int64_t H, int64_t N, int64_t C, int64_t S,
                               int64_t tg_stride_n, int64_t tg_stride_s, int64_t blank, int fast_math,
                               float *nll, float *gfac, void *stream);
int mr_ctc2d_backward_apply_f32(const float *grad_out, int64_t grad_out_stride, const float *log_probs,
                                const float *gfac, int64_t T, int64_t H, int64_t N, int64_t C, int fast_math,
                                float *grad, void *stream);

/* Fused epilogue of the 2D-CTC head (decoders/ctc_decoder2d.py:37-45): from the two conv branches' raw outputs
 *   mask_logits [N,1,H,W] (before nn.Softmax(dim=2), :21) and cls_logits [N,C,H,W] (before softmax(dim=1), :41)
 * straight to log_probs [W,H,N,C] = log(max(softmax_H(mask) * softmax_C(cls), tiny)).permute(3,2,0,1)   (fp32).
 * Backward: either the explicit gradient grad_log_probs [W,H,N,C], or (grad_log_probs = NULL) the 2D-CTC training
 * factor gfac [W,N,C] + grad_out [N] of mr_ctc2d_forward_train_f32, so that d(log_probs) never exists in HBM.
 * Outputs grad_cls_logits [N,C,H,W], grad_mask_logits [N,1,H,W].  MR_ERR_UNSUPPORTED for charsets too large for the
 * shared-memory tile (C > ~750 forward). */
int mr_ctc2d_head_fwd_f32(const float *mask_logits, const float *cls_logits, int N, int C, int H, int W, float tiny,
                          float *log_probs, void *stream);
int mr_ctc2d_head_bwd_f32(const float *mask_logits, const float *cls_logits, const float *grad_log_probs, const float *gfac,
                          const float *grad_out, int64_t grad_out_stride, int N, int C, int H, int W, float tiny,
                          float *grad_cls_logits, float *grad_mask_logits, void *stream);

/* ------------------------------------------------------------------------------------------------
 * 1D CTC head of the CRNN decoder (replaces the `log_softmax -> nn.CTCLoss(zero_infinity=True)` call,
 * decoders/crnn.py:47-48,95-99; arithmetic restated in decoders/ctc_loss.py:65-122).  fp32.
 * ---------------------------------------------------------------------------------------------- */
/* out[r,:] = log_softmax(x[r,:]) for `rows` rows of C classes (decoders/crnn.py:96). */
int mr_log_softmax_rows_f32(const float *x, int64_t rows, int64_t C, float *out, void *stream);
/* log_probs [T,N,C]; writes nll [N] (raw, may be +inf) and gfac [T,N,C] with aten's gradient convention:
 * d nll_b / d log_probs[t,b,c] = exp(lp) * gfac   (0 for t >= input_length, and for nll=+inf when zero_infinity). */
int mr_ctc1d_forward_train_f32(const float *log_probs, const int64_t *targets, const int64_t *input_lengths,
                               const int64_t *target_lengths, int64_t T, int64_t N, int64_t C, int64_t S,
                               int64_t tg_stride_n, int64_t tg_stride_s, int64_t blank, int zero_infinity,
                               int fast_math, float *nll, float *gfac, void *stream);
/* grad_logits [T,N,C] = scale[b] * log_softmax_backward(exp(lp) * gfac): the CTC gradient pushed through the
 * log_softmax, scale[b] = upstream gradient of nll_b (1 / (N * target_length) for the 'mean' reduction). */
int mr_ctc1d_backward_logits_f32(const float *log_probs, const float *gfac, const float *scale, int64_t T, int64_t N,
                                 int64_t C, float *grad_logits, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Deformable convolution v1 / v2  (replaces pybind module assets.ops.dcn.deform_conv_cuda:
 * assets/ops/dcn/src/deform_conv_cuda.cpp:681-695).  fp32, NCHW contiguous input [B,C,H,W] and weight
 * [Cout, C/group, kh, kw].  offset / mask (and their gradients) are addressed per sample as
 * base + b*bstride (elements) and then FLAT with (Ho, Wo) strides, as the reference kernels do
 * (deform_conv_cuda_kernel.cu:599-609) — the caller's tensors may have a larger spatial size.
 * mask == NULL selects DCNv1 (deform_conv_forward_cuda & co., deform_conv_cuda.cpp:151-484).
 * `workspace` is caller-allocated scratch for the column matrix: at least
 * mr_dcn_workspace_bytes(1, ...) bytes; with room for nb samples the op processes nb samples per launch.
 * The GEMMs are cuBLAS SGEMM (plain fp32); the first call per device creates a cuBLAS handle (which
 * allocates cuBLAS's own workspace).
 * ---------------------------------------------------------------------------------------------- */
int64_t mr_dcn_workspace_bytes(int64_t nb, int64_t C, int64_t kh, int64_t kw, int64_t Ho, int64_t Wo);

/* modulated_deform_conv_cuda_forward (deform_conv_cuda.cpp:486-564) / deform_conv_forward_cuda (:151-258).
 * Writes output [B,Cout,Ho,Wo] (+bias when bias != NULL). */
int mr_dcn_forward_f32(const float *input, const float *weight, const float *bias, const float *offset,
                       int64_t offset_bstride, const float *mask, int64_t mask_bstride, float *output,
                       float *workspace, int64_t workspace_bytes, int B, int C, int H, int W, int Cout, int kh, int kw,
                       int sh, int sw, int ph, int pw, int dh, int dw, int group, int dg, void *stream);

/* Fused forward (csrc/dcn_tcgen05.cu): the same result as mr_dcn_forward_f32 without a column matrix in HBM -- one tcgen05
 * implicit GEMM whose A operand is the bilinear gather itself (bf16 hi/lo split, three MMAs per K block: fp32-level accuracy).
 * group = deformable_group = 1, C % 64 == 0, Cout % 128 == 0; workspace >= mr_dcn_fused_workspace_bytes(...) (NHWC copy of
 * the input + packed weights), 256-byte aligned.  Returns MR_ERR_UNSUPPORTED otherwise; mr_dcn_forward_f32 tries it first. */
int64_t mr_dcn_fused_workspace_bytes(int64_t B, int64_t C, int64_t H, int64_t W, int64_t Cout, int64_t kh, int64_t kw);
int mr_dcn_forward_fused_f32(const float *input, const float *weight, const float *bias, const float *offset,
                             int64_t offset_bstride, const float *mask, int64_t mask_bstride, float *output,
                             float *workspace, int64_t workspace_bytes, int B, int C, int H, int W, int Cout, int kh, int kw,
                             int sh, int sw, int ph, int pw, int dh, int dw, int group, int dg, void *stream);

/* Fused weight gradient (csrc/dcn_tcgen05.cu), the deform_conv_cuda.cpp:645-658 step (im2col + SGEMM per sample in the reference)
 * as one tcgen05 GEMM over the pixels whose B operand is the bilinear gather itself: grad_weight += scale * go (*) columns.
 * Same eligibility as the fused forward; workspace >= mr_dcn_fused_wgrad_workspace_bytes(...).  mr_dcn_backward_f32 tries it first. */
int64_t mr_dcn_fused_wgrad_workspace_bytes(int64_t B, int64_t C, int64_t H, int64_t W, int64_t Cout, int64_t Ho, int64_t Wo);
int mr_dcn_wgrad_fused_f32(const float *input, const float *offset, int64_t offset_bstride, const float *mask, int64_t mask_bstride,
                           const float *grad_output, float *grad_weight, float scale, float *workspace, int64_t workspace_bytes,
                           int B, int C, int H, int W, int Cout, int kh, int kw, int sh, int sw, int ph, int pw, int dh, int dw,
                           int group, int dg, void *stream);

/* Fused backward (csrc/dcn_tcgen05.cu): the weight gradient above plus the data gradient -- the deform_conv_cuda.cpp:611-614 SGEMM
 * (W^T . grad_output) and the K9 / K10 kernels (deform_conv_cuda_kernel.cu:634-766) as one tcgen05 kernel whose epilogue scatters
 * grad_input and reduces grad_offset / grad_mask, no column-gradient matrix in HBM.  group = deformable_group = 1, C % 128 == 0,
 * Cout % 128 == 0; workspace >= mr_dcn_fused_backward_workspace_bytes(...).  Same argument meaning as mr_dcn_backward_f32 (without
 * grad_bias); returns MR_ERR_UNSUPPORTED otherwise; mr_dcn_backward_f32 tries it first. */
int64_t mr_dcn_fused_backward_workspace_bytes(int64_t B, int64_t C, int64_t H, int64_t W, int64_t Cout, int64_t Ho, int64_t Wo,
                                              int64_t kh, int64_t kw);
int mr_dcn_backward_fused_f32(const float *input, const float *weight, const float *offset, int64_t offset_bstride, const float *mask,
                              int64_t mask_bstride, const float *grad_output, float *grad_input, float *grad_weight,
                              float *grad_offset, int64_t grad_offset_bstride, float *grad_mask, int64_t grad_mask_bstride,
                              float weight_grad_scale, float *workspace, int64_t workspace_bytes, int B, int C, int H, int W, int Cout,
                              int kh, int kw, int sh, int sw, int ph, int pw, int dh, int dw, int group, int dg, void *stream);

/* modulated_deform_conv_cuda_backward (deform_conv_cuda.cpp:566-679) / deform_conv_backward_input_cuda (:260-371)
 * + deform_conv_backward_parameters_cuda (:373-484).  grad_input / grad_weight / grad_bias are ACCUMULATED into
 * (the caller zero-fills them, functions/deform_conv.py:150-154); grad_offset / grad_mask entries are assigned with
 * the flat (Ho,Wo) layout.  Any of the five gradient pointers may be NULL to skip it.  weight_grad_scale is the
 * `scale` of deform_conv_backward_parameters_cuda (1 for DCNv2). */
int mr_dcn_backward_f32(const float *input, const float *weight, const float *offset, int64_t offset_bstride,
                        const float *mask, int64_t mask_bstride, const float *grad_output, float *grad_input,
                        float *grad_weight, float *grad_bias, float *grad_offset, int64_t grad_offset_bstride,
                        float *grad_mask, int64_t grad_mask_bstride, float weight_grad_scale, float *workspace,
                        int64_t workspace_bytes, int B, int C, int H, int W, int Cout, int kh, int kw, int sh, int sw,
                        int ph, int pw, int dh, int dw, int group, int dg, void *stream);

/* ------------------------------------------------------------------------------------------------
 * CRNN training engine building blocks (replace the ATen / cuDNN composition behind backbones/crnn.py:46-59 and
 * decoders/crnn.py:8-24,80-104).  Activations are NHWC ("rows" = N*H*W pixels x C channels); dtype codes:
 * 0 = float32, 1 = bfloat16.  Vector kernels need C % 4 == 0 (fp32) / C % 8 == 0 (bf16).
 * ---------------------------------------------------------------------------------------------- */
int mr_nchw_to_nhwc(const float *x, int N, int C, int H, int W, int Cp, int dtype, void *y, void *stream);
int mr_nhwc_to_nchw(const void *x, int N, int C, int H, int W, int Cp, int dtype, float *y, void *stream);
/* stride-1 convolution lowering: col [N*Ho*Wo, Kp], column (i*kw + j)*C + c; columns >= kh*kw*C are zero. */
int mr_im2col_nhwc(const void *x, int N, int H, int W, int C, int kh, int kw, int ph, int pw, int Kp, int dtype,
                   void *col, void *stream);
int mr_col2im_nhwc(const void *dcol, int N, int H, int W, int C, int kh, int kw, int ph, int pw, int Kp, int dtype,
                   void *dx, void *stream);
/* conv epilogue fused with nn.MaxPool2d(k, s, p): y = maxpool(relu(x + bias)); idx = first arg-max (uint8). */
int mr_bias_relu_pool_fwd(const void *x, const float *bias, int N, int H, int W, int C, int kh, int kw, int sh, int sw,
                          int ph, int pw, int dtype, void *y, unsigned char *idx, void *stream);
/* backward also returns the conv-bias gradient dbias[C] = column sums of dz (fused; `sums` = scratch of C doubles);
 * dbias may be NULL. */
int mr_bias_relu_pool_bwd(const void *dy, const void *y, const unsigned char *idx, int N, int H, int W, int C, int kh,
                          int kw, int sh, int sw, int ph, int pw, int dtype, void *dz, float *dbias, double *sums,
                          void *stream);
int mr_bias_act(const void *x, const float *bias, int64_t rows, int C, int relu, int dtype, void *y, void *stream);
/* nn.BatchNorm2d in training mode over (x + bias): batch stats, running-stat update, normalise; `sums` = scratch of
 * 2*C doubles.  mr_bn_apply is the eval-mode affine transform with given mean / invstd. */
int mr_bn_train_fwd(const void *x, const float *bias, const float *gamma, const float *beta, float *running_mean,
                    float *running_var, float momentum, float eps, int64_t rows, int C, int dtype, void *y, float *mean,
                    float *invstd, double *sums, void *stream);
int mr_bn_apply(const void *x, const float *bias, const float *mean, const float *invstd, const float *gamma,
                const float *beta, int64_t rows, int C, int dtype, void *y, void *stream);
/* backward: `sums` = scratch of 3*C doubles; dbias (nullable) = column sums of dx (gradient of the conv bias). */
int mr_bn_train_bwd(const void *dy, const void *x, const float *bias, const float *mean, const float *invstd,
                    const float *gamma, int64_t rows, int C, int dtype, void *dx, float *dgamma, float *dbeta,
                    float *dbias, double *sums, void *stream);
/* out[c] (= or +=) sum_r a[r,c] (bias gradients); `sums` = scratch of 2*C doubles. */
int mr_colsum(const void *a, int64_t rows, int C, int dtype, float *out, int accumulate, double *sums, void *stream);
/* nn.LSTM cell, gate order i,f,g,o; one launch advances `ndir` (1 or 2) directions of a bidirectional layer; the
 * per-direction arguments are HOST arrays of `ndir` device pointers.  fwd: gates [B,4H] pre-activations in,
 * activations out (in place); c_prev[d] may be NULL (first step).  bwd: c_prev[d] / dh_rec[d] may be NULL. */
int mr_lstm_cell_fwd(void *const *gates, const float *const *b_ih, const float *const *b_hh, const float *const *c_prev,
                     float *const *c_out, void *const *h_out, int64_t ldh, void *const *h_state, int ndir, int B, int H,
                     int dtype, void *stream);
int mr_lstm_cell_bwd(const void *const *gates, const float *const *c, const float *const *c_prev,
                     const void *const *dh_out, int64_t ldh, const void *const *dh_rec, float *const *dc,
                     void *const *dgates, int ndir, int B, int H, int dtype, void *stream);
/* torch.optim.Adam step over one flat fp32 buffer (training/optimizer_scheduler.py:17-22 builds torch.optim.Adam). */
int mr_adam_step(float *p, const float *g, float *m, float *v, int64_t n, float lr, float beta1, float beta2, float eps,
                 int64_t step, float grad_scale, void *bf16_shadow, void *stream);
int mr_cast(const void *x, int src_dtype, int64_t n, int dst_dtype, void *y, void *stream);
/* Row-major C[M,N] = alpha * op(A) op(B) + beta * C, fp32 accumulate (plain library GEMM: cuBLAS). */
int mr_gemm(const void *A, const void *B, void *C, int64_t M, int64_t N, int64_t K, int64_t lda, int64_t ldb,
            int64_t ldc, int transA, int transB, int in_dtype, int out_dtype, float alpha, float beta, void *stream);
int mr_gemm_batched(const void *A, const void *B, void *C, int64_t M, int64_t N, int64_t K, int64_t lda, int64_t ldb,
                    int64_t ldc, int64_t strideA, int64_t strideB, int64_t strideC, int batch, int transA, int transB,
                    int in_dtype, int out_dtype, float alpha, float beta, void *stream);

/* Hand-written Blackwell GEMM (tcgen05.mma + TMEM accumulators + TMA operand staging), bf16 in / fp32 accumulate.
 * Same storage convention as mr_gemm; supported forms (transA,transB) = (0,1) and (1,0); optional per-column bias
 * and ReLU in the epilogue; beta = 1 accumulates atomically into fp32 C and enables split-K.  Returns
 * MR_ERR_UNSUPPORTED for shapes / alignments it does not cover (the caller then uses mr_gemm). */
int mr_gemm_tcgen05(const void *A, const void *B, void *C, int64_t M, int64_t N, int64_t K, int64_t lda, int64_t ldb,
                    int64_t ldc, int transA, int transB, int out_dtype, const float *bias, int relu, float beta,
                    int splits, void *stream);

/* Implicit-GEMM stride-1 convolution (nn.Conv2d of backbones/crnn.py:46-49) on NHWC bf16, tcgen05 + TMA + gathered
 * activation tiles: y[N*Ho*Wo, Cout] = conv(x[N,H,W,C], Wm[Cout, kh*kw*C]) (+bias, ReLU); C % 64 == 0.  With
 * flipped/transposed weights and padding (k-1-p) the same entry computes the input gradient. */
int mr_conv_fprop_tcgen05(const void *x, const void *Wm, void *y, int N, int H, int W, int C, int Cout, int kh, int kw,
                          int ph, int pw, int out_dtype, const float *bias, int relu, void *stream);
/* General forms with stride and dilation (the trunk convolutions of backbones/resnet.py:110-256, resnet_dilated.py:50-69,
 * ppm.py:6-44, fpn_top_down.py:6-30 and the 2D-CTC head branches decoders/ctc_decoder2d.py:16-27): same kernels, the stride is
 * the activation tensor map's traversal stride, the dilation scales the tap's coordinate offset. */
int mr_conv2d_fprop_tcgen05(const void *x, const void *Wm, void *y, int N, int H, int W, int C, int Cout, int kh, int kw,
                            int sh, int sw, int ph, int pw, int dh, int dw, int out_dtype, const float *bias, int relu,
                            void *stream);
int mr_conv2d_wgrad_tcgen05(const void *dz, const void *x, float *dWm, int N, int H, int W, int C, int Cout, int kh, int kw,
                            int sh, int sw, int ph, int pw, int dh, int dw, int splits, void *stream);
/* Implicit-GEMM weight gradient: dWm[Cout, kh*kw*C] fp32 += dz[N,Ho,Wo,Cout]^T (*) x[N,H,W,C] (atomic, split-K). */
int mr_conv_wgrad_tcgen05(const void *dz, const void *x, float *dWm, int N, int H, int W, int C, int Cout, int kh, int kw,
                          int ph, int pw, int splits, void *stream);

/* Fused LSTM time steps on tcgen05 (recurrent GEMM + cell in one launch, both directions): gate columns are
 * UNIT-MAJOR (column 4*j + g = gate g in {i,f,g,o} of hidden unit j), H % 64 == 0, bf16.  Every per-direction argument
 * is a HOST array of 2 device pointers.  fwd: gates[d] [B,4H] holds the x-projection on entry and the activated gates
 * on exit; bias[d] [4H] = b_ih + b_hh (unit-major); have_h = 0 on the first step.  bwd: dG_next[d] = gate gradients of
 * the step processed just before (have_rec = 0 on the first backward step); dc[d] [B,H] is updated in place. */
int mr_lstm_step_fwd_tcgen05(const void *const *h_prev, const void *const *Whh, void *const *gates,
                             const float *const *bias, const float *const *c_prev, float *const *c_out,
                             void *const *h_out, int64_t ldh, void *const *h_next, int have_h, int B, int H,
                             void *stream);
int mr_lstm_step_bwd_tcgen05(const void *const *dG_next, const void *const *Whh, const void *const *gates,
                             const float *const *c, const float *const *c_prev, const void *const *dh_out, int64_t ldh,
                             float *const *dc, void *const *dgates, int have_rec, int B, int H, void *stream);

/* Whole-sequence recurrence of ONE bidirectional LSTM layer in a single persistent launch (csrc/lstm_seq_tcgen05.cu):
 * replaces the T per-step launches of the cuDNN LSTM the reference calls (decoders/crnn.py:13,17 nn.LSTM;
 * SURVEY.md section 8 A7).  bf16 operands, unit-major gate columns, H % 64 == 0.
 *   Whh   : HOST array of 2 device pointers, [4H, H] bf16 unit-major rows (direction 0 = forward in time, 1 = reverse)
 *   G     : [2, T, B, 4H] bf16 -- x-projection on entry, activated gates (i,f,g,o) on exit
 *   bias  : HOST array of 2 device pointers, [4H] fp32 unit-major (b_ih + b_hh)
 *   C     : [2, T, B, H] fp32 cell states, out;   Y : [T, B, 2H] bf16 layer output, out (direction d -> columns d*H..)
 *   flags : [2*ceil(B/128) + 1] uint32 scratch (zeroed by the call); after completion the last word is 0, or a non-zero
 *           code if an inter-CTA wait timed out (results then undefined)
 * bwd:  dY [T, B, 2H] bf16 -> dG [2, T, B, 4H] bf16 gate gradients (the weight/input gradients are plain GEMMs on dG);
 *       WhhT = the recurrent weights TRANSPOSED, HOST array of 2 device pointers to [H, 4H] bf16 (unit-major columns).
 * MR_ERR_UNSUPPORTED when the CTA grid cannot be co-resident on this device or H exceeds the shared-memory budget
 * (fwd H <= 512, bwd H <= 256): callers then use the per-step entry points above. */
int mr_lstm_seq_fwd_tcgen05(const void *const *Whh, void *G, const float *const *bias, float *C, void *Y,
                            unsigned *flags, int T, int B, int H, void *stream);
int mr_lstm_seq_bwd_tcgen05(const void *const *WhhT, const void *G, const float *C, const void *dY, void *dG,
                            unsigned *flags, int T, int B, int H, void *stream);
/* Development aid: device buffer [T][32] of int64 clock stamps written by CTA (0,0,0) of the next mr_lstm_seq_* launches
 * (NULL switches it off); slot meaning in csrc/lstm_seq_tcgen05.cu. */
int mr_lstm_seq_set_trace(void *buf);

/* Deformable position-sensitive RoI pooling (assets/ops/dcn/src/deform_pool_cuda.cpp:29-81 ->
 * deform_pool_cuda_kernel.cu:52-263; python surface functions/deform_pool.py:7-69).  fp32.
 *   data [batch, channels, H, W]; rois [num_rois, 5] = (image index, x1, y1, x2, y2); trans [num_rois, channels_trans,
 *   part, part] (ignored when no_trans); out / top_count [num_rois, output_dim, pooled, pooled] (top_count = number of
 *   in-range samples per bin, float, consumed by the backward).  backward ACCUMULATES into in_grad / trans_grad. */
int mr_deform_psroi_pool_forward_f32(const float *data, const float *rois, const float *trans, int batch, int channels,
                                     int height, int width, int num_rois, int channels_trans, int no_trans,
                                     float spatial_scale, int output_dim, int group_size, int pooled_size, int part_size,
                                     int sample_per_part, float trans_std, float *out, float *top_count, void *stream);
int mr_deform_psroi_pool_backward_f32(const float *out_grad, const float *data, const float *rois, const float *trans,
                                      const float *top_count, int batch, int channels, int height, int width, int num_rois,
                                      int channels_trans, int no_trans, float spatial_scale, int output_dim, int group_size,
                                      int pooled_size, int part_size, int sample_per_part, float trans_std, float *in_grad,
                                      float *trans_grad, void *stream);

/* Recognition input step on the GPU (SURVEY.md section 8 row N3; data/processes/resize_image.py:29-57 modes "resize" / "pad",
 * normalize_image.py:10-17, make_recognition_label.py:13-32): a ragged batch of decoded HWC 3-channel images (uint8 or fp32)
 * -> cv2.resize-equivalent bilinear resize to [dst_h, valid_w[n]] at the left of a zero [dst_h, dst_w] canvas, minus
 * mean3 (float64, host pointer), / 255, CHW fp32 [N,3,dst_h,dst_w]; and label byte strings -> class indices through a
 * 256-entry table, blank-padded to max_size, with lengths = min(len, max_size).  Array arguments live on the device. */
int mr_resize_normalize_f32(const void *src, int src_is_u8, const int64_t *offsets, const int *heights, const int *widths,
                            const int *valid_w, int N, int dst_h, int dst_w, const double *mean3_host, float *out,
                            void *stream);
int mr_pack_labels(const unsigned char *text, const int64_t *offsets, int N, const int *lut, int max_size, int *labels,
                   int *lengths, void *stream);

/* Weight layout packs of the training engine (one launch instead of permute / pad / flip / gather / cast chains).
 * mr_conv_weight_pack: nn.Conv2d weight [Cout,Cin,kh,kw] fp32 (backbones/crnn.py:37-44) -> GEMM operand in `dtype`:
 *   mode 0: forward matrix [Cout, Kp], column (i*kw + j)*Cp + c, zero padded (Cp >= Cin, Kp >= kh*kw*Cp);
 *   mode 1: input-gradient matrix [Cin, kh*kw*Cout], taps flipped and (Cout,Cin) transposed.
 * mr_gate_rows_permute: nn.LSTM weight / bias rows [4H, cols] fp32 between the reference's gate-major order (i|f|g|o
 *   blocks) and the unit-major order of the tcgen05 LSTM kernels; `b` (nullable) is added (b_ih + b_hh). */
int mr_conv_weight_pack(const float *w, int Cout, int Cin, int kh, int kw, int Cp, int Kp, int mode, int dtype, void *out,
                        void *stream);
int mr_gate_rows_permute(const float *a, const float *b, int H, int cols, int inverse, int dtype, void *out, void *stream);

/* Greedy CTC decoding to label indices (structure/representers/ctc_representer.py:22-34, ctc_representer2d.py:27-51):
 * arg-max class per column (2D: along the arg-max-height path of classify*mask), then collapse repeats / skip
 * `unknown` / drop blanks.  prob strides (sN,sC,sH,sW) in elements; mask nullable with strides (mN,mH,mW).
 * out int32 [N,W] blank-padded.  mr_blank_after_first_blank: sequence_recognition_representer.py:23-28. */
int mr_ctc_greedy_decode(const float *prob, const float *mask, int N, int C, int H, int W, int64_t sN, int64_t sC,
                         int64_t sH, int64_t sW, int64_t mN, int64_t mH, int64_t mW, int blank, int unknown, int *out,
                         void *stream);
int mr_blank_after_first_blank(int *pred, int N, int W, int blank, void *stream);

/* ---- attention recogniser head: the greedy decoding loop (decoders/attention_decoder.py:119-131, AttentionRNNCell.forward :187-231)
 * as ONE persistent cooperative kernel (csrc/attn_decode.cu).  All tensors fp32, contiguous unless a stride is given:
 *   projected [N][L][H]   = attn.attn.weight[:, H:] . memory + attn.attn.bias   (step-invariant half of the energies, caller-computed)
 *   memory    [N][L][H+E] = encoder grid with the position one-hots appended (decoder_input of the reference, batch-major)
 *   wa_h      H rows of ld_wa floats = attn.attn.weight[:, :H];  v [H] = attn.v
 *   wordtab   [V][H]      = word_linear(embedding.weight)  (row w = the embedded previous symbol w)
 *   w_ih [3H][2H+E], b_ih [3H], w_hh [3H][H], b_hh [3H] = decoder.rnn (GRUCell, gates r, z, n);  w_out [V][H], b_out [V] = decoder.out
 * Output pred [N][S] (argmax per step, int32; the reference's early exit is applied by the caller) and, if prob != NULL, the per-step
 * softmax [N][S][V].  workspace >= mr_attn_decode_workspace_bytes(N, H, E), 256-byte aligned.  mr_attn_decode_status reads back the
 * error word (non-zero: a grid barrier timed out and the results are invalid). */
int64_t mr_attn_decode_workspace_bytes(int64_t N, int64_t H, int64_t E);
int mr_attn_decode_f32(const float *projected, const float *memory, const float *wa_h, int64_t ld_wa, const float *v,
                       const float *wordtab, const float *w_ih, const float *b_ih, const float *w_hh, const float *b_hh,
                       const float *w_out, const float *b_out, int *pred, float *prob, void *workspace, int64_t workspace_bytes,
                       int N, int L, int H, int E, int V, int S, int blank, void *stream);
int mr_attn_decode_status(const void *workspace, int64_t N, int64_t H, int64_t E, void *stream, int *status);

/* ---- attention recogniser head: the TRAINING loop (decoders/attention_decoder.py:96-117 around AttentionRNNCell.forward :187-231) as
 * one persistent cooperative kernel per direction (csrc/attn_decode.cu).  Inputs as for mr_attn_decode_f32, plus
 *   targets [N][S] int32, lengths [N] int32 (the per-step NLL counts while step <= lengths[n], attention_decoder.py:104)
 *   coin [S] int32 (1: the target is fed back, 0: the step's own argmax -- the reference's `gt_as_output` draw, :51-54, :107-110)
 *   swap, noise [S][N] int32 (step dropout, :111-116: where swap is 1 the fed-back symbol is replaced by noise)
 * The caller makes the random draws on the host in the reference's order.  Outputs: loss [N] (sum over the steps), attn [N][S][L]
 * (the attention maps the reference returns) and the per-step state the backward needs:
 *   h_all [S+1][N][H] (slice t = hidden state after t steps), fh_all [S][N][H] (= Wa_h . h), x_all [S][N][Xp] (GRU inputs, row stride
 *   Xp = 2H+E rounded up to a multiple of 4 floats; H % 4 == 0 is required),
 *   gates [S][N][4][H] (r, z, n, W_hn h + b_hn), logp [S][N][V] (log-softmax of the step outputs), word [S][N] (symbol fed into step t).
 * sync: 2 x uint32 scratch (arrival counter, error word: mr_attn_sync_status). */
int mr_attn_train_fwd_f32(const float *projected, const float *memory, const float *wa_h, int64_t ld_wa, const float *v,
                          const float *wordtab, const float *w_ih, const float *b_ih, const float *w_hh, const float *b_hh,
                          const float *w_out, const float *b_out, const int *targets, const int *lengths, const int *coin,
                          const int *swap, const int *noise, float *h_all, float *fh_all, float *x_all, float *gates, float *logp,
                          float *attn, int *word, float *loss, void *sync, int N, int L, int H, int E, int V, int S, int blank,
                          void *stream);
/* Backward through time of the loop above for the upstream gradient grad_loss [N] of `loss`.  Written (zero-filled here first):
 *   dprojected [N][L][H], dmemory [N][L][H+E], dv [H], dwordtab [V][H]                  -- complete gradients
 *   dlogits [S][N][V], dgi / dgh [S][N][3H], dfh [S][N][H]                              -- per-step pre-activation gradients; the weight
 *       gradients are plain dense products over the S*N rows, left to the caller:  dW_out = dlogits^T . h_all[1:],  dW_ih = dgi^T . x_all[:, :, :2H+E],
 *       dW_hh = dgh^T . h_all[:-1],  dWa_h = dfh^T . h_all[:-1],  the bias gradients are the column sums of dlogits / dgi / dgh
 *   dx [N][2H+E], dh [N][H]                                                              -- scratch */
int mr_attn_train_bwd_f32(const float *projected, const float *memory, const float *wa_h, int64_t ld_wa, const float *v,
                          const float *w_ih, const float *w_hh, const float *w_out, const float *h_all, const float *fh_all,
                          const float *gates, const float *logp, const float *attn, const int *word, const int *targets,
                          const int *lengths, const float *grad_loss, float *dlogits, float *dgi, float *dgh, float *dfh, float *dx,
                          float *dh, float *dprojected, float *dmemory, float *dv, float *dwordtab, void *sync, int N, int L, int H,
                          int E, int V, int S, void *stream);
int mr_attn_sync_status(const void *sync, void *stream, int *status);

/* ------------------------------------------------------------------------------------------------
 * DB text detector: SegDetector's probability maps and L1BalanceCELoss (decoders/seg_detector.py:117-147,
 * decoders/seg_detector_loss.py:157-185, balance_cross_entropy_loss.py:40-54, dice_loss.py:31-42, l1_loss.py:9-11).
 * fp32 maps, fp32 element math, fp64 sums.  Every map is contiguous.
 * ---------------------------------------------------------------------------------------------- */

/* b = sigmoid(x_b), t = sigmoid(x_t), tb = 1 / (1 + exp(-k (b - t))), n elements each (accurate expf). */
int mr_db_maps_fwd_f32(const float *x_b, const float *x_t, int64_t n, float k, float *b, float *t, float *tb, void *stream);
/* Gradients of the maps above from the saved b, t, tb; any of grad_b / grad_t / grad_tb may be NULL (= zero). */
int mr_db_maps_bwd_f32(const float *grad_b, const float *grad_t, const float *grad_tb, const float *b, const float *t,
                       const float *tb, int64_t n, float k, float *grad_xb, float *grad_xt, void *stream);
/* Bytes of the loss workspace for N samples of HW pixels: 8 per (sample, pixel) plus a fixed ~84 KB. */
int64_t mr_db_loss_workspace_bytes(int64_t N, int64_t HW);
/* L1BalanceCELoss forward without host synchronisation.  b, t, tb, gt: (N,1,H,W); mask, thresh_map, thresh_mask: (N,H,W);
 * gt and mask take values in [0, 1]; 1 <= N <= 256.  Writes out[4] = (loss, bce_loss, thresh_loss (dice), l1_loss) and
 * keeps in `workspace` what mr_db_loss_bwd_f32 reads (pass the same workspace, unmodified, to the backward). */
int mr_db_loss_fwd_f32(const float *b, const float *t, const float *tb, const float *gt, const float *mask,
                       const float *thresh_map, const float *thresh_mask, int64_t N, int64_t HW, float eps,
                       float l1_scale, float bce_scale, float negative_ratio, float bce_eps, void *workspace,
                       int64_t workspace_bytes, float *out, void *stream);
/* Backward for the upstream gradients grad_out[4] of the four outputs (device memory): writes grad_b, grad_t, grad_tb
 * (N,HW) each.  Among the copies tied at the selection threshold the remainder is split evenly. */
int mr_db_loss_bwd_f32(const float *grad_out, const float *b, const float *t, const float *gt, const float *mask,
                       const float *thresh_map, const float *thresh_mask, int64_t N, int64_t HW, float l1_scale,
                       float bce_scale, const void *workspace, int64_t workspace_bytes, float *grad_b, float *grad_t,
                       float *grad_tb, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MEGREADER_B200_H */
