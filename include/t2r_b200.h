/*
 * t2r_b200.h — C-ABI of libt2r_b200.so: the B200 (sm_100a) kernels underneath the
 * Tensor2Robot per-replay-batch hot path (SURVEY.md §8 B-2).
 *
 * The reference (google-research/tensor2robot) has no FFI: every hot-path op is a
 * TensorFlow library call made from Python.  Each entry point below therefore cites the
 * reference *call site* (file:line under /root/reference) whose arithmetic it replaces.
 *
 * Conventions
 *   - extern "C", plain C types only.  Every function returns int32 status (0 = OK,
 *     negative = T2R_ERR_*); t2r_last_error() returns a thread-local message.
 *   - No hidden allocation: the caller (PyTorch caching allocator) owns every device and
 *     pinned buffer.  Functions never synchronise; `stream` is a cudaStream_t passed as void*.
 *   - Activations are NHWC ("channels last"), bf16 unless stated; parameters/optimizer
 *     state are fp32; conv weights are OHWI ([Cout][KH][KW][Cin]).
 *   - Descriptors are POD structs versioned by a leading uint32 struct_size.
 */
#ifndef T2R_B200_H_
#define T2R_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define T2R_OK 0
#define T2R_ERR_INVALID_ARG (-1)
#define T2R_ERR_CUDA (-2)
#define T2R_ERR_UNSUPPORTED (-3)
#define T2R_ERR_PARSE (-4)
#define T2R_ERR_IO (-5)

/* ---- library ------------------------------------------------------------------------ */
int32_t t2r_version(void);
const char* t2r_last_error(void);
/* Number of kernels launched by this library in this process (bench.py "gpu_launches"). */
int64_t t2r_launch_count(void);
void t2r_launch_count_reset(void);

/* ---- convolution / GEMM on tcgen05 tensor cores -------------------------------------- */
/* Replaces slim.conv2d / tf.layers.conv2d / slim.fully_connected call sites:
 *   research/qtopt/networks.py:443-591 (Grasping44 convs, fc0/fc1),
 *   layers/film_resnet_model.py:89-105 (conv2d_fixed_padding), :618 (final dense).
 * Implicit GEMM: M = N*Ho*Wo output pixels, N = Cout, K = KH*KW*Cin; bf16 operands staged by
 * TMA into 128B-swizzled shared memory, fp32 accumulation in TMEM. */
#define T2R_EPI_BIAS 1      /* y += bias[c]                       */
#define T2R_EPI_RESIDUAL 2  /* y += residual (same shape as y)     */
#define T2R_EPI_RELU 4      /* y = max(y, 0)                       */
#define T2R_EPI_OUT_F32 8   /* y written as fp32 instead of bf16   */

typedef struct T2RConvDesc {
  uint32_t struct_size;
  int32_t N, H, W, Cin;   /* input  [N,H,W,Cin]                               */
  int32_t Cout, KH, KW;   /* filter [Cout,KH,KW,Cin]                          */
  int32_t stride;         /* 1 or 2, same in both dims                        */
  int32_t pad_top, pad_left; /* zero padding before the first row / column    */
  int32_t Ho, Wo;         /* output [N,Ho,Wo,Cout]; end padding is implied    */
  int32_t flags;          /* T2R_EPI_* (fprop only)                           */
} T2RConvDesc;

/* TF padding arithmetic (SURVEY §8c-1): SAME => out=ceil(in/s), pad_before=pad_total/2. */
int32_t t2r_conv_same_padding(int32_t in, int32_t k, int32_t stride, int32_t* out,
                              int32_t* pad_before);

/* y = conv(x, w) (+bias)(+residual)(relu).  Requires Cin % 64 == 0, Cout % 64 == 0. */
int32_t t2r_conv2d_fprop(const T2RConvDesc* d, const void* x, const void* w_ohwi,
                         const float* bias, const void* residual, void* y, void* stream);
/* Same, and the epilogue also accumulates the batch-norm statistics of the bf16 output it writes:
 * stats[c] += sum_rows y[.,c], stats[Cout + c] += sum_rows y[.,c]^2 (fp64, caller zeroes; the
 * layout t2r_bn_stats produces, so t2r_bn_finalize consumes it directly).  Fuses the statistics
 * pass of slim.batch_norm / tf.layers.batch_normalization that follows every convolution
 * (research/qtopt/networks.py:443-448, layers/film_resnet_model.py:50-57).  stats may be NULL. */
int32_t t2r_conv2d_fprop_stats(const T2RConvDesc* d, const void* x, const void* w_ohwi,
                               const float* bias, const void* residual, void* y, double* stats,
                               void* stream);
/* dx = conv_transpose(dy, w).  w_dgrad is [Cin][KH*KW][Cout] bf16 (see t2r_pack_weights).
 * accumulate != 0: dx += result.  Requires Cout % 64 == 0, Cin % 64 == 0. */
int32_t t2r_conv2d_dgrad(const T2RConvDesc* d, const void* dy, const void* w_dgrad, void* dx,
                         int32_t accumulate, void* stream);
/* dw (fp32, OHWI) += dy^T * im2col(x): split-K over pixels with fp32 atomics; the caller
 * zeroes dw once per step.  Requires Cin % 64 == 0, Cout % 64 == 0. */
int32_t t2r_conv2d_wgrad(const T2RConvDesc* d, const void* x, const void* dy, float* dw,
                         void* stream);
/* ---- batch-norm operand fusion of the training step ----------------------------------------
 * In the reference every convolution of a ResNet block reads z = relu(batch_norm(x)) (pre-activation blocks,
 * layers/film_resnet_model.py:283-340 with batch_norm :50-57), and TensorFlow materialises z.  On B200 the
 * normalise-and-rectify pass is pure HBM traffic (4 B per element forward, 4 B for the reduction of the backward),
 * so the kernels below take the RAW tensor x plus the per-channel affine scale[c] = gamma*invstd, shift[c] =
 * beta - mean*scale (t2r_bn_finalize) and never write z:
 *   fprop_bnrelu : y = conv1x1(relu(scale*x + shift), w) (+residual); the A tile is rewritten in shared memory.
 *   wgrad_bnrelu : dw += dy^T * relu(scale*x + shift), same rewrite of the X tiles.
 *   dgrad_bnrelu : g = conv_transpose(dy, w) * [scale*x + shift > 0] (any geometry), and the epilogue accumulates
 *                  red[c] += sum g, red[Cin + c] += sum g*x (fp64 [2*Cin], caller zeroes): exactly what
 *                  t2r_bn_backward's reduction pass computes, so t2r_bn_backward_presummed can follow directly.
 *                  accumulate != 0: g += ... and the reduction then covers the COMPLETE sum (call it last, and
 *                  use plain t2r_conv2d_dgrad for the earlier contributions).  Launches the epilogue cannot fuse
 *                  (halo kernel, accumulation) run the stand-alone reduction pass instead: same results.
 * Values are bit-identical to t2r_bn_apply + t2r_conv2d_* on the materialised z (same fmaf, same bf16 rounding).
 * fprop / wgrad require KH = KW = 1 and no padding (zero padding must stay zero after the affine map). */
int32_t t2r_conv2d_fprop_bnrelu(const T2RConvDesc* d, const void* x_raw, const float* bn_scale,
                                const float* bn_shift, const void* w_ohwi, const void* residual, void* y,
                                double* stats, void* stream);
int32_t t2r_conv2d_wgrad_bnrelu(const T2RConvDesc* d, const void* x_raw, const float* bn_scale,
                                const float* bn_shift, const void* dy, float* dw, void* stream);
int32_t t2r_conv2d_dgrad_bnrelu(const T2RConvDesc* d, const void* dy, const void* w_dgrad, const void* x_raw,
                                const float* bn_scale, const float* bn_shift, void* g, int32_t accumulate,
                                double* red, void* stream);
/* Batch-norm backward through the GEMMs of a 1x1 stride-1 unpadded consumer y = conv1x1(z, w), z = relu(scale*x +
 * shift), m = [scale*x + shift > 0], g = m * conv_transpose(dy, w).  Three launches replace the data gradient, the
 * reduction pass and the apply pass:
 *   wgrad_bnsums      : dw += dy^T * z as scale * P + shift * Q with P = dy^T (m*x), Q = dy^T m (one MMA yields both),
 *                       and sums[c] += sum_n w[n, c] * Q[n, c] (= sum g), sums[Cin + c] += sum_n w[n, c] * P[n, c]
 *                       (= sum g*x); sums fp64 [2*Cin], caller zeroes; w_dgrad is the bf16 [Cin][Cout] copy the data
 *                       gradient multiplies with.
 *   bn_backward_gemm_finalize : dgamma / dbeta (written) and coef = [kb | kc] fp32 [2*C], the per-channel
 *                       coefficients of dx = scale*g + kb*x + kc.
 *   dgrad_bnapply     : dx = scale * m * conv_transpose(dy, w) + kb*x + kc (+ dpass, may be null) in the epilogue of
 *                       the TMA data-gradient kernel, from the fp32 accumulator; g is never written.
 * dgrad_bnapply_supported(d) returns 1 when d is such a convolution and its data gradient runs on the TMA-epilogue
 * kernel (Cin <= 128, or a multiple of 256 with Cout <= 256); dgrad_bnapply fails with T2R_ERR_ARG otherwise. */
int32_t t2r_conv2d_wgrad_bnsums(const T2RConvDesc* d, const void* x_raw, const float* bn_scale, const float* bn_shift,
                                const void* dy, const void* w_dgrad, float* dw, double* sums, void* stream);
int32_t t2r_bn_backward_gemm_finalize(const double* sums, int64_t rows, int32_t C, const float* mean,
                                      const float* invstd, const float* scale, float* dgamma, float* dbeta,
                                      float* coef, void* stream);
int32_t t2r_conv2d_dgrad_bnapply_supported(const T2RConvDesc* d);
int32_t t2r_conv2d_dgrad_bnapply(const T2RConvDesc* d, const void* dy, const void* w_dgrad, const void* x_raw,
                                 const float* bn_scale, const float* bn_shift, const float* coef, const void* dpass,
                                 void* dx, void* stream);
/* ---- high-precision PREDICT path (csrc/hp.cu) ----------------------------------------------
 * fp32 activations; a convolution y = conv(x, w) is evaluated as bf16x3: x3 = [hi | lo | hi] (t2r_hp_split3), w3 =
 * [w_hi | w_hi | w_lo] (t2r_hp_pack_weights3), then t2r_conv2d_fprop with Cin' = 3*Cin and T2R_EPI_OUT_F32 (fp32
 * accumulation): products are exact in fp32 and the operands carry 16 mantissa bits, which brings the critics'
 * q_predicted within 1e-4 of the fp32 restatement of research/qtopt/networks.py:343-615 /
 * layers/film_resnet_model.py:525-629 (tests/test_high_precision_gpu.py) where bf16 storage gives ~1e-2.
 * The fp32 pooling / merge / add kernels are the inference-only counterparts of the bf16 ones below. */
int32_t t2r_hp_split3(const float* x, void* x3_bf16, int64_t rows, int32_t C, void* stream);
int32_t t2r_hp_pack_weights3(const float* w_ohwi, void* w3_bf16, int32_t Cout, int32_t taps, int32_t Cin, void* stream);
int32_t t2r_maxpool_f32_fwd(const float* x, float* y, int32_t N, int32_t H, int32_t W, int32_t C, int32_t k,
                            int32_t stride, int32_t pad_top, int32_t pad_left, int32_t Ho, int32_t Wo, void* stream);
int32_t t2r_global_mean_f32_fwd(const float* x, float* y, int32_t N, int32_t HW, int32_t C, void* stream);
/* tile_batch(x, A) + ctx[:, None, None, :] in fp32 (research/qtopt/networks.py:513-522). */
int32_t t2r_add_context_f32_fwd(const float* x, const float* ctx, float* y, int32_t B, int32_t A, int32_t HW, int32_t C,
                                void* stream);
int32_t t2r_add_f32(const float* a, const float* b, float* y, int64_t n, void* stream);

/* fp32 master OHWI -> bf16 OHWI (w_fprop) and bf16 [Cin][taps][Cout] (w_dgrad; may be NULL). */
int32_t t2r_pack_weights(const float* w, void* w_fprop, void* w_dgrad, int32_t Cout,
                         int32_t taps, int32_t Cin, void* stream);
/* Small-Cin stem (Cin=3): explicit im2col into a K-padded bf16 matrix [N*Ho*Wo, Kpad]
 * (column k = (kh*KW+kw)*Cin + c, zero for k >= KH*KW*Cin), consumed by the 1x1 path above.
 * x is bf16 NHWC.  Replaces conv1_1 6x6/2 (networks.py:443-450) and the 7x7/2 ResNet stem
 * (film_resnet_model.py:561-565). */
int32_t t2r_im2col_small_cin(const T2RConvDesc* d, const void* x, void* a, int32_t Kpad,
                             void* stream);

/* Stem convolution (Cin = 3) WITHOUT im2col.  The image lives in a zero-padded bf16 buffer built by
 * t2r_stem_pack_image (logical pixel (ih,iw) at padded (ih+pad_top, iw+pad_left)), in one of two layouts
 * chosen by rows = (KW <= 8 && stride == 2) ? 2 : 1:
 *   rows = 1: xp[N][Hp][Wp][4]    (channel 3 = 0)        K chunk = [16 px][4 ch] of one filter row
 *   rows = 2: xp[N][Hp/2][Wp][8]  (row pair interleaved)  K chunk = [8 px][2 rows][4 ch]
 * so that the 64 values under an output pixel are 128 contiguous bytes, which overlapping-window TMA
 * maps deliver directly as the A operand (7x7/2: K = 256 instead of the 448 of rows = 1).  Weights:
 * w_stem bf16 [Cout][chunks][64] in the same order, chunks = ceil(KH/rows), zero where kw >= KW,
 * c == 3 or kh >= KH; K = t2r_stem_k(KH, KW, stride).  Requires Wp even, Hp % rows == 0,
 * Wp >= stride*(Wo-1) + 16/rows, Hp >= stride*(Ho-1) + chunks*rows.
 * Same reference call sites as t2r_im2col_small_cin. */
int32_t t2r_stem_pack_image(const void* x_nhwc3, void* xp, int32_t N, int32_t H, int32_t W, int32_t Hp,
                            int32_t Wp, int32_t pad_top, int32_t pad_left, int32_t KW, int32_t stride,
                            void* stream);
int32_t t2r_stem_k(int32_t KH, int32_t KW, int32_t stride);
int32_t t2r_pad_nhwc3_c4(const void* x_nhwc3, void* x4p, int32_t N, int32_t H, int32_t W, int32_t Hp,
                         int32_t Wp, int32_t pad_top, int32_t pad_left, void* stream);
int32_t t2r_stem_conv_fprop(const T2RConvDesc* d, const void* x4p, int32_t Hp, int32_t Wp,
                            const void* w_stem, const float* bias, void* y, void* stream);
int32_t t2r_stem_conv_wgrad(const T2RConvDesc* d, const void* x4p, int32_t Hp, int32_t Wp, const void* dy,
                            float* dw_stem, void* stream);
/* Clears the padded slots of dw_stem fp32 [Cout][t2r_stem_k] after t2r_stem_conv_wgrad. */
int32_t t2r_stem_mask_grad(float* dw_stem, int32_t Cout, int32_t KH, int32_t KW, int32_t stride,
                           void* stream);

/* Spatial softmax (layers/spatial_softmax.py:29-88): x bf16 [N,H,W,C] -> points fp32 [N,2C], the expected
 * (x, y) position of every channel's softmax over H*W with x_j = 2j/(W-1)-1, y_i = 2i/(H-1)-1, laid out
 * INTERLEAVED (x_1,y_1,x_2,y_2,...) as the reference's reshape of concat([x,y],1) produces; softmax
 * (optional, bf16 [N,H,W,C]) is the heat map.  bwd: gradient w.r.t. x from dpoints (the softmax is
 * recomputed). */
int32_t t2r_spatial_softmax_fwd(const void* x, float* points, void* softmax, int32_t N, int32_t H, int32_t W,
                                int32_t C, void* stream);
int32_t t2r_spatial_softmax_bwd(const void* x, const float* points, const float* dpoints, void* dx, int32_t N,
                                int32_t H, int32_t W, int32_t C, void* stream);

/* PCGrad gradient surgery (research/qtopt/pcgrad.py:123-154, per-variable implementation) on flat gradient buffers.
 * grads: fp32 [T][stride], row t = the gradient of task loss t over the whole flat parameter buffer; variable v is
 * the segment [seg_off[v], seg_off[v] + seg_len[v]) (device int64 [V]); use_pcgrad (device uint8 [V], may be NULL =
 * all) marks the variables that pass the allow / deny lists, the others receive the plain sum of the task gradients.
 * out[seg] = sum over tasks of the sequentially projected gradients, eps = 1e-5 in the reference.  Workspaces:
 * gram fp32 [V][T][T], coef fp32 [V][T].  1 <= T <= 8.  Elements of `out` outside every segment are left untouched. */
int32_t t2r_pcgrad_project(const float* grads, int32_t T, int64_t stride, const int64_t* seg_off,
                           const int64_t* seg_len, const uint8_t* use_pcgrad, int32_t V, float eps, float* gram,
                           float* coef, float* out, void* stream);

/* ---- fp32 kernels of the small pose_env networks (layers/vision_layers.py:30-158, 277-350;
 * research/pose_env/pose_env_models.py:118-181): 32-channel layers on 64x64 frames, below one tensor-core
 * tile, hence CUDA-core kernels.  x NHWC fp32, w HWIO fp32 (the TF layout), padding given explicitly. */
int32_t t2r_conv2d_direct_f32_fwd(const float* x, const float* w, const float* bias, float* y, int32_t N, int32_t H,
                                  int32_t W, int32_t Cin, int32_t Cout, int32_t KH, int32_t KW, int32_t stride,
                                  int32_t pad_top, int32_t pad_left, int32_t Ho, int32_t Wo, void* stream);
int32_t t2r_conv2d_direct_f32_dgrad(const float* dy, const float* w, float* dx, int32_t N, int32_t H, int32_t W,
                                    int32_t Cin, int32_t Cout, int32_t KH, int32_t KW, int32_t stride, int32_t pad_top,
                                    int32_t pad_left, int32_t Ho, int32_t Wo, void* stream);
/* dw is overwritten (Cout <= 256). */
int32_t t2r_conv2d_direct_f32_wgrad(const float* x, const float* dy, float* dw, int32_t N, int32_t H, int32_t W,
                                    int32_t Cin, int32_t Cout, int32_t KH, int32_t KW, int32_t stride, int32_t pad_top,
                                    int32_t pad_left, int32_t Ho, int32_t Wo, void* stream);
/* slim.layer_norm: moments over the D values of each of the N samples, per-channel gamma / beta (channel =
 * index mod C), optional fused ReLU; mean / rstd [N] are saved for the backward pass, which overwrites
 * dgamma / dbeta [C] (both may be NULL). */
int32_t t2r_layer_norm_f32_fwd(const float* x, const float* gamma, const float* beta, float* y, float* mean, float* rstd,
                               int32_t N, int32_t D, int32_t C, float eps, int32_t relu, void* stream);
int32_t t2r_layer_norm_f32_bwd(const float* x, const float* dy, const float* gamma, const float* beta, const float* mean,
                               const float* rstd, float* dx, float* dgamma, float* dbeta, int32_t N, int32_t D,
                               int32_t C, int32_t relu, void* stream);
/* fp32 variant of t2r_spatial_softmax_* (any channel count). */
int32_t t2r_spatial_softmax_f32_fwd(const float* x, float* points, float* softmax, int32_t N, int32_t H, int32_t W,
                                    int32_t C, void* stream);
int32_t t2r_spatial_softmax_f32_bwd(const float* x, const float* points, const float* dpoints, float* dx, int32_t N,
                                    int32_t H, int32_t W, int32_t C, void* stream);
/* pose_env critic action merge (pose_env_models.py:141-149): y[j] = x[j mod Nx] + ctx[j] broadcast over HW,
 * x [Nx,HW,C], ctx [Nc,C], y [Nc,HW,C], Nc a multiple of Nx.  bwd: dx and / or dctx (either may be NULL). */
int32_t t2r_tile_add_context_f32_fwd(const float* x, const float* ctx, float* y, int32_t Nx, int32_t Nc, int32_t HW,
                                     int32_t C, void* stream);
int32_t t2r_tile_add_context_f32_bwd(const float* dy, float* dx, float* dctx, int32_t Nx, int32_t Nc, int32_t HW,
                                     int32_t C, void* stream);
/* tf.nn.relu on fp32 (the default activation of the pose_env critic's fully connected layers). */
int32_t t2r_relu_f32_fwd(const float* x, float* y, int64_t n, void* stream);
int32_t t2r_relu_f32_bwd(const float* dy, const float* y, float* dx, int64_t n, void* stream);
/* MockT2RModel layers (utils/mocks.py:160-176): tf.nn.elu and tf.layers.batch_normalization(training=False) on fp32
 * [rows, C]: y = (x - mean) * rsqrt(var + eps) * gamma + beta; bwd overwrites dgamma / dbeta [C] (may both be NULL). */
int32_t t2r_elu_f32_fwd(const float* x, float* y, int64_t n, void* stream);
int32_t t2r_elu_f32_bwd(const float* dy, const float* y, float* dx, int64_t n, void* stream);
/* The batch-norm normaliser and the FiLM conditioning of the spatial-softmax tower (layers/vision_layers.py:72-86,
 * 100-141): slim.batch_norm(is_training=True, decay, epsilon, scale optional -> gamma may be NULL) on fp32 [rows, C]
 * with an optional fused ReLU (moving statistics updated in place, batch mean / rstd saved for the backward), and
 * y = relu((1 + film[n, c]) * x + film[n, C + c]) on fp32 [N, HW, C] with film fp32 [N, 2C]; bwd writes dx and
 * dfilm (same layout). */
int32_t t2r_bn_train_f32_fwd(const float* x, const float* gamma, const float* beta, float* y, float* moving_mean,
                             float* moving_var, float* save_mean, float* save_rstd, int64_t rows, int32_t C, float eps,
                             float decay, int32_t relu, void* stream);
int32_t t2r_bn_train_f32_bwd(const float* x, const float* y, const float* dy, const float* gamma, const float* save_mean,
                             const float* save_rstd, float* dx, float* dgamma, float* dbeta, int64_t rows, int32_t C,
                             int32_t relu, void* stream);
int32_t t2r_film_relu_f32_fwd(const float* x, const float* film, float* y, int32_t N, int32_t HW, int32_t C, void* stream);
int32_t t2r_film_relu_f32_bwd(const float* x, const float* film, const float* dy, float* dx, float* dfilm, int32_t N,
                              int32_t HW, int32_t C, void* stream);
int32_t t2r_bn_infer_f32_fwd(const float* x, const float* gamma, const float* beta, const float* mean, const float* var,
                             float* y, int64_t rows, int32_t C, float eps, void* stream);
int32_t t2r_bn_infer_f32_bwd(const float* x, const float* dy, const float* gamma, const float* mean, const float* var,
                             float* dx, float* dgamma, float* dbeta, int64_t rows, int32_t C, float eps, void* stream);

/* ---- fp32 CUDA-core GEMM for the tiny action-context / logit layers -------------------- */
/* C[M,N] = alpha * op(A) * op(B) + beta * C, row-major, op = transpose if flag set.
 * Replaces slim.fully_connected on grasp params and logits (networks.py:488-503,566-573). */
int32_t t2r_sgemm(int32_t transA, int32_t transB, int32_t M, int32_t N, int32_t K, float alpha,
                  const float* A, int32_t lda, const float* B, int32_t ldb, float beta, float* C,
                  int32_t ldc, void* stream);
int32_t t2r_bias_add_f32(float* y, const float* bias, int64_t rows, int32_t C, void* stream);
int32_t t2r_colsum_f32(const float* x, float* out, int64_t rows, int32_t C, void* stream);
/* out[0] += scale * sum(x^2): the slim l2_regularizer loss term (SURVEY 8c-5). */
int32_t t2r_sumsq_f32(const float* x, float* out, int64_t n, float scale, void* stream);
int32_t t2r_cast_f32_to_bf16(const float* x, void* y, int64_t n, void* stream);
/* Inference-mode batch norm folded into the producing convolution (is_training=False graphs of
 * slim.conv2d(normalizer_fn=slim.batch_norm) / tf.layers conv -> batch_normalization):
 * w_bf16[co, k] = bf16(w[co, k] * scale[co]); the shift becomes the convolution's bias. */
int32_t t2r_fold_bn_weights(const float* w_ohwi, const float* scale, void* w_bf16, int32_t Cout, int64_t K,
                            void* stream);
int32_t t2r_cast_bf16_to_f32(const void* x, float* y, int64_t n, void* stream);

/* ---- batch norm (slim.batch_norm / tf.layers.batch_normalization, training + inference) - */
/* x: bf16 [rows, C].  stats: fp64 [2*C] workspace (sum, sumsq), zeroed by the call.
 * Reference: film_resnet_model.py:50-57 (momentum .997 eps 1e-5), networks.py:396-410
 * (decay .9997 eps .001); SURVEY §8c-4 (biased var to normalise, Bessel var into moving). */
int32_t t2r_bn_stats(const void* x, int64_t rows, int32_t C, double* stats, void* stream);
/* out[c] = sum_r x[r,c] for bf16 x (bias gradients); stats: fp64 [2*C] workspace. */
int32_t t2r_colsum_bf16(const void* x, int64_t rows, int32_t C, double* stats, float* out, void* stream);
/* From stats: mean/var -> scale = gamma*rsqrt(var+eps), shift = beta - mean*scale; saves
 * mean and invstd (fp32 [C] each) for backward; updates moving stats in place with
 * moving = moving*momentum + batch*(1-momentum) (variance Bessel-corrected).
 * gamma may be NULL (scale=False).  moving_* may be NULL. */
int32_t t2r_bn_finalize(const double* stats, int64_t rows, int32_t C, const float* gamma,
                        const float* beta, float eps, float momentum, float* moving_mean,
                        float* moving_var, float* mean, float* invstd, float* scale,
                        float* shift, void* stream);
/* Inference: scale/shift from moving statistics. */
int32_t t2r_bn_infer_params(int32_t C, const float* gamma, const float* beta,
                            const float* moving_mean, const float* moving_var, float eps,
                            float* scale, float* shift, void* stream);
/* y = act(x*scale[c] + shift[c]); optional FiLM per image (film [N, 2C] fp32: gamma|beta,
 * applied as (1+g)*v + b before the ReLU, film_resnet_model.py:108-115); rows_per_image
 * = H*W of that tensor.  relu != 0 applies ReLU. */
int32_t t2r_bn_apply(const void* x, void* y, int64_t rows, int32_t C, const float* scale,
                     const float* shift, const float* film, int64_t rows_per_image,
                     int32_t relu, void* stream);
/* Backward of y = relu?(bn(x)) w.r.t. x, gamma, beta.  dy, x: bf16 [rows,C].
 * red: fp64 [2*C] workspace.  dgamma/dbeta: fp32 [C], both written (required).
 * dres (optional, bf16 [rows,C]) is added to dx (residual-branch gradient). */
int32_t t2r_bn_backward(const void* dy, const void* x, const void* dres, void* dx, int64_t rows,
                        int32_t C, const float* gamma, const float* mean, const float* invstd,
                        const float* scale, const float* shift, int32_t relu, double* red,
                        float* dgamma, float* dbeta, void* stream);
/* Second half of t2r_bn_backward for callers that already hold red[c] = sum dz, red[C + c] = sum dz*x with
 * dz = dy*[scale*x + shift > 0] (t2r_conv2d_dgrad_bnrelu): dgamma / dbeta from red, then
 * dx = scale*dz - (scale*dgamma*invstd/rows)*(x - mean) - scale*dbeta/rows (+ dres).  The mask is re-applied
 * (idempotent), so dy may hold either the masked or the unmasked gradient. */
int32_t t2r_bn_backward_presummed(const void* dy, const void* x, const void* dres, void* dx, int64_t rows,
                                  int32_t C, const float* mean, const float* invstd, const float* scale,
                                  const float* shift, int32_t relu, const double* red, float* dgamma,
                                  float* dbeta, void* stream);

/* Backward of y = relu?((1 + film_gamma[n,c]) * bn(x) + film_beta[n,c]) (FiLM-conditioned batch norm,
 * layers/film_resnet_model.py:108-115): film fp32 [N][2C] (gamma part then beta part), dfilm same shape
 * (written), sums_ws fp32 [N][2][C] workspace; other arguments as t2r_bn_backward. */
int32_t t2r_bn_film_backward(const void* dy, const void* x, const float* film, const void* dres, void* dx,
                             float* dfilm, int64_t rows, int32_t C, int64_t rows_per_image,
                             const float* mean, const float* invstd, const float* scale, const float* shift,
                             int32_t relu, float* sums_ws, float* dgamma, float* dbeta, void* stream);

/* ---- pooling / reductions / elementwise ------------------------------------------------ */
/* slim.max_pool2d SAME/VALID (networks.py:452,459,528; film_resnet_model.py:575-579).
 * argmax: uint8 [N,Ho,Wo,C] window-relative index of the first maximum (TF tie rule). */
int32_t t2r_maxpool_fwd(const void* x, void* y, uint8_t* argmax, int32_t N, int32_t H, int32_t W,
                        int32_t C, int32_t k, int32_t stride, int32_t pad_top, int32_t pad_left,
                        int32_t Ho, int32_t Wo, void* stream);
int32_t t2r_maxpool_bwd(const void* dy, const uint8_t* argmax, void* dx, int32_t N, int32_t H,
                        int32_t W, int32_t C, int32_t k, int32_t stride, int32_t pad_top,
                        int32_t pad_left, int32_t Ho, int32_t Wo, void* stream);
/* tf.reduce_mean over H,W (film_resnet_model.py:611-613): bf16 [N,HW,C] -> bf16 [N,C]. */
int32_t t2r_global_mean_fwd(const void* x, void* y, int32_t N, int32_t HW, int32_t C,
                            void* stream);
int32_t t2r_global_mean_bwd(const void* dy, void* dx, int32_t N, int32_t HW, int32_t C,
                            void* stream);
/* Tile + broadcast add of the action context (networks.py:513-522, tile_batch + tf.add):
 * y[(b*A+a), p, c] = x[b, p, c] + ctx[(b*A+a), c]; never materialises the tile of x. */
int32_t t2r_add_context_fwd(const void* x, const void* ctx, void* y, int32_t B, int32_t A,
                            int32_t HW, int32_t C, void* stream);
/* dx[b,p,c] = sum_a dy[(b*A+a),p,c]; dctx[(b*A+a),c] = sum_p dy[(b*A+a),p,c]. */
/* Inference fusion of the merge with the batch norm (+ReLU) that consumes it:
 * y[(b*A+a),p,:] = relu?((x[b,p,:] + ctx[(b*A+a),:]) * scale + shift), scale / shift from t2r_bn_infer_params. */
int32_t t2r_add_context_affine_fwd(const void* x, const void* ctx, const float* scale, const float* shift, void* y,
                                   int32_t B, int32_t A, int32_t HW, int32_t C, int32_t relu, void* stream);
int32_t t2r_add_context_bwd(const void* dy, void* dx, void* dctx, int32_t B, int32_t A,
                            int32_t HW, int32_t C, void* stream);
/* y = a + b (bf16), used for gradient fan-in. */
int32_t t2r_add_bf16(const void* a, const void* b, void* y, int64_t n, void* stream);
/* y = relu(a + b), bf16, n % 8 == 0: the shortcut add + ReLU that closes a ResNet v1 block
 * (layers/film_resnet_model.py:156-166, 268-276). */
int32_t t2r_add_relu_bf16(const void* a, const void* b, void* y, int64_t n, void* stream);
int32_t t2r_relu_bwd_bf16(const void* dy, const void* y, void* dx, int64_t n, void* stream);

/* ---- image preprocessing (HBM-bound) --------------------------------------------------- */
/* Fused crop + uint8->float (x * (1/255), SURVEY §8c-3) + photometric distortion + clip.
 * Reference: research/qtopt/t2r_models.py:277-308, preprocessors/image_transformations.py:
 * 25-101 (crops), :176-264 (ApplyPhotometricImageDistortions).  One parameter set per image
 * (the reference draws one per batch; replicate the scalar to reproduce it). */
typedef struct T2RDistortParams {   /* per image, fp32 */
  float brightness_delta;  /* added after conversion; 0 = off                             */
  float saturation_scale;  /* HSV saturation multiplier; 1 = off                          */
  float hue_delta;         /* HSV hue shift in [-1,1] turns; 0 = off                      */
  float contrast_scale;    /* (x-mean_c)*c+mean_c with per-image per-channel mean; 1 = off */
  float noise_stddev;      /* gaussian noise level; 0 = off                               */
  int32_t crop_y, crop_x;  /* crop offsets into the source image                          */
  int32_t reserved;
} T2RDistortParams;
/* src u8 [N,H,W,3]; dst bf16 or fp32 [N,h,w,3] (out_f32 selects).  chan_mean: fp32 [N,3]
 * workspace used when any contrast_scale != 1 (computed by the call).  seed/offset: Philox
 * stream for the noise. */
int32_t t2r_crop_convert_distort(const uint8_t* src, void* dst, const T2RDistortParams* params,
                                 float* chan_mean, int32_t N, int32_t H, int32_t W, int32_t h,
                                 int32_t w, int32_t out_f32, int32_t use_contrast,
                                 uint64_t seed, uint64_t offset, void* stream);
/* tf.image.resize_images bilinear, TF1 legacy sampling (align_corners=False, no half-pixel
 * centres: src = dst * in/out), preprocessors/distortion.py:56-107.  fp32 NHWC. */
/* The same photometric distortions on an already converted float image [N,H,W,3] (BC-Z distorts AFTER the
 * resize: preprocessors/distortion.py:56-107); params[n].crop_* must be 0.  In place (dst == src) is allowed
 * when use_contrast is 0. */
int32_t t2r_distort_f32(const float* src, float* dst, const T2RDistortParams* params, float* chan_mean,
                        int32_t N, int32_t H, int32_t W, int32_t use_contrast, uint64_t seed, uint64_t offset,
                        void* stream);
int32_t t2r_resize_bilinear_legacy(const float* src, float* dst, int32_t N, int32_t H, int32_t W,
                                   int32_t C, int32_t h, int32_t w, void* stream);
/* ApplyPhotometricImageDistortionsCheap (preprocessors/image_transformations.py:365-384): dst = src ** g_c per
 * channel (n elements, channel = index mod C, C <= 4). */
int32_t t2r_channel_gamma_f32(const float* src, float* dst, int64_t n, int32_t C, float g0, float g1, float g2, float g3,
                              void* stream);
/* ApplyDepthImageDistortions (image_transformations.py:403-459) for one tensor of the list:
 * dst = clip(alpha * src + N(0, noise_stddev), min_depth, max_depth); Philox stream (seed, offset). */
int32_t t2r_depth_distort_f32(const float* src, float* dst, int64_t n, float alpha, float noise_stddev, float min_depth,
                              float max_depth, uint64_t seed, uint64_t offset, void* stream);

/* ---- losses ---------------------------------------------------------------------------- */
/* q = sigmoid(logit); loss = mean(-(y log(q+eps) + (1-y) log(1-q+eps))), eps = 1e-7
 * (tf.losses.log_loss; research/qtopt/t2r_models.py:229-239, models/critic_model.py:171-192).
 * Writes q [n], loss [1] (accumulated: caller zeroes), dlogit [n] = dloss/dlogit. */
int32_t t2r_sigmoid_logloss(const float* logit, const float* label, float* q, float* loss,
                            float* dlogit, int64_t n, void* stream);
int32_t t2r_sigmoid_f32(const float* logit, float* q, int64_t n, void* stream);

/* ---- CEM + Bellman target (utils/cross_entropy.py:30-154, policies/policies.py:105-184) - */
/* samples[b,a,d] = mean[b,d] + std[b,d] * N(0,1) (Philox4x32-10 + Box-Muller). */
int32_t t2r_cem_sample(const float* mean, const float* stddev, float* samples, int32_t B,
                       int32_t A, int32_t D, uint64_t seed, uint64_t offset, void* stream);
/* Per row b: stable ascending sort of values[b,:], elites = last num_elites; writes
 * mean[b,:], std[b,:] (ddof=1) of the elite samples, best_value[b] = max, best_index[b] =
 * first argmax (np.argmax).  A <= 1024. */
int32_t t2r_cem_refit(const float* samples, const float* values, float* mean, float* stddev,
                      float* best_value, int32_t* best_index, int32_t B, int32_t A, int32_t D,
                      int32_t num_elites, void* stream);
/* y[b] = r[b] + gamma * (1 - done[b]) * max_q[b]   (QT-Opt target; SURVEY A-23: absent from
 * the reference, parity unpinned). */
int32_t t2r_bellman_target(const float* reward, const float* done, const float* max_q,
                           float gamma, float* target, int64_t n, void* stream);

/* ---- optimizers (models/optimizers.py:61-146, research/qtopt/optimizer_builder.py:25-96) */
/* All state fp32, flat contiguous buffers of n elements.  grad_scale multiplies the raw
 * gradient (1/world_size after the NCCL sum).  Elements [0, n_decay) additionally receive
 * the slim l2_regularizer gradient l2 * w (SURVEY §8c-5).  ema (optional) is updated as
 * ema = d*ema + (1-d)*w with the *new* w.  w_bf16 (optional) receives the bf16 copy. */
int32_t t2r_momentum_step(float* w, const float* g, float* accum, float* ema, void* w_bf16,
                          int64_t n, int64_t n_decay, float lr, float momentum, float l2,
                          float grad_scale, float ema_decay, void* stream);
/* TF Adam: lr_t = lr*sqrt(1-b2^t)/(1-b1^t); m,v updates; w -= lr_t*m/(sqrt(v)+eps). */
int32_t t2r_adam_step(float* w, const float* g, float* m, float* v, float* ema, void* w_bf16,
                      int64_t n, int64_t n_decay, float lr, float beta1, float beta2, float eps,
                      int64_t step, float l2, float grad_scale, float ema_decay, void* stream);

/* TF RMSPropOptimizer (not centered; research/qtopt/optimizer_builder.py:76-81): ms = decay*ms + (1-decay)*g^2 (the
 * slot starts at ONE, as TF initialises it), mom = momentum*mom + lr*g/sqrt(ms + eps), w -= mom; l2 / grad_scale /
 * EMA / bf16 refresh as in the other steps.  All three steps move 16-byte vectors: buffers 16-byte aligned, n and
 * n_decay multiples of 4 (nn.VariableStore pads every variable to 64 elements). */
int32_t t2r_rmsprop_step(float* w, const float* g, float* ms, float* mom, float* ema, void* w_bf16, int64_t n,
                         int64_t n_decay, float lr, float decay, float momentum, float eps, float l2,
                         float grad_scale, float ema_decay, void* stream);

/* Mixup (research/bcz/model.py:164-172): y[b] = lambda*x[b] + (1-lambda)*x[B-1-b] on fp32 [B, inner]; x != y. */
int32_t t2r_mixup_reverse_f32(const float* x, float* y, int32_t B, int64_t inner, float lambda, void* stream);

/* ---- weighted loss tail (BC-Z) ------------------------------------------------------------
 * research/bcz/model.py:476-585 (training_outputs): tf.losses.huber_loss / mean_squared_error / log_loss per action
 * component with weights = component weight x (1 - stop_token), the quaternion-norm penalty and the first-waypoint
 * diagnostics, all with Reduction.SUM_BY_NONZERO_WEIGHTS: loss = sum(l_i w_i) / max(#{w_i != 0}, 1).
 * One launch evaluates up to T2R_MAX_LOSS_SEGMENTS segments (flat fp32 arrays viewed as [rows, cols]):
 *   element weight = weight x (row_mask ? (complement ? 1 - row_mask[row] : row_mask[row]) : 1), zero when row_mod > 0
 *   and row % row_mod != 0 (row_mod = number of waypoints selects the first waypoint of every sample);
 *   labels == NULL -> every label is label_const; SIGMOID_LOG takes logits and also writes sigmoid(x) to sigmoid_out.
 * losses[s] receives the segment loss, losses[n_segments] the sum over segments with in_total != 0; dpredictions (if
 * not NULL) the gradient of losses[s] w.r.t. the predictions / logits. */
#define T2R_LOSS_HUBER 0
#define T2R_LOSS_MSE 1
#define T2R_LOSS_SIGMOID_LOG 2
#define T2R_MAX_LOSS_SEGMENTS 16
typedef struct T2RLossSegment {
  uint32_t struct_size;
  int32_t kind;                 /* T2R_LOSS_* */
  const float* predictions;     /* [n] */
  const float* labels;          /* [n] or NULL */
  const float* row_mask;        /* [n / cols] or NULL */
  float* dpredictions;          /* [n] or NULL */
  float* sigmoid_out;           /* [n] or NULL (SIGMOID_LOG only) */
  int64_t n;
  int32_t cols;
  int32_t row_mod;
  int32_t row_mask_is_complement;
  int32_t in_total;
  float weight, delta, label_const, reserved;
} T2RLossSegment;
int32_t t2r_weighted_losses(const T2RLossSegment* segments, int32_t n_segments, float* losses, void* stream);

/* ---- host-side record path (no GPU): TFRecord framing + tf.Example wire format ---------- */
/* Reference: utils/tfdata.py:174-210,629-689 (reader), :273-424 (tf.parse_example). */
uint32_t t2r_crc32c(const uint8_t* data, uint64_t n);
uint32_t t2r_masked_crc32c(const uint8_t* data, uint64_t n);
/* Index an in-memory TFRecord file: writes up to max_records (offset,length) pairs of the
 * record payloads; returns the record count or a negative error (CRC mismatch => PARSE). */
int64_t t2r_tfrecord_index(const uint8_t* file, uint64_t file_len, uint64_t* offsets,
                           uint64_t* lengths, int64_t max_records, int32_t verify_crc);
/* A parse plan: for each feature key, a dtype, element count and destination. */
#define T2R_DT_FLOAT 1
#define T2R_DT_INT64 2
#define T2R_DT_BYTES 3
typedef struct T2RFeaturePlan {
  const char* key;
  int32_t dtype;     /* T2R_DT_*                                                         */
  int32_t count;     /* fixed element count (FixedLenFeature); <0 => varlen, |count|=max */
  int32_t required;  /* missing key => error when non-zero                               */
  void* dst;         /* FLOAT: float[B*count]; INT64: int64[B*count];
                        BYTES: (const uint8_t*)[B*count] pointers into the record        */
  uint64_t* dst_len; /* BYTES: byte length per element; varlen: element count per row    */
  float pad_float;   /* varlen default                                                   */
  int64_t pad_int64;
} T2RFeaturePlan;
int32_t t2r_example_parse_batch(const uint8_t* const* records, const uint64_t* lengths,
                                int32_t B, T2RFeaturePlan* plan, int32_t n_features);
/* tf.SequenceExample feature_lists (tf.io.parse_sequence_example with FixedLenSequenceFeature(allow_missing),
 * utils/tfdata.py:352-384).  The context part of a SequenceExample has the wire layout of an Example and is
 * parsed by t2r_example_parse_batch.  plan[i].count = values per step; plan[i].dst = [B][max_steps][count]
 * (BYTES: pointers, with dst_len of the same shape), zero-initialised by the caller = the padding.
 * steps[i*B + b] receives the number of steps of feature i in record b; a missing key has 0 steps.
 * max_steps == 0: only `steps` is produced (first pass, to size the dense batch). */
int32_t t2r_sequence_example_parse_batch(const uint8_t* const* records, const uint64_t* lengths,
                                         int32_t B, const T2RFeaturePlan* plan, int32_t n_features,
                                         int32_t max_steps, int64_t* steps);

/* ---- metric learning (Grasp2Vec) ------------------------------------------------------------ */
/* n-pairs loss with labels = range(B) (research/grasp2vec/losses.py:152-181 ->
 * tf.contrib.losses.metric_learning.npairs_loss): loss = mean_i(logsumexp_j(a_i . p_j) - a_i . p_i)
 * + 0.25 * reg_lambda * (mean_i |a_i|^2 + mean_i |p_i|^2); also writes d loss / d anchor, d positive.
 * anchor, positive, d_*: fp32 [B, D]; sim_ws fp32 [B, B]; row_ws fp32 [B]; loss fp32 [1]. */
int32_t t2r_npairs_loss(const float* anchor, const float* positive, int32_t B, int32_t D, float reg_lambda,
                        float* sim_ws, float* row_ws, float* loss, float* d_anchor, float* d_positive,
                        void* stream);
/* Triplet loss with semi-hard negative mining (research/grasp2vec/losses.py:51-71 ->
 * tf.contrib.losses.metric_learning.triplet_semihard_loss; the mining is restated in layers/tec.py:322-383):
 * squared Euclidean pairwise distances, per (anchor, positive) the smallest negative distance beyond the
 * positive one, else the largest negative distance; mean of max(margin + d_ap - d_an, 0) over the positive
 * pairs.  emb fp32 [M, D], labels int32 [M]; ws: 3*M*M + M + 2 floats; writes loss [1] and d loss / d emb. */
int32_t t2r_triplet_semihard_loss(const float* emb, const int32_t* labels, int32_t M, int32_t D, float margin,
                                  float* ws, float* loss, float* d_emb, void* stream);
/* y = max(x, 0) on bf16 (tf.nn.relu outside a fused epilogue; backward: t2r_relu_bwd_bf16). */
int32_t t2r_relu_fwd_bf16(const void* x, void* y, int64_t n, void* stream);

/* ---- JPEG decode, split host / device (utils/tfdata.py:426-484 -> tf.image.decode_image) ---- *
 * Baseline sequential Huffman JPEG (SOF0/SOF1, 8 bit, one interleaved scan, restart intervals; grey or
 * YCbCr 4:4:4 / 4:2:2 / 4:2:0).  Host: headers + Huffman entropy decoding into quantised coefficient
 * blocks (serial per image, threaded over the batch).  Device: dequantisation, libjpeg's ISLOW inverse
 * DCT, fancy (triangle) chroma upsampling and the fixed-point YCbCr -> RGB tables: bit-exact with
 * libjpeg(-turbo) defaults, i.e. with what TensorFlow decodes.  Anything else is rejected with
 * T2R_ERR_PARSE (the caller may fall back to its host decoder). */
typedef struct T2RJpegInfo {
  uint32_t struct_size;
  int32_t width, height, ncomp;      /* ncomp 1 (grey) or 3 (YCbCr)                                  */
  int32_t comp_id[3], h[3], v[3], tq[3];
  int32_t hmax, vmax, mcux, mcuy;    /* MCU grid: mcux x mcuy MCUs of (8*hmax) x (8*vmax) pixels      */
  int32_t restart_interval;
  int32_t reserved;
  int64_t coef_offset[3];            /* component c: int16 [mcuy*v][mcux*h][64], natural order        */
  int64_t coef_count;                /* int16 elements of one image                                   */
  uint16_t qt[4][64];                /* quantisation tables, natural order                            */
} T2RJpegInfo;
int32_t t2r_jpeg_parse(const uint8_t* data, uint64_t len, T2RJpegInfo* info);
/* coef: host (pinned) int16 [B][coef_stride]; infos[b] is filled for every image. */
int32_t t2r_jpeg_entropy_decode_batch(const uint8_t* const* data, const uint64_t* lens, int32_t B,
                                      T2RJpegInfo* infos, int16_t* coef, int64_t coef_stride);
/* Complete decode on host threads into out uint8 [B,H,W,channels] (channels 3: RGB, grey replicated; 1: luma): the
 * 'host' image decoder of the record parser for baseline JPEGs, same integer arithmetic as the device half, i.e.
 * bit-identical with libjpeg(-turbo).  Every stream must be H x W; unsupported streams give T2R_ERR_PARSE. */
int32_t t2r_jpeg_decode_host_batch(const uint8_t* const* data, const uint64_t* lens, int32_t B, int32_t H, int32_t W,
                                   int32_t channels, uint8_t* out);
/* Device half.  All B images share the geometry of `geom` (width, height, sampling factors: the spec's
 * static shape); qt: device uint16 [B][4][64] (per-image tables); coef: device int16 [B][coef_stride];
 * planes: device uint8 workspace [B][coef_count] (IDCT output per component); out: uint8 [B,H,W,channels],
 * channels 3 (RGB; grey replicated) or 1 (luma). */
int32_t t2r_jpeg_idct_color(const int16_t* coef, const uint16_t* qt, const T2RJpegInfo* geom, uint8_t* planes,
                            uint8_t* out, int32_t B, int64_t coef_stride, int32_t channels, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* T2R_B200_H_ */
