// conv_common.cuh — declarations shared by the tcgen05 convolution kernels.
#pragma once
#include "common.cuh"

namespace t2r {

// One filter tap of an implicit-GEMM convolution.
struct ConvTap {
  int8_t map;       // which activation tensor map (stride phase)
  int8_t dh, dw;    // coordinate offset inside that map
  int8_t pad;
  int32_t kchunk0;  // first 64-wide K chunk of this tap in the weight matrix
};
constexpr int kMaxTaps = 32;

// Pick the TW x TH = `pixels` rectangle that wastes the fewest padded pixels.
void pick_tile(int Ho, int Wo, int pixels, int* TW, int* TH);
// Tensor maps (box 64 x TW x TH x 1, 128B swizzle) for the stride*stride phases of a
// [N,H,W,C] bf16 tensor; unused slots are filled with map 0.
int make_phase_maps(CUtensorMap* maps, const void* x, int N, int H, int W, int C, int stride,
                    int TW, int TH);

constexpr int kMaxStatChannels = 2048;

// Internal flag bits above the public T2R_EPI_* ones: batch-norm fusions of the training step.
//   kEpiBnBwd  (data gradients): the epilogue turns the gradient w.r.t. z = relu(bn_scale * x + bn_shift) into
//              g = dz * [z > 0] (x = bn_x, the tensor the batch norm normalised, same shape / strides as the
//              output) and accumulates stats[c] += sum g, stats[Cout + c] += sum g * x: the reduction pass of
//              the batch-norm backward (bn_bwd_reduce_kernel, norm.cu) without its two HBM reads.
//   kProBnRelu (1x1 fprop): the activation tensor map points at the RAW tensor x and four extra warps rewrite
//              every landed A tile in shared memory as relu(bn_scale * x + bn_shift) before the MMA reads it: the
//              batch-norm apply pass (bn_apply_rows_kernel) without writing / re-reading z.
//   kEpiBnApply (1x1 stride-1 data gradients, TMA epilogue only): the batch-norm reduction is already known
//              (t2r_conv2d_wgrad_bnsums + t2r_bn_backward_gemm_finalize), so the epilogue writes the batch-norm input
//              gradient directly: dx = bn_scale * [bn_scale * x + bn_shift > 0] * acc + kb * x + kc (+ residual,
//              the pass-through gradient), bn_coef = [kb | kc].  Neither g nor any column sum is produced.
constexpr int kEpiBnBwd = 1 << 8;
constexpr int kProBnRelu = 1 << 9;
constexpr int kEpiBnApply = 1 << 10;

struct IgemmParams {
  CUtensorMap tmap_a[4];
  CUtensorMap tmap_b;
  ConvTap taps[kMaxTaps];
  int n_taps;
  int chunks_per_tap;  // Cin / 64
  int TW, TH;          // tile rectangle, TW*TH == 128
  int tiles_w, tiles_h;
  int N, Ho, Wo;       // output iteration space (a strided view for dgrad phases)
  int Cout;
  int n_tiles_n;
  int total_tiles;
  long long os_n, os_h, os_w;  // output element strides of the view
  void* out;
  const void* residual;
  const float* bias;
  int flags;
  double* stats;  // optional fp64 [2*Cout]: per-channel sum / sum of squares of the bf16 output (fused bn_stats)
  const void* bn_x;        // kEpiBnBwd: the normalised tensor, addressed like `out`
  const float* bn_scale;   // kEpiBnBwd / kEpiBnApply: [Cout] of the output view; kProBnRelu: [Cin]
  const float* bn_shift;
  const float* bn_coef;    // kEpiBnApply: fp32 [2 * Cout], kb then kc
};

// The tap-table kernel with a TMA epilogue (conv_igemm_tma.cu): residual tile in by TMA, output tile
// out by TMA.  block_n is 64 or 128; bf16 output only.
int conv_igemm_tma_launch(const IgemmParams& p, int block_n, cudaStream_t stream);

// Stem (Cin = 3) K layout: a 64-wide chunk holds `rows` filter rows of 16/rows pixels x 4 channels
// ([16 px][4 ch] for rows = 1, [8 px][2 rows][4 ch] over the row-pair image layout for rows = 2).
// rows = 2 (K = ceil(KH/2)*64) when KW <= 8 and stride == 2, else 1 (K = KH*64).
inline int stem_rows_per_chunk(int KW, int stride) { return (KW <= 8 && stride == 2) ? 2 : 1; }
// Activation maps for the stem over the padded image (t2r_stem_pack_image layout); < 0 on error.
int make_stem_maps(CUtensorMap* maps, const void* x4p, int N, int Hp, int Wp, int KW, int stride, int Ho, int Wo,
                   int TW, int TH);
// Tap table of the stem; returns the number of taps (= 64-wide K chunks).
int make_stem_taps(ConvTap* taps, int KH, int KW, int stride);

// Stride-1 KxK convolution through the shared-memory halo kernel (conv_halo.cu).
struct HaloRequest {
  const void* x;       // [N,H,W,C] bf16, the tensor the taps slide over
  int N, H, W, C;
  const void* w;       // [Cout][Ktot] bf16, K-major
  uint64_t Ktot;
  ConvTap taps[kMaxTaps];
  int n_taps;
  int Ho, Wo, Cout;    // output iteration space and its channel count
  long long os_n, os_h, os_w;
  void* out;
  const void* residual;
  const float* bias;
  int flags;
  double* stats;       // optional fused bn_stats output, fp64 [2*Cout]
  const void* bn_x;    // kEpiBnBwd operands (see IgemmParams)
  const float* bn_scale;
  const float* bn_shift;
};
bool conv_halo_eligible(int stride, int n_taps, int k_channels, int n_channels);
int conv_halo_launch(const HaloRequest& r, cudaStream_t stream);

// Weight gradient of stride-1 KxK convolutions with 64 input channels through the halo kernel
// (conv_wgrad_halo.cu).
bool conv_wgrad_halo_eligible(int stride, int n_taps, int Cin, int Cout);
// Reduction pass of the batch-norm backward (norm.cu): red[c] += sum dz, red[C + c] += sum dz * x with
// dz = dy * [scale * x + shift > 0] when relu; red is fp64 [2C], caller-zeroed.
int bn_bwd_reduce_launch(const void* dy, const void* x, long long rows, int C, const float* mean, const float* invstd,
                         const float* scale, const float* shift, int relu, double* red, cudaStream_t stream);

int conv_wgrad_halo_launch(const void* x, const void* dy, float* dw, int N, int H, int W, int Ho, int Wo, int Cout,
                           const ConvTap* taps, int n_taps, cudaStream_t stream);

}  // namespace t2r
