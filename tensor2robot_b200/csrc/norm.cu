// norm.cu — batch normalisation (training + inference) over bf16 [rows, C] tensors.
//
// HBM-bound kernels: 16-byte vector loads (8 bf16 channels per thread), fp32 per-thread partial
// sums, fp64 cross-block combination.  Semantics follow slim.batch_norm /
// tf.layers.batch_normalization(fused=True) as used by research/qtopt/networks.py:396-410 and
// layers/film_resnet_model.py:50-57: normalise with the biased batch variance, feed the
// Bessel-corrected variance into the moving average, epsilon inside the sqrt.
#include <algorithm>
#include <cstdlib>

#include "conv_common.cuh"

namespace t2r {

struct RowPartition {
  int cgb;          // column groups (of 8 channels) handled per block in x
  int lanes_r;      // row lanes per block
  int col_blocks;   // grid.y
  long long rows_per_block;
  int row_blocks;   // grid.x
};

// blocks_per_sm: resident CTAs per SM of the kernel that uses the partition (register limited), so
// that the grid is exactly one full wave: a 4/SM grid on a kernel that fits 3/SM runs a second,
// third-full wave and loses a third of the bandwidth.
static RowPartition partition(long long rows, int C, int blocks_per_sm = 4) {
  RowPartition p;
  const int cg = C / 8;
  p.cgb = std::min(cg, 256);
  while (256 % p.cgb != 0) --p.cgb;  // keep 256 % cgb == 0 (C = 192 -> cg 24 -> cgb 16)
  p.col_blocks = (cg + p.cgb - 1) / p.cgb;
  p.lanes_r = 256 / p.cgb;
  const long long target_blocks = std::max(1LL, (long long)num_sms() * blocks_per_sm / p.col_blocks);
  long long rpb = (rows + target_blocks - 1) / target_blocks;
  rpb = std::max<long long>(rpb, p.lanes_r);
  rpb = (rpb + p.lanes_r - 1) / p.lanes_r * p.lanes_r;
  p.rows_per_block = rpb;
  p.row_blocks = int((rows + rpb - 1) / rpb);
  static const int interleave = std::getenv("T2R_BN_INTERLEAVE") ? atoi(std::getenv("T2R_BN_INTERLEAVE")) : 1;
  if (interleave) p.rows_per_block = -1;
  return p;
}

__device__ __forceinline__ void unpack8(const uint4 q, float (&f)[8]) {
  f[0] = bf16_lo(q.x); f[1] = bf16_hi(q.x); f[2] = bf16_lo(q.y); f[3] = bf16_hi(q.y);
  f[4] = bf16_lo(q.z); f[5] = bf16_hi(q.z); f[6] = bf16_lo(q.w); f[7] = bf16_hi(q.w);
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 q;
  q.x = pack_bf16(f[0], f[1]); q.y = pack_bf16(f[2], f[3]);
  q.z = pack_bf16(f[4], f[5]); q.w = pack_bf16(f[6], f[7]);
  return q;
}

// Block-level reduce of 16 per-thread partials across the row lanes, then fp64 atomics.
__device__ __forceinline__ void block_reduce_16(float (&a)[8], float (&b)[8], int cgb, int lanes_r,
                                                int cgi, int C, double* out_a, double* out_b) {
  __shared__ float sm[256][17];
  const int tid = threadIdx.x;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sm[tid][j] = a[j];
    sm[tid][8 + j] = b[j];
  }
  __syncthreads();
  // thread t < cgb*16 sums value (t % 16) of column group (t / 16) over the row lanes
  for (int t = tid; t < cgb * 16; t += 256) {
    const int g = t / 16, j = t % 16;
    float s = 0.f;
    for (int r = 0; r < lanes_r; ++r) s += sm[r * cgb + g][j];
    const int cg_global = blockIdx.y * cgb + g;
    const int c = cg_global * 8 + (j & 7);
    if (c < C) atomicAdd((j < 8 ? out_a : out_b) + c, double(s));
  }
  (void)cgi;
}

__global__ void __launch_bounds__(256) bn_stats_kernel(const uint4* __restrict__ x, long long rows,
                                                       int C, int cgb, int lanes_r,
                                                       long long rows_per_block, double* stats) {
  const int cg = C / 8;
  const int g = threadIdx.x % cgb, rl = threadIdx.x / cgb;
  const int cgi = blockIdx.y * cgb + g;
  float s[8] = {0, 0, 0, 0, 0, 0, 0, 0}, q[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (cgi < cg) {
    // rows_per_block < 0: interleaved mode, the blocks sweep the tensor together in chunks of lanes_r rows
    const bool il = rows_per_block < 0;
    const long long r0 = il ? blockIdx.x * (long long)lanes_r : blockIdx.x * rows_per_block;
    const long long r1 = il ? rows : min(r0 + rows_per_block, rows);
    const long long rstep = il ? (long long)gridDim.x * lanes_r : (long long)lanes_r;
#pragma unroll 4
    for (long long r = r0 + rl; r < r1; r += rstep) {
      float f[8];
      unpack8(x[r * cg + cgi], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        s[j] += f[j];
        q[j] += f[j] * f[j];
      }
    }
  }
  block_reduce_16(s, q, cgb, lanes_r, cgi, C, stats, stats + C);
}

__global__ void bn_finalize_kernel(const double* stats, long long rows, int C, const float* gamma,
                                   const float* beta, float eps, float momentum, float* moving_mean,
                                   float* moving_var, float* mean_out, float* invstd_out,
                                   float* scale, float* shift) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double mean = stats[c] / double(rows);
  double var = stats[C + c] / double(rows) - mean * mean;
  if (var < 0) var = 0;
  const float invstd = float(1.0 / sqrt(var + double(eps)));
  const float sc = gamma ? gamma[c] * invstd : invstd;
  const float b = beta ? beta[c] : 0.f;
  mean_out[c] = float(mean);
  invstd_out[c] = invstd;
  scale[c] = sc;
  shift[c] = b - float(mean) * sc;
  if (moving_mean) moving_mean[c] = moving_mean[c] * momentum + float(mean) * (1.f - momentum);
  if (moving_var) {
    const double unbiased = rows > 1 ? var * double(rows) / double(rows - 1) : var;
    moving_var[c] = moving_var[c] * momentum + float(unbiased) * (1.f - momentum);
  }
}

__global__ void bn_infer_params_kernel(int C, const float* gamma, const float* beta,
                                       const float* moving_mean, const float* moving_var, float eps,
                                       float* scale, float* shift) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float invstd = rsqrtf(moving_var[c] + eps);
  const float sc = gamma ? gamma[c] * invstd : invstd;
  scale[c] = sc;
  shift[c] = (beta ? beta[c] : 0.f) - moving_mean[c] * sc;
}

template <bool FILM>
__global__ void __launch_bounds__(256) bn_apply_kernel(const uint4* __restrict__ x, uint4* __restrict__ y,
                                                       long long total8, int cg,
                                                       const float* __restrict__ scale,
                                                       const float* __restrict__ shift,
                                                       const float* __restrict__ film,
                                                       long long rows_per_image, int relu) {
  const int C = cg * 8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total8;
       i += (long long)gridDim.x * blockDim.x) {
    const int g = int(i % cg);
    float f[8];
    unpack8(x[i], f);
    const float4 s0 = __ldg(reinterpret_cast<const float4*>(scale) + 2 * g);
    const float4 s1 = __ldg(reinterpret_cast<const float4*>(scale) + 2 * g + 1);
    const float4 h0 = __ldg(reinterpret_cast<const float4*>(shift) + 2 * g);
    const float4 h1 = __ldg(reinterpret_cast<const float4*>(shift) + 2 * g + 1);
    const float sc[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
    const float sh[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = fmaf(f[j], sc[j], sh[j]);
    if (FILM) {
      const long long img = (i / cg) / rows_per_image;
      const float* fg = film + img * 2 * C + g * 8;
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = fmaf(1.f + __ldg(fg + j), f[j], __ldg(fg + C + j));
    }
    if (relu) {
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = fmaxf(f[j], 0.f);
    }
    y[i] = pack8(f);
  }
}

// pass 1 of backward: sum(dz), sum(dz * xhat) per channel, dz = dy * [relu mask]
__global__ void __launch_bounds__(256, 4) bn_bwd_reduce_kernel(
    const uint4* __restrict__ dy, const uint4* __restrict__ x, long long rows, int C, int cgb,
    int lanes_r, long long rows_per_block, const float* __restrict__ mean,
    const float* __restrict__ invstd, const float* __restrict__ scale,
    const float* __restrict__ shift, int relu, double* red) {
  const int cg = C / 8;
  const int g = threadIdx.x % cgb, rl = threadIdx.x / cgb;
  const int cgi = blockIdx.y * cgb + g;
  float s[8] = {0, 0, 0, 0, 0, 0, 0, 0}, q[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (cgi < cg) {
    // q accumulates sum(dz * x) (raw); bn_bwd_finalize turns it into sum(dz * xhat) = invstd * (q - mean * s),
    // which keeps mean / invstd out of the loop (16 registers -> one more resident CTA per SM).
    float sc[8], sh[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      sc[j] = scale[cgi * 8 + j];
      sh[j] = shift[cgi * 8 + j];
    }
    // rows_per_block < 0: interleaved mode, the blocks sweep the tensor together in chunks of lanes_r rows
    const bool il = rows_per_block < 0;
    const long long r0 = il ? blockIdx.x * (long long)lanes_r : blockIdx.x * rows_per_block;
    const long long r1 = il ? rows : min(r0 + rows_per_block, rows);
    const long long rstep = il ? (long long)gridDim.x * lanes_r : (long long)lanes_r;
#pragma unroll 2
    for (long long r = r0 + rl; r < r1; r += rstep) {
      float fx[8], fd[8];
      unpack8(x[r * cg + cgi], fx);
      unpack8(dy[r * cg + cgi], fd);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float z = fmaf(fx[j], sc[j], sh[j]);
        const float dz = (relu && !(z > 0.f)) ? 0.f : fd[j];
        s[j] += dz;
        q[j] = fmaf(dz, fx[j], q[j]);
      }
    }
  }
  block_reduce_16(s, q, cgb, lanes_r, cgi, C, red, red + C);
}

__global__ void bn_bwd_finalize_kernel(const double* red, int C, const float* mean, const float* invstd,
                                       float* dgamma, float* dbeta) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  dbeta[c] = float(red[c]);
  dgamma[c] = float((red[C + c] - double(mean[c]) * red[c]) * double(invstd[c]));
}

// t2r_bn_backward_gemm_finalize: sums[c] = sum g, sums[C + c] = sum g * x from t2r_conv2d_wgrad_bnsums.  Writes
// dgamma / dbeta as bn_bwd_finalize_kernel and the apply coefficients kb, kc of bn_bwd_apply_kernel into coef [2C].
__global__ void bn_bwd_gemm_finalize_kernel(const double* sums, int C, float inv_rows, const float* mean,
                                            const float* invstd, const float* scale, float* dgamma, float* dbeta,
                                            float* coef) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float db = float(sums[c]);
  const float dg = float((sums[C + c] - double(mean[c]) * sums[c]) * double(invstd[c]));
  dbeta[c] = db;
  dgamma[c] = dg;
  const float t = scale[c] * dg * inv_rows * invstd[c];
  coef[c] = -t;
  coef[C + c] = t * mean[c] - scale[c] * db * inv_rows;
}

// pass 2: dx = scale * (dz - sum(dz)/rows - xhat * sum(dz*xhat)/rows) (+ dres)
//            = scale*dz + kb*x + kc   with per-channel kb, kc.
// Row-partitioned like the reductions: a thread owns one 8-channel group, so the coefficients
// stay in registers and the loop body is 2-3 16-byte loads and one 16-byte store per 8 elements.
template <bool RES>
__global__ void __launch_bounds__(256) bn_bwd_apply_kernel(
    const uint4* __restrict__ dy, const uint4* __restrict__ x, const uint4* __restrict__ dres,
    uint4* __restrict__ dx, long long rows, int C, int cgb, int lanes_r, long long rows_per_block,
    float inv_rows, const float* __restrict__ mean, const float* __restrict__ invstd,
    const float* __restrict__ scale, const float* __restrict__ shift, const float* __restrict__ dgamma,
    const float* __restrict__ dbeta, int relu) {
  const int cg = C / 8;
  const int g = threadIdx.x % cgb, rl = threadIdx.x / cgb;
  const int cgi = blockIdx.y * cgb + g;
  if (cgi >= cg) return;
  float sc[8], sh[8], kb[8], kc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int c = cgi * 8 + j;
    sc[j] = scale[c];
    sh[j] = shift[c];
    const float t = sc[j] * dgamma[c] * inv_rows * invstd[c];
    kb[j] = -t;
    kc[j] = t * mean[c] - sc[j] * dbeta[c] * inv_rows;
  }
  // rows_per_block < 0: interleaved mode, the blocks sweep the tensor together in chunks of lanes_r rows
  const bool il = rows_per_block < 0;
  const long long r0 = il ? blockIdx.x * (long long)lanes_r : blockIdx.x * rows_per_block;
  const long long r1 = il ? rows : min(r0 + rows_per_block, rows);
  const long long rstep = il ? (long long)gridDim.x * lanes_r : (long long)lanes_r;
#pragma unroll 2
  for (long long r = r0 + rl; r < r1; r += rstep) {
    const long long i = r * cg + cgi;
    float fx[8], fd[8], fo[8];
    const uint4 qx = x[i], qd = dy[i];
    uint4 qr;
    if (RES) qr = dres[i];
    unpack8(qx, fx);
    unpack8(qd, fd);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float z = fmaf(fx[j], sc[j], sh[j]);
      const float dz = (relu && !(z > 0.f)) ? 0.f : fd[j];
      fo[j] = fmaf(sc[j], dz, fmaf(kb[j], fx[j], kc[j]));
    }
    if (RES) {
      float fr[8];
      unpack8(qr, fr);
#pragma unroll
      for (int j = 0; j < 8; ++j) fo[j] += fr[j];
    }
    dx[i] = pack8(fo);
  }
}

// y = relu?(x*scale + shift), row-partitioned (no FiLM).
__global__ void __launch_bounds__(256, 6) bn_apply_rows_kernel(const uint4* __restrict__ x, uint4* __restrict__ y,
                                                            long long rows, int C, int cgb, int lanes_r,
                                                            long long rows_per_block,
                                                            const float* __restrict__ scale,
                                                            const float* __restrict__ shift, int relu) {
  const int cg = C / 8;
  const int g = threadIdx.x % cgb, rl = threadIdx.x / cgb;
  const int cgi = blockIdx.y * cgb + g;
  if (cgi >= cg) return;
  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sc[j] = scale[cgi * 8 + j];
    sh[j] = shift[cgi * 8 + j];
  }
  // rows_per_block < 0: interleaved mode, the blocks sweep the tensor together in chunks of lanes_r rows
  const bool il = rows_per_block < 0;
  const long long r0 = il ? blockIdx.x * (long long)lanes_r : blockIdx.x * rows_per_block;
  const long long r1 = il ? rows : min(r0 + rows_per_block, rows);
  const long long rstep = il ? (long long)gridDim.x * lanes_r : (long long)lanes_r;
#pragma unroll 4
  for (long long r = r0 + rl; r < r1; r += rstep) {
    const long long i = r * cg + cgi;
    float f[8];
    unpack8(x[i], f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      f[j] = fmaf(f[j], sc[j], sh[j]);
      if (relu) f[j] = fmaxf(f[j], 0.f);
    }
    y[i] = pack8(f);
  }
}

int bn_bwd_reduce_launch(const void* dy, const void* x, long long rows, int C, const float* mean, const float* invstd,
                         const float* scale, const float* shift, int relu, double* red, cudaStream_t stream) {
  const RowPartition pr = partition(rows, C, 4);   // <= 64 registers/thread: 4 CTAs per SM
  bn_bwd_reduce_kernel<<<dim3(pr.row_blocks, pr.col_blocks), 256, 0, stream>>>(
      static_cast<const uint4*>(dy), static_cast<const uint4*>(x), rows, C, pr.cgb, pr.lanes_r,
      pr.rows_per_block, mean, invstd, scale, shift, relu, red);
  T2R_LAUNCH_OK();
  return T2R_OK;
}

static inline int grid_for(long long n) {
  return int(std::min<long long>(std::max<long long>((n + 255) / 256, 1), 148LL * 16));
}

// ---------------------------------------------------------------------------------------------
// FiLM batch norm backward:  h = x*sc + sh,  z = (1 + g[n,c]) * h + b[n,c],  y = relu?(z)
// (layers/film_resnet_model.py:108-115 after :50-57).  Per-image sums first:
//   S1[n,c] = sum_pixels dz,  S3[n,c] = sum_pixels dz * x,   dz = dy * [z > 0]
// from which d b = S1, d g = sc*S3 + sh*S1 and the batch-norm sums over dh = (1 + g) * dz follow.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bn_film_bwd_reduce_kernel(
    const uint4* __restrict__ dy, const uint4* __restrict__ x, const float* __restrict__ film, int HW, int cg,
    const float* __restrict__ scale, const float* __restrict__ shift, int relu, float* __restrict__ sums) {
  __shared__ float sm[8][32][17];
  const int n = blockIdx.x;
  const int g = blockIdx.y * 32 + threadIdx.x;
  const int C = cg * 8;
  float s1[8] = {0, 0, 0, 0, 0, 0, 0, 0}, s3[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (g < cg) {
    float sc[8], sh[8], fg[8], fb[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      sc[j] = scale[g * 8 + j];
      sh[j] = shift[g * 8 + j];
      fg[j] = 1.f + film[(long long)n * 2 * C + g * 8 + j];
      fb[j] = film[(long long)n * 2 * C + C + g * 8 + j];
    }
    for (int p = threadIdx.y; p < HW; p += 8) {
      const long long i = ((long long)n * HW + p) * cg + g;
      float fx[8], fd[8];
      unpack8(x[i], fx);
      unpack8(dy[i], fd);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float z = fmaf(fg[j], fmaf(fx[j], sc[j], sh[j]), fb[j]);
        const float dz = (relu && !(z > 0.f)) ? 0.f : fd[j];
        s1[j] += dz;
        s3[j] = fmaf(dz, fx[j], s3[j]);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sm[threadIdx.y][threadIdx.x][j] = s1[j];
    sm[threadIdx.y][threadIdx.x][8 + j] = s3[j];
  }
  __syncthreads();
  if (threadIdx.y == 0 && g < cg) {
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      float s = 0.f;
      for (int r = 0; r < 8; ++r) s += sm[r][threadIdx.x][j];
      sums[((long long)n * 2 + (j >> 3)) * C + g * 8 + (j & 7)] = s;   // [N][2][C]
    }
  }
}

// dfilm [N][2C] (gamma part, beta part) and the batch-norm sums (fp64 over images).
__global__ void bn_film_bwd_finalize_kernel(const float* sums, const float* film, int N, int C, const float* mean,
                                            const float* invstd, const float* scale, const float* shift,
                                            float* dfilm, float* dgamma, float* dbeta) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double sdh = 0.0, sdhx = 0.0;
  for (int n = 0; n < N; ++n) {
    const float s1 = sums[((long long)n * 2) * C + c], s3 = sums[((long long)n * 2 + 1) * C + c];
    const float g1 = 1.f + film[(long long)n * 2 * C + c];
    dfilm[(long long)n * 2 * C + c] = fmaf(scale[c], s3, shift[c] * s1);   // d gamma_film = sum dz * h
    dfilm[(long long)n * 2 * C + C + c] = s1;                               // d beta_film  = sum dz
    sdh += double(g1) * s1;
    sdhx += double(g1) * s3;
  }
  dbeta[c] = float(sdh);
  dgamma[c] = float((sdhx - double(mean[c]) * sdh) * double(invstd[c]));
}

__global__ void __launch_bounds__(256) bn_film_bwd_apply_kernel(
    const uint4* __restrict__ dy, const uint4* __restrict__ x, const uint4* __restrict__ dres, uint4* __restrict__ dx,
    const float* __restrict__ film, long long total8, int HW, int cg, float inv_rows, const float* __restrict__ mean,
    const float* __restrict__ invstd, const float* __restrict__ scale, const float* __restrict__ shift,
    const float* __restrict__ dgamma, const float* __restrict__ dbeta, int relu) {
  const int C = cg * 8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total8;
       i += (long long)gridDim.x * blockDim.x) {
    const int g = int(i % cg);
    const long long n = (i / cg) / HW;
    float fx[8], fd[8], fo[8];
    unpack8(x[i], fx);
    unpack8(dy[i], fd);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = g * 8 + j;
      const float sc = scale[c], sh = shift[c];
      const float fg = 1.f + film[n * 2 * C + c], fb = film[n * 2 * C + C + c];
      const float z = fmaf(fg, fmaf(fx[j], sc, sh), fb);
      const float dh = ((relu && !(z > 0.f)) ? 0.f : fd[j]) * fg;
      const float t = sc * dgamma[c] * inv_rows * invstd[c];
      fo[j] = fmaf(sc, dh, fmaf(-t, fx[j], t * mean[c] - sc * dbeta[c] * inv_rows));
    }
    if (dres != nullptr) {
      float fr[8];
      unpack8(dres[i], fr);
#pragma unroll
      for (int j = 0; j < 8; ++j) fo[j] += fr[j];
    }
    dx[i] = pack8(fo);
  }
}

}  // namespace t2r

using namespace t2r;

extern "C" int32_t t2r_bn_stats(const void* x, int64_t rows, int32_t C, double* stats, void* stream) {
  T2R_CHECK_ARG(x && stats && rows > 0 && C > 0 && C % 8 == 0, "bn_stats: C=%d must be a multiple of 8", C);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  T2R_CUDA_OK(cudaMemsetAsync(stats, 0, sizeof(double) * 2 * C, st));
  const RowPartition p = partition(rows, C);
  bn_stats_kernel<<<dim3(p.row_blocks, p.col_blocks), 256, 0, st>>>(
      static_cast<const uint4*>(x), rows, C, p.cgb, p.lanes_r, p.rows_per_block, stats);
  T2R_LAUNCH_OK();
  return T2R_OK;
}

extern "C" int32_t t2r_bn_finalize(const double* stats, int64_t rows, int32_t C, const float* gamma,
                                   const float* beta, float eps, float momentum, float* moving_mean,
                                   float* moving_var, float* mean, float* invstd, float* scale,
                                   float* shift, void* stream) {
  T2R_CHECK_ARG(stats && mean && invstd && scale && shift && rows > 0 && C > 0, "bn_finalize: bad args");
  bn_finalize_kernel<<<(C + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      stats, rows, C, gamma, beta, eps, momentum, moving_mean, moving_var, mean, invstd, scale, shift);
  T2R_LAUNCH_OK();
  return T2R_OK;
}

extern "C" int32_t t2r_bn_infer_params(int32_t C, const float* gamma, const float* beta,
                                       const float* moving_mean, const float* moving_var, float eps,
                                       float* scale, float* shift, void* stream) {
  T2R_CHECK_ARG(moving_mean && moving_var && scale && shift && C > 0, "bn_infer_params: bad args");
  bn_infer_params_kernel<<<(C + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      C, gamma, beta, moving_mean, moving_var, eps, scale, shift);
  T2R_LAUNCH_OK();
  return T2R_OK;
}

extern "C" int32_t t2r_bn_apply(const void* x, void* y, int64_t rows, int32_t C, const float* scale,
                                const float* shift, const float* film, int64_t rows_per_image,
                                int32_t relu, void* stream) {
  T2R_CHECK_ARG(x && y && scale && shift && rows > 0 && C > 0 && C % 8 == 0, "bn_apply: bad args");
  T2R_CHECK_ARG(!film || rows_per_image > 0, "bn_apply: film needs rows_per_image");
  const long long total8 = rows * (C / 8);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (film)
    bn_apply_kernel<true><<<grid_for(total8), 256, 0, st>>>(static_cast<const uint4*>(x), static_cast<uint4*>(y),
                                                            total8, C / 8, scale, shift, film, rows_per_image, relu);
  else {
    const RowPartition p = partition(rows, C, 6);   // <= 40 registers/thread: 6 CTAs per SM
    bn_apply_rows_kernel<<<dim3(p.row_blocks, p.col_blocks), 256, 0, st>>>(
        static_cast<const uint4*>(x), static_cast<uint4*>(y), rows, C, p.cgb, p.lanes_r, p.rows_per_block, scale,
        shift, relu);
  }
  T2R_LAUNCH_OK();
  return T2R_OK;
}

extern "C" int32_t t2r_bn_backward(const void* dy, const void* x, const void* dres, void* dx,
                                   int64_t rows, int32_t C, const float* gamma, const float* mean,
                                   const float* invstd, const float* scale, const float* shift,
                                   int32_t relu, double* red, float* dgamma, float* dbeta,
                                   void* stream) {
  (void)gamma;
  T2R_CHECK_ARG(dy && x && dx && mean && invstd && scale && shift && red && dgamma && dbeta,
                "bn_backward: null pointer");
  T2R_CHECK_ARG(rows > 0 && C > 0 && C % 8 == 0, "bn_backward: bad shape");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  T2R_CUDA_OK(cudaMemsetAsync(red, 0, sizeof(double) * 2 * C, st));
  if (int rc = bn_bwd_reduce_launch(dy, x, rows, C, mean, invstd, scale, shift, relu, red, st)) return rc;
  return t2r_bn_backward_presummed(dy, x, dres, dx, rows, C, mean, invstd, scale, shift, relu, red, dgamma, dbeta,
                                   stream);
}

extern "C" int32_t t2r_bn_backward_presummed(const void* dy, const void* x, const void* dres, void* dx,
                                             int64_t rows, int32_t C, const float* mean, const float* invstd,
                                             const float* scale, const float* shift, int32_t relu,
                                             const double* red, float* dgamma, float* dbeta, void* stream) {
  T2R_CHECK_ARG(dy && x && dx && mean && invstd && scale && shift && red && dgamma && dbeta,
                "bn_backward_presummed: null pointer");
  T2R_CHECK_ARG(rows > 0 && C > 0 && C % 8 == 0, "bn_backward_presummed: bad shape");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const RowPartition p = partition(rows, C, 4);    // 64 registers/thread: 4 CTAs per SM
  bn_bwd_finalize_kernel<<<(C + 127) / 128, 128, 0, st>>>(red, C, mean, invstd, dgamma, dbeta);
  T2R_LAUNCH_OK();
  const float inv_rows = 1.f / float(rows);
  const dim3 grid(p.row_blocks, p.col_blocks);
  if (dres)
    bn_bwd_apply_kernel<true><<<grid, 256, 0, st>>>(
        static_cast<const uint4*>(dy), static_cast<const uint4*>(x), static_cast<const uint4*>(dres),
        static_cast<uint4*>(dx), rows, C, p.cgb, p.lanes_r, p.rows_per_block, inv_rows, mean, invstd, scale,
        shift, dgamma, dbeta, relu);
  else
    bn_bwd_apply_kernel<false><<<grid, 256, 0, st>>>(
        static_cast<const uint4*>(dy), static_cast<const uint4*>(x), nullptr, static_cast<uint4*>(dx), rows, C,
        p.cgb, p.lanes_r, p.rows_per_block, inv_rows, mean, invstd, scale, shift, dgamma, dbeta, relu);
  T2R_LAUNCH_OK();
  return T2R_OK;
}

extern "C" int32_t t2r_bn_backward_gemm_finalize(const double* sums, int64_t rows, int32_t C, const float* mean,
                                                 const float* invstd, const float* scale, float* dgamma, float* dbeta,
                                                 float* coef, void* stream) {
  T2R_CHECK_ARG(sums && mean && invstd && scale && dgamma && dbeta && coef, "bn_backward_gemm_finalize: null pointer");
  T2R_CHECK_ARG(rows > 0 && C > 0, "bn_backward_gemm_finalize: bad shape");
  bn_bwd_gemm_finalize_kernel<<<(C + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      sums, C, 1.f / float(rows), mean, invstd, scale, dgamma, dbeta, coef);
  T2R_LAUNCH_OK();
  return T2R_OK;
}

extern "C" int32_t t2r_bn_film_backward(const void* dy, const void* x, const float* film, const void* dres, void* dx,
                                        float* dfilm, int64_t rows, int32_t C, int64_t rows_per_image,
                                        const float* mean, const float* invstd, const float* scale,
                                        const float* shift, int32_t relu, float* sums_ws, float* dgamma,
                                        float* dbeta, void* stream) {
  T2R_CHECK_ARG(dy && x && film && dx && dfilm && mean && invstd && scale && shift && sums_ws && dgamma && dbeta,
                "bn_film_backward: null pointer");
  T2R_CHECK_ARG(rows > 0 && C > 0 && C % 8 == 0 && rows_per_image > 0 && rows % rows_per_image == 0 &&
                    rows_per_image < (1LL << 31), "bn_film_backward: bad shape");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int N = int(rows / rows_per_image), cg = C / 8, HW = int(rows_per_image);
  bn_film_bwd_reduce_kernel<<<dim3(N, (cg + 31) / 32), dim3(32, 8), 0, st>>>(
      static_cast<const uint4*>(dy), static_cast<const uint4*>(x), film, HW, cg, scale, shift, relu, sums_ws);
  T2R_LAUNCH_OK();
  bn_film_bwd_finalize_kernel<<<(C + 127) / 128, 128, 0, st>>>(sums_ws, film, N, C, mean, invstd, scale, shift, dfilm,
                                                               dgamma, dbeta);
  T2R_LAUNCH_OK();
  const long long total8 = rows * cg;
  bn_film_bwd_apply_kernel<<<grid_for(total8), 256, 0, st>>>(
      static_cast<const uint4*>(dy), static_cast<const uint4*>(x), static_cast<const uint4*>(dres),
      static_cast<uint4*>(dx), film, total8, HW, cg, 1.f / float(rows), mean, invstd, scale, shift, dgamma, dbeta, relu);
  T2R_LAUNCH_OK();
  return T2R_OK;
}

// Column sums of a bf16 [rows, C] matrix (bias gradients): the bn_stats partition (fills every SM)
// followed by a fp64 -> fp32 conversion.
namespace t2r {
__global__ void colsum_finalize_kernel(const double* stats, int C, float* out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) out[c] = float(stats[c]);
}
}  // namespace t2r

extern "C" int32_t t2r_colsum_bf16(const void* x, int64_t rows, int32_t C, double* stats, float* out,
                                   void* stream) {
  T2R_CHECK_ARG(out != nullptr, "colsum_bf16: null output");
  if (int32_t rc = t2r_bn_stats(x, rows, C, stats, stream)) return rc;
  t2r::colsum_finalize_kernel<<<(C + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(stats, C, out);
  T2R_LAUNCH_OK();
  return T2R_OK;
}
