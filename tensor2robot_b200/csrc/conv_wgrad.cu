// conv_wgrad.cu — convolution weight gradient on tcgen05 (sm_100a).
//
//   dW[co, tap, ci] = sum over output pixels  dY[pix, co] * X[pix shifted by tap, ci]
//
// The reduction dimension (K of the GEMM) is the pixel index, which is the *slow* dimension of
// both NHWC operands, so both operands are fed to the tensor core as MN-major tiles: a TMA box
// of [64 pixels x 64 channels] lands in shared memory as 64 rows of 128 bytes (128B swizzle),
// which is exactly the canonical MN-major SW128 UMMA layout (8-row atoms, SBO = 1024 B), and
// several 64-channel tiles side by side form the M / N extent (LBO = tile size).
//
//   A: two X tiles  -> M = 128 rows = 128 consecutive columns of the OHWI weight row
//        (k = tap*Cin + ci; for Cin = 64 the two tiles are two filter taps)
//   B: BLOCK_N/64 dY tiles -> N = BLOCK_N output channels
//   D: [128 x BLOCK_N] fp32 per "group" in TMEM; a CTA owns up to 512/BLOCK_N groups and a
//      range of pixel tiles (split-K), and flushes with fp32 atomics (red.global.add.f32).
//
// The dY tiles of a pixel tile are shared by all groups of the CTA, so they travel through their
// own (shallow) ring and are loaded once per pixel tile; the X tiles stream through a deeper ring.
// (L2 -> SMEM traffic per MMA drops from 12 KB to 8 KB at BLOCK_N = 256, 8 -> 5 KB at 128.)
//
// Replaces the autodiff filter gradients of slim.conv2d / tf.layers.conv2d
// (research/qtopt/networks.py:443-591, layers/film_resnet_model.py:89-105).
#include <algorithm>
#include <cstdlib>

#include "conv_common.cuh"

namespace t2r {


struct WgradParams {
  CUtensorMap tmap_x[4];
  CUtensorMap tmap_dy;
  ConvTap taps[kMaxTaps];
  int chunks_per_tap;  // Cin / 64
  int n_slots;         // taps * chunks_per_tap (64-wide column blocks of the weight row)
  int n_groups;        // ceil(n_slots / 2)
  int groups_per_cta;  // G
  int n_gsets;         // ceil(n_groups / G)
  int n_chunks_n;      // Cout / BLOCK_N
  int ksplits;
  int TW, TH, tiles_w, tiles_h;
  int total_ptiles;    // N * tiles_w * tiles_h
  int Ktot;            // taps * Cin
  int Cout;
  float* dw;
  // kPro: x is the RAW tensor a batch norm normalised; the (otherwise idle) epilogue warps rewrite every landed
  // X tile as relu(bn_scale * x + bn_shift) before the MMA reads it (see kProBnRelu, conv_common.cuh)
  const float* bn_scale;
  const float* bn_shift;
  // kBnSums: 1x1 consumer of z = relu(bn_scale * x + bn_shift), x raw.  A group is ONE 64-channel chunk c: the
  // transform warps rewrite its landed x tile as m * x and write m = [bn_scale * x + bn_shift > 0] into the second
  // A slot, so that TMEM rows 0-63 hold P[c, n] = sum dy * m * x and rows 64-127 Q[c, n] = sum dy * m.  The epilogue
  // adds dw[n, c] += bn_scale * P + bn_shift * Q (= sum dy * z) and bn_sums[c] += sum_n w[c, n] * Q (= sum g),
  // bn_sums[Cin + c] += sum_n w[c, n] * P (= sum g * x), g = m * (dy conv_transpose w): the batch-norm reduction
  // without a pass over g.  w_dgrad: the bf16 [Cin][Cout] weights the data gradient multiplies with.
  const uint16_t* w_dgrad;
  double* bn_sums;
};

enum WgradMode { kWgPlain = 0, kWgBnRelu = 1, kWgBnSums = 2 };

// kWgBnSums operand transform on kN 16-byte pieces (8 channels, `step` bytes apart) of a SW128 x tile: x -> m * x in
// place and m (bf16 1.0 / 0.0) at the same position `mask_off` bytes further.  Both are exact in bf16; the mask test
// is the fmaf of bn_bwd_reduce_kernel (norm.cu).
template <int kN>
__device__ __forceinline__ void bnmask_pieces(uint32_t piece, uint32_t step, uint32_t mask_off, const float (&sc)[8],
                                              const float (&sh)[8]) {
  uint4 q[kN];
#pragma unroll
  for (int i = 0; i < kN; ++i)
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(q[i].x), "=r"(q[i].y), "=r"(q[i].z), "=r"(q[i].w)
                 : "r"(piece + uint32_t(i) * step)
                 : "memory");
#pragma unroll
  for (int i = 0; i < kN; ++i) {
    uint32_t w[4] = {q[i].x, q[i].y, q[i].z, q[i].w}, keep[4];
#pragma unroll
    for (int k = 0; k < 4; ++k)
      keep[k] = (fmaf(bf16_lo(w[k]), sc[2 * k], sh[2 * k]) > 0.f ? 0x0000FFFFu : 0u) |
                (fmaf(bf16_hi(w[k]), sc[2 * k + 1], sh[2 * k + 1]) > 0.f ? 0xFFFF0000u : 0u);
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(piece + uint32_t(i) * step), "r"(w[0] & keep[0]),
                 "r"(w[1] & keep[1]), "r"(w[2] & keep[2]), "r"(w[3] & keep[3])
                 : "memory");
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(piece + uint32_t(i) * step + mask_off),
                 "r"(keep[0] & 0x3F803F80u), "r"(keep[1] & 0x3F803F80u), "r"(keep[2] & 0x3F803F80u),
                 "r"(keep[3] & 0x3F803F80u)
                 : "memory");
  }
}

template <int BLOCK_N>
struct WgradCfg {
  static constexpr int kTileBytes = 64 * 128;  // 64 pixels x 64 channels bf16
  static constexpr int kNB = BLOCK_N / 64;
  static constexpr int kXBytes = 2 * kTileBytes;     // one group's A operand
  static constexpr int kDyBytes = kNB * kTileBytes;  // the pixel tile's B operand
  static constexpr int kXStages = BLOCK_N == 64 ? 10 : (BLOCK_N == 128 ? 8 : 6);
  static constexpr int kDyStages = 3;
  static constexpr int kMaxGroups = 512 / BLOCK_N;
  static constexpr int kSmemBytes = kXStages * kXBytes + kDyStages * kDyBytes + 1024 + 512;
};

template <int BLOCK_N, int kMode>
__global__ void __launch_bounds__(256, 1) conv_wgrad_kernel(const __grid_constant__ WgradParams p) {
  using Cfg = WgradCfg<BLOCK_N>;
  constexpr bool kPro = kMode != kWgPlain;   // the epilogue warps transform the landed X tiles
  constexpr bool kSums = kMode == kWgBnSums;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t dy_base = smem_base + Cfg::kXStages * Cfg::kXBytes;
  const uint32_t bar_base = dy_base + Cfg::kDyStages * Cfg::kDyBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (Cfg::kXStages + s); };
  auto dfull_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::kXStages + s); };
  auto dempty_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::kXStages + Cfg::kDyStages + s); };
  const uint32_t tfull_bar = bar_base + 8u * (2 * Cfg::kXStages + 2 * Cfg::kDyStages);
  const uint32_t tmem_ptr_addr = tfull_bar + 8u;
  auto ready_bar = [&](int s) { return tfull_bar + 16u + 8u * s; };
  volatile uint32_t* tmem_ptr_gen =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_ptr_addr - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < 4; ++i) tma_prefetch_desc(&p.tmap_x[i]);
    tma_prefetch_desc(&p.tmap_dy);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < Cfg::kXStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
      if (kPro) mbar_init(ready_bar(s), 4);
    }
    for (int s = 0; s < Cfg::kDyStages; ++s) {
      mbar_init(dfull_bar(s), 1);
      mbar_init(dempty_bar(s), 1);
    }
    mbar_init(tfull_bar, 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_ptr_addr, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_gen;

  // work item: (group set, output-channel chunk, pixel-tile range)
  int item = blockIdx.x;
  const int ks = item % p.ksplits; item /= p.ksplits;
  const int nc = item % p.n_chunks_n; item /= p.n_chunks_n;
  const int gs = item;
  const int g0 = gs * p.groups_per_cta;
  const int g1 = min(g0 + p.groups_per_cta, p.n_groups);
  const int pt0 = int((long long)p.total_ptiles * ks / p.ksplits);
  const int pt1 = int((long long)p.total_ptiles * (ks + 1) / p.ksplits);
  const int tiles_per_img = p.tiles_w * p.tiles_h;
  const int n0 = nc * BLOCK_N;

  if (warp == 0 || warp == 2 || warp == 3) {
    // Three producer warps (one per free SM sub-partition) take the loads round-robin: a TMA tile
    // load costs its whole latency per issuing warp, so one thread cannot keep the ring full
    // (profiles/r01_ncu_summary.md, section 3.3).
    if (lane == 0) {
      const int pid = warp == 0 ? 0 : warp - 1;
      int stage = 0, ds = 0, turn = 0, dturn = 0;
      uint32_t phase = 0, dphase = 0;
      for (int pt = pt0; pt < pt1; ++pt) {
        const int img = pt / tiles_per_img;
        const int rem = pt - img * tiles_per_img;
        const int oh0 = (rem / p.tiles_w) * p.TH;
        const int ow0 = (rem % p.tiles_w) * p.TW;
        if (dturn == pid) {
          mbar_wait(dempty_bar(ds), dphase ^ 1u);
          mbar_expect_tx(dfull_bar(ds), Cfg::kDyBytes);
#pragma unroll
          for (int j = 0; j < Cfg::kNB; ++j)
            tma_load_4d(dy_base + ds * Cfg::kDyBytes + j * Cfg::kTileBytes, &p.tmap_dy, dfull_bar(ds), n0 + j * 64,
                        ow0, oh0, img);
        }
        if (++dturn == 3) dturn = 0;
        if (++ds == Cfg::kDyStages) {
          ds = 0;
          dphase ^= 1u;
        }
        for (int g = g0; g < g1; ++g) {
          if (turn == pid) {
            mbar_wait(empty_bar(stage), phase ^ 1u);
            const uint32_t sa = smem_base + stage * Cfg::kXBytes;
            mbar_expect_tx(full_bar(stage), kSums ? Cfg::kTileBytes : Cfg::kXBytes);
            if (kSums) tma_load_4d(sa, &p.tmap_x[0], full_bar(stage), g * 64, ow0, oh0, img);
#pragma unroll
            for (int h = 0; h < (kSums ? 0 : 2); ++h) {
              int slot = 2 * g + h;
              if (slot >= p.n_slots) slot = p.n_slots - 1;  // duplicate: rows are never stored
              const int t = slot / p.chunks_per_tap;
              const int c = slot - t * p.chunks_per_tap;
              const ConvTap tap = p.taps[t];
              tma_load_4d(sa + h * Cfg::kTileBytes, &p.tmap_x[tap.map], full_bar(stage), c * 64, ow0 + tap.dw,
                          oh0 + tap.dh, img);
            }
          }
          if (++turn == 3) turn = 0;
          if (++stage == Cfg::kXStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // whole warp converged, elected lane issues (see conv_igemm.cu)
    {
      constexpr uint32_t idesc = make_idesc_bf16(128, BLOCK_N, 1, 1);
      const uint64_t a_base = make_smem_desc_sw128(smem_base, Cfg::kTileBytes, 1024);
      const uint64_t b_base = make_smem_desc_sw128(dy_base, Cfg::kTileBytes, 1024);
      int stage = 0, ds = 0;
      uint32_t phase = 0, dphase = 0;
      for (int pt = pt0; pt < pt1; ++pt) {
        mbar_wait(dfull_bar(ds), dphase);
        const uint64_t bs = b_base + uint64_t(uint32_t(ds) * uint32_t(Cfg::kDyBytes >> 4));
        for (int g = g0; g < g1; ++g) {
          mbar_wait(kPro ? ready_bar(stage) : full_bar(stage), phase);
          tc_fence_after();
          const uint64_t as_ = a_base + uint64_t(uint32_t(stage) * uint32_t(Cfg::kXBytes >> 4));
          const uint32_t d_tmem = tmem_base + (g - g0) * BLOCK_N;
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)  // 64 pixels = 4 x (K = 16)
            umma_bf16_elect(d_tmem, as_ + uint64_t(kk * 128), bs + uint64_t(kk * 128), idesc,
                            (pt > pt0 || kk > 0) ? 1u : 0u);
          umma_commit_elect(empty_bar(stage));
          if (++stage == Cfg::kXStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
        umma_commit_elect(dempty_bar(ds));
        if (++ds == Cfg::kDyStages) {
          ds = 0;
          dphase ^= 1u;
        }
      }
      umma_commit_elect(tfull_bar);
    }
  } else if (warp >= 4) {
    const int quad = warp - 4;
    const int row = quad * 32 + lane;
    if (kSums) {
      // operand transform: 128 threads over the 64 rows x 8 chunks of the group's x tile, 4 rows r0 + 16 i each
      const int t = threadIdx.x - 128;
      const uint32_t j = uint32_t(t) & 7u, r0 = uint32_t(t) >> 3;
      const uint32_t piece0 = r0 * 128u + ((j ^ (r0 & 7u)) << 4);
      int stage = 0;
      uint32_t phase = 0;
      for (int pt = pt0; pt < pt1; ++pt)
        for (int g = g0; g < g1; ++g) {
          float sc[8], sh[8];
          load8(p.bn_scale + g * 64 + j * 8, sc);
          load8(p.bn_shift + g * 64 + j * 8, sh);
          mbar_wait(full_bar(stage), phase);
          bnmask_pieces<4>(smem_base + stage * Cfg::kXBytes + piece0, 2048u, Cfg::kTileBytes, sc, sh);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(ready_bar(stage));
          if (++stage == Cfg::kXStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
    } else if (kPro) {
      // operand transform: thread t works on tile h = t / 64 of the stage (64 rows x 128 B), logical chunk t & 7 of
      // rows ((t & 63) >> 3) + 8 i: a quarter warp covers one full row, a thread's rows share r & 7
      const int t = threadIdx.x - 128;
      const int h = t >> 6;
      const uint32_t j = uint32_t(t) & 7u, r0 = (uint32_t(t) & 63u) >> 3;
      const uint32_t piece0 = uint32_t(h) * Cfg::kTileBytes + r0 * 128u + ((j ^ r0) << 4);
      int stage = 0;
      uint32_t phase = 0;
      for (int pt = pt0; pt < pt1; ++pt)
        for (int g = g0; g < g1; ++g) {
          int slot = 2 * g + h;
          if (slot >= p.n_slots) slot = p.n_slots - 1;
          const int c = slot % p.chunks_per_tap;
          float sc[8], sh[8];
          load8(p.bn_scale + c * 64 + j * 8, sc);
          load8(p.bn_shift + c * 64 + j * 8, sh);
          mbar_wait(full_bar(stage), phase);
          bnrelu_pieces_inplace<8>(smem_base + stage * Cfg::kXBytes + piece0, 1024u, sc, sh);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(ready_bar(stage));
          if (++stage == Cfg::kXStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
    }
    if (kSums && pt1 > pt0) {
      // Thread `row` holds P (rows 0-63) or Q (rows 64-127) of channel c = row & 63.  Both halves go through shared
      // memory (the idle X ring, double-buffered so one barrier per 32 columns suffices); each thread then finishes
      // 16 of the 32 columns of its channel.
      mbar_wait(tfull_bar, 0);
      tc_fence_after();
      float* xch = reinterpret_cast<float*>(smem_raw + (smem_base - smem_u32(smem_raw)));
      const int c = row & 63, jh = (row >> 6) * 16;
      int b = 0;
      for (int g = g0; g < g1; ++g) {
        const int k = g * 64 + c;
        const float sc = p.bn_scale[k], sh = p.bn_shift[k];
        float s_p = 0.f, s_q = 0.f;
#pragma unroll 1
        for (int c0 = 0; c0 < BLOCK_N; c0 += 32, b ^= 1) {
          uint32_t v[32];
          tmem_ld_32x32(tmem_base + (uint32_t(quad * 32) << 16) + (g - g0) * BLOCK_N + c0, v);
          tmem_ld_wait();
          float* buf = xch + b * 4096;   // [P | Q][32 columns][64 channels]
#pragma unroll
          for (int j = 0; j < 32; ++j) buf[((row >> 6) * 32 + j) * 64 + c] = __uint_as_float(v[j]);
          asm volatile("bar.sync 1, 128;" ::: "memory");
          const uint4* wp = reinterpret_cast<const uint4*>(p.w_dgrad + (long long)k * p.Cout + n0 + c0 + jh);
          const uint4 w0 = __ldg(wp), w1 = __ldg(wp + 1);
          const uint32_t wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
          float* dst = p.dw + (long long)(n0 + c0 + jh) * p.Ktot + k;
#pragma unroll
          for (int jj = 0; jj < 16; ++jj) {
            const float pv = buf[(jh + jj) * 64 + c], qv = buf[(32 + jh + jj) * 64 + c];
            const float w = (jj & 1) ? bf16_hi(wv[jj >> 1]) : bf16_lo(wv[jj >> 1]);
            atomicAdd(dst + (long long)jj * p.Ktot, fmaf(sc, pv, sh * qv));
            s_p = fmaf(w, pv, s_p);
            s_q = fmaf(w, qv, s_q);
          }
        }
        atomicAdd(p.bn_sums + k, double(s_q));
        atomicAdd(p.bn_sums + p.Ktot + k, double(s_p));
      }
    } else if (pt1 > pt0) {
      mbar_wait(tfull_bar, 0);
      tc_fence_after();
      for (int g = g0; g < g1; ++g) {
        const int k = g * 128 + row;  // column of the OHWI weight row
        const bool kvalid = k < p.Ktot;
#pragma unroll 1
        for (int c0 = 0; c0 < BLOCK_N; c0 += 32) {
          uint32_t v[32];
          tmem_ld_32x32(tmem_base + (uint32_t(quad * 32) << 16) + (g - g0) * BLOCK_N + c0, v);
          tmem_ld_wait();
          if (kvalid) {
            float* dst = p.dw + (long long)(n0 + c0) * p.Ktot + k;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (n0 + c0 + j < p.Cout) atomicAdd(dst + (long long)j * p.Ktot, __uint_as_float(v[j]));
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

static inline int floor_div(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }

template <int BLOCK_N>
static int launch_wgrad(WgradParams& p, cudaStream_t stream) {
  using Cfg = WgradCfg<BLOCK_N>;
  static bool configured = false;
  if (!configured) {
    T2R_CUDA_OK(cudaFuncSetAttribute(conv_wgrad_kernel<BLOCK_N, kWgPlain>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    T2R_CUDA_OK(cudaFuncSetAttribute(conv_wgrad_kernel<BLOCK_N, kWgBnRelu>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    T2R_CUDA_OK(cudaFuncSetAttribute(conv_wgrad_kernel<BLOCK_N, kWgBnSums>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    configured = true;
  }
  p.groups_per_cta = std::min(p.n_groups, Cfg::kMaxGroups);
  p.n_gsets = int(ceil_div(p.n_groups, p.groups_per_cta));
  p.n_chunks_n = int(ceil_div(p.Cout, BLOCK_N));
  const int base_items = p.n_gsets * p.n_chunks_n;
  // Split the pixel range so that the grid fills the SMs `waves` times WITHOUT spilling into a partial
  // extra wave (one CTA per SM: a 297-CTA grid costs three rounds, not two).
  static const int waves = std::getenv("T2R_WGRAD_WAVES") ? atoi(std::getenv("T2R_WGRAD_WAVES")) : 1;
  int ks = std::max(1, waves * num_sms() / base_items);
  ks = std::max(1, std::min(ks, std::max(1, p.total_ptiles / 4)));
  p.ksplits = ks;
  const int grid = base_items * ks;
  if (p.bn_sums != nullptr)
    conv_wgrad_kernel<BLOCK_N, kWgBnSums><<<grid, 256, Cfg::kSmemBytes, stream>>>(p);
  else if (p.bn_scale != nullptr)
    conv_wgrad_kernel<BLOCK_N, kWgBnRelu><<<grid, 256, Cfg::kSmemBytes, stream>>>(p);
  else
    conv_wgrad_kernel<BLOCK_N, kWgPlain><<<grid, 256, Cfg::kSmemBytes, stream>>>(p);
  T2R_LAUNCH_OK();
  return T2R_OK;
}

}  // namespace t2r

using namespace t2r;

static int32_t wgrad_impl(const T2RConvDesc* d, const void* x, const float* bn_scale, const float* bn_shift,
                          const void* dy, float* dw, const void* w_dgrad, double* bn_sums, void* stream);

extern "C" int32_t t2r_conv2d_wgrad(const T2RConvDesc* d, const void* x, const void* dy,
                                    float* dw, void* stream) {
  return wgrad_impl(d, x, nullptr, nullptr, dy, dw, nullptr, nullptr, stream);
}

extern "C" int32_t t2r_conv2d_wgrad_bnrelu(const T2RConvDesc* d, const void* x_raw, const float* bn_scale,
                                           const float* bn_shift, const void* dy, float* dw, void* stream) {
  T2R_CHECK_ARG(d != nullptr && d->struct_size == sizeof(T2RConvDesc), "bad T2RConvDesc size");
  T2R_CHECK_ARG(bn_scale && bn_shift, "conv2d_wgrad_bnrelu: null scale / shift");
  T2R_CHECK_ARG(d->KH == 1 && d->KW == 1 && d->pad_top == 0 && d->pad_left == 0,
                "conv2d_wgrad_bnrelu: only 1x1 convolutions without padding fuse the batch-norm apply");
  return wgrad_impl(d, x_raw, bn_scale, bn_shift, dy, dw, nullptr, nullptr, stream);
}

extern "C" int32_t t2r_conv2d_wgrad_bnsums(const T2RConvDesc* d, const void* x_raw, const float* bn_scale,
                                           const float* bn_shift, const void* dy, const void* w_dgrad, float* dw,
                                           double* bn_sums, void* stream) {
  T2R_CHECK_ARG(d != nullptr && d->struct_size == sizeof(T2RConvDesc), "bad T2RConvDesc size");
  T2R_CHECK_ARG(bn_scale && bn_shift && w_dgrad && bn_sums, "conv2d_wgrad_bnsums: null pointer");
  T2R_CHECK_ARG(d->KH == 1 && d->KW == 1 && d->stride == 1 && d->pad_top == 0 && d->pad_left == 0,
                "conv2d_wgrad_bnsums: 1x1 stride-1 convolutions without padding only");
  return wgrad_impl(d, x_raw, bn_scale, bn_shift, dy, dw, w_dgrad, bn_sums, stream);
}

static int32_t wgrad_impl(const T2RConvDesc* d, const void* x, const float* bn_scale, const float* bn_shift,
                          const void* dy, float* dw, const void* w_dgrad, double* bn_sums, void* stream) {
  T2R_CHECK_ARG(d != nullptr && d->struct_size == sizeof(T2RConvDesc), "bad T2RConvDesc size");
  T2R_CHECK_ARG(d->stride == 1 || d->stride == 2, "stride must be 1 or 2");
  T2R_CHECK_ARG(d->KH * d->KW <= kMaxTaps, "filter too large");
  T2R_CHECK_ARG(d->Cin % 64 == 0 && d->Cout % 64 == 0, "Cin/Cout must be multiples of 64");
  T2R_CHECK_ARG(x && dy && dw, "null pointer");
  WgradParams p;
  memset(&p, 0, sizeof(p));
  pick_tile(d->Ho, d->Wo, 64, &p.TW, &p.TH);
  if (make_phase_maps(p.tmap_x, x, d->N, d->H, d->W, d->Cin, d->stride, p.TW, p.TH) != 0)
    return T2R_ERR_CUDA;
  CUtensorMap dy_maps[4];
  if (make_phase_maps(dy_maps, dy, d->N, d->Ho, d->Wo, d->Cout, 1, p.TW, p.TH) != 0)
    return T2R_ERR_CUDA;
  p.tmap_dy = dy_maps[0];
  p.chunks_per_tap = d->Cin / 64;
  int t = 0;
  for (int kh = 0; kh < d->KH; ++kh)
    for (int kw = 0; kw < d->KW; ++kw, ++t) {
      const int ih = kh - d->pad_top, iw = kw - d->pad_left;
      const int ph = ((ih % d->stride) + d->stride) % d->stride;
      const int pw = ((iw % d->stride) + d->stride) % d->stride;
      p.taps[t].map = int8_t(ph * d->stride + pw);
      p.taps[t].dh = int8_t(floor_div(ih, d->stride));
      p.taps[t].dw = int8_t(floor_div(iw, d->stride));
      p.taps[t].kchunk0 = t * p.chunks_per_tap;
    }
  if (bn_sums == nullptr && conv_wgrad_halo_eligible(d->stride, t, d->Cin, d->Cout))
    return conv_wgrad_halo_launch(x, dy, dw, d->N, d->H, d->W, d->Ho, d->Wo, d->Cout, p.taps, t,
                                  static_cast<cudaStream_t>(stream));
  p.n_slots = t * p.chunks_per_tap;
  p.n_groups = bn_sums != nullptr ? p.n_slots : (p.n_slots + 1) / 2;
  p.tiles_w = int(ceil_div(d->Wo, p.TW));
  p.tiles_h = int(ceil_div(d->Ho, p.TH));
  p.total_ptiles = d->N * p.tiles_w * p.tiles_h;
  p.Ktot = t * d->Cin;
  p.Cout = d->Cout;
  p.dw = dw;
  p.bn_scale = bn_scale;
  p.bn_shift = bn_shift;
  p.w_dgrad = static_cast<const uint16_t*>(w_dgrad);
  p.bn_sums = bn_sums;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (d->Cout % 256 == 0) return launch_wgrad<256>(p, st);
  if (d->Cout % 128 == 0) return launch_wgrad<128>(p, st);
  return launch_wgrad<64>(p, st);
}

// Weight gradient of the stem convolution over the padded NHWC4 image (see t2r_stem_conv_fprop):
// dw_stem fp32 [Cout][KH][64] += dy^T * windows; entries of padded slots (kw >= KW or c == 3) are
// garbage by construction and must be cleared with t2r_stem_mask_grad.
extern "C" int32_t t2r_stem_conv_wgrad(const T2RConvDesc* d, const void* x4p, int32_t Hp, int32_t Wp,
                                       const void* dy, float* dw_stem, void* stream) {
  T2R_CHECK_ARG(d && d->struct_size == sizeof(T2RConvDesc) && x4p && dy && dw_stem, "stem_conv_wgrad: bad args");
  T2R_CHECK_ARG(d->Cin == 3 && d->KW <= 16 && d->KH <= kMaxTaps && d->Cout % 64 == 0 && d->stride >= 1 &&
                    d->stride <= 2, "stem_conv_wgrad: unsupported geometry");
  WgradParams p;
  memset(&p, 0, sizeof(p));
  pick_tile(d->Ho, d->Wo, 64, &p.TW, &p.TH);
  if (make_stem_maps(p.tmap_x, x4p, d->N, Hp, Wp, d->KW, d->stride, d->Ho, d->Wo, p.TW, p.TH) < 0) return T2R_ERR_CUDA;
  CUtensorMap dy_maps[4];
  if (make_phase_maps(dy_maps, dy, d->N, d->Ho, d->Wo, d->Cout, 1, p.TW, p.TH) != 0) return T2R_ERR_CUDA;
  p.tmap_dy = dy_maps[0];
  p.chunks_per_tap = 1;
  p.n_slots = make_stem_taps(p.taps, d->KH, d->KW, d->stride);
  p.n_groups = (p.n_slots + 1) / 2;
  p.tiles_w = int(ceil_div(d->Wo, p.TW));
  p.tiles_h = int(ceil_div(d->Ho, p.TH));
  p.total_ptiles = d->N * p.tiles_w * p.tiles_h;
  p.Ktot = p.n_slots * 64;
  p.Cout = d->Cout;
  p.dw = dw_stem;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (d->Cout % 256 == 0) return launch_wgrad<256>(p, st);
  if (d->Cout % 128 == 0) return launch_wgrad<128>(p, st);
  return launch_wgrad<64>(p, st);
}
