// conv_igemm.cu — implicit-GEMM convolution forward / data-gradient on tcgen05 (sm_100a).
//
// One persistent, warp-specialised kernel serves conv fprop, conv dgrad and plain GEMM
// (a 1x1 "conv" over a [1,1,M,K] image).  The convolution is expressed as a *tap table*:
// for every filter tap the producer issues one 4-D TMA tile load of the activation tensor
// at a shifted coordinate (out-of-bounds rows/columns are zero-filled by TMA, which is the
// zero padding), plus one 2-D TMA load of the matching weight slice.  Strided convolutions
// read through per-phase tensor maps (even/odd rows x even/odd columns of the same buffer,
// expressed with doubled strides), so stride 2 costs nothing extra.
//
//   A (activations): 128 output pixels (a TW x TH rectangle of one image) x 64 channels,
//                    K-major, 128B-swizzled  -> 16 KB per stage
//   B (weights)    : BLOCK_N output channels x 64, K-major, 128B-swizzled
//   D (accumulator): 128 lanes x BLOCK_N fp32 columns in TMEM, double buffered
//
// Warp roles (384 threads): warps 0, 2, 3 = TMA producers, warp 1 = MMA issuer, warp 2 also = TMEM
// allocator, warps 4..11 = epilogue (TMEM -> registers -> bias/residual/ReLU -> global), two
// warpgroups splitting the BLOCK_N accumulator columns.
//
// Replaces: slim.conv2d / tf.layers.conv2d (research/qtopt/networks.py:443-591,
// layers/film_resnet_model.py:89-105) and their autodiff data gradients.
#include <algorithm>
#include <cstdlib>
#include <vector>

#include "conv_common.cuh"

namespace t2r {


template <int BLOCK_N>
struct IgemmCfg {
  static constexpr int kABytes = 128 * 128;
  static constexpr int kBBytes = BLOCK_N * 128;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = BLOCK_N == 64 ? 8 : (BLOCK_N == 128 ? 6 : 4);
  static constexpr int kTmemCols = 2 * BLOCK_N;  // 128 / 256 / 512: all powers of two
  static constexpr int kStoreStageBytes = 8 * 2048;   // one 32 rows x 64 B tile per epilogue warp
  static constexpr int kStatBytes = 2 * kMaxStatChannels * 4;  // per-CTA fp32 partials of the fused bn_stats
  static constexpr int kSmemBytes =
      kStages * kStageBytes + 1024 /*align*/ + 256 /*barriers*/ + kStoreStageBytes + kStatBytes;
};

// kPro: four extra warps (12..15) apply relu(bn_scale * x + bn_shift) to every landed A tile in place
// (kProBnRelu, conv_common.cuh); the MMA warp then waits on the `ready` barriers instead of `full`.
template <int BLOCK_N, bool kPro>
__global__ void __launch_bounds__(kPro ? 512 : 384, 1) conv_igemm_kernel(const __grid_constant__ IgemmParams p) {
  using Cfg = IgemmCfg<BLOCK_N>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + Cfg::kStages * Cfg::kStageBytes;
  // barrier layout: full[kStages], empty[kStages], tmem_full[2], tmem_empty[2], tmem_ptr
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (Cfg::kStages + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::kStages + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::kStages + 2 + s); };
  const uint32_t tmem_ptr_addr = bar_base + 8u * (2 * Cfg::kStages + 4);
  auto ready_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::kStages + 5 + s); };
  const uint32_t store_stage_base = bar_base + 256u;
  float* stat_acc = reinterpret_cast<float*>(smem_raw + (store_stage_base + Cfg::kStoreStageBytes - smem_u32(smem_raw)));
  volatile uint32_t* tmem_ptr_gen =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_ptr_addr - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < 4; ++i) tma_prefetch_desc(&p.tmap_a[i]);
    tma_prefetch_desc(&p.tmap_b);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < Cfg::kStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
      if (kPro) mbar_init(ready_bar(s), 4);  // one arrival per transformer warp
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), 8);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_ptr_addr, Cfg::kTmemCols);
    tmem_relinquish();
  }
  if (p.stats != nullptr)
    for (int i = threadIdx.x; i < 2 * p.Cout; i += blockDim.x) stat_acc[i] = 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_gen;

  const int k_iters = p.n_taps * p.chunks_per_tap;
  const int tiles_per_img = p.tiles_w * p.tiles_h;

  if (warp == 0 || warp == 2 || warp == 3) {
    // ===================== TMA producers =====================
    // A tile load costs its full latency (~280 cycles from L2, ~640 from DRAM) per *issuing warp*, no
    // matter how many are queued (profiles/r01_ncu_summary.md, section 3.3): one producer thread caps
    // the fill rate at box_bytes / latency.  Three warps on three different SM sub-partitions take
    // the k-iterations round-robin; every ring slot still has exactly one producer per use.
    if (lane == 0) {
      const int pid = warp == 0 ? 0 : warp - 1;
      int stage = 0, turn = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        const int nt = tile % p.n_tiles_n;
        const int mt = tile / p.n_tiles_n;
        const int img = mt / tiles_per_img;
        const int rem = mt - img * tiles_per_img;
        const int oh0 = (rem / p.tiles_w) * p.TH;
        const int ow0 = (rem % p.tiles_w) * p.TW;
        for (int t = 0; t < p.n_taps; ++t) {
          const ConvTap tap = p.taps[t];
          for (int c = 0; c < p.chunks_per_tap; ++c) {
            if (turn == pid) {
              mbar_wait(empty_bar(stage), phase ^ 1u);
              const uint32_t sa = smem_base + stage * Cfg::kStageBytes;
              const uint32_t sb = sa + Cfg::kABytes;
              mbar_expect_tx(full_bar(stage), Cfg::kStageBytes);
              tma_load_4d(sa, &p.tmap_a[tap.map], full_bar(stage), c * 64, ow0 + tap.dw, oh0 + tap.dh, img);
              tma_load_2d(sb, &p.tmap_b, full_bar(stage), (tap.kchunk0 + c) * 64, nt * BLOCK_N);
            }
            if (++turn == 3) turn = 0;
            if (++stage == Cfg::kStages) {
              stage = 0;
              phase ^= 1u;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // The whole warp runs the loop converged and an elected lane issues (umma_bf16_elect): descriptors
    // are a precomputed base plus a 16-byte-unit offset, all warp-uniform (tests/native/exp_mma_issue.cu).
    {
      constexpr uint32_t idesc = make_idesc_bf16(128, BLOCK_N, 0, 0);
      const uint64_t a_base = make_smem_desc_sw128(smem_base, 16, 1024);
      const uint64_t b_base = make_smem_desc_sw128(smem_base + Cfg::kABytes, 16, 1024);
      int stage = 0, as = 0;
      uint32_t phase = 0, aphase = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        mbar_wait(tempty_bar(as), aphase ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BLOCK_N;
        for (int k = 0; k < k_iters; ++k) {
          mbar_wait(kPro ? ready_bar(stage) : full_bar(stage), phase);
          tc_fence_after();
          const uint64_t so = uint64_t(uint32_t(stage) * uint32_t(Cfg::kStageBytes >> 4));
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            umma_bf16_elect(d_tmem, a_base + so + uint64_t(kk * 2), b_base + so + uint64_t(kk * 2), idesc,
                            (k > 0 || kk > 0) ? 1u : 0u);
          umma_commit_elect(empty_bar(stage));
          if (++stage == Cfg::kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
        umma_commit_elect(tfull_bar(as));
        if (++as == 2) {
          as = 0;
          aphase ^= 1u;
        }
      }
    }
  } else if (kPro && warp >= 12) {
    // ===================== operand transform: 4 warps =====================
    // Thread t owns the logical 16-byte chunk (t & 7) = 8 channels of rows (t >> 3) + 16 i of the 128-row A tile:
    // a quarter warp covers one full 128-byte row (no bank conflicts) and all of a thread's rows share r & 7.
    const int t = threadIdx.x - 384;
    const uint32_t j = uint32_t(t) & 7u, r0 = uint32_t(t) >> 3;
    const uint32_t piece0 = r0 * 128u + ((j ^ (r0 & 7u)) << 4);
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      for (int tp = 0; tp < p.n_taps; ++tp)
        for (int c = 0; c < p.chunks_per_tap; ++c) {
          float sc[8], sh[8];
          load8(p.bn_scale + c * 64 + j * 8, sc);
          load8(p.bn_shift + c * 64 + j * 8, sh);
          mbar_wait(full_bar(stage), phase);
          bnrelu_pieces_inplace<8>(smem_base + stage * Cfg::kStageBytes + piece0, 2048u, sc, sh);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(ready_bar(stage));
          if (++stage == Cfg::kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
    }
  } else if (warp >= 4) {
    // ===================== epilogue: 8 warps =====================
    // Warp w may read TMEM lanes 32*(w%4)..+31 (one output pixel per thread); the two warpgroups
    // split the BLOCK_N columns.  The residual (bf16, same addressing as the output) of the next
    // 32-column chunk is prefetched into registers before the accumulator wait / while the current
    // chunk is converted, so its DRAM latency is off the critical path.
    const int ew = warp - 4;
    const int quad = ew & 3;
    const int half = ew >> 2;
    constexpr int kColsPerWG = BLOCK_N / 2;
    constexpr int kChunks = kColsPerWG / 32;
    const int row = quad * 32 + lane;
    const int th = row / p.TW;
    const int tw = row - th * p.TW;
    const bool out_f32 = (p.flags & T2R_EPI_OUT_F32) != 0;
    const bool has_res = (p.flags & T2R_EPI_RESIDUAL) != 0;
    const bool bnbwd = (p.flags & kEpiBnBwd) != 0;   // never together with a residual
    const bool has_aux = has_res || bnbwd;
    const __nv_bfloat16* aux = static_cast<const __nv_bfloat16*>(bnbwd ? p.bn_x : p.residual);
    int as = 0;
    uint32_t aphase = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const int nt = tile % p.n_tiles_n;
      const int mt = tile / p.n_tiles_n;
      const int img = mt / tiles_per_img;
      const int rem = mt - img * tiles_per_img;
      const int oh = (rem / p.tiles_w) * p.TH + th;
      const int ow = (rem % p.tiles_w) * p.TW + tw;
      const bool valid = (oh < p.Ho) && (ow < p.Wo);
      const long long pix_off = img * p.os_n + oh * p.os_h + ow * p.os_w;
      const int ch0 = nt * BLOCK_N + half * kColsPerWG;
      // rows this lane STORES: instruction i of a chunk writes rows 8i + lane/4 of the warp's 32
      // (4 lanes x 16 B = the row's 64 contiguous bytes), see the staging below.
      long long roff[4];
      bool rvalid[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = quad * 32 + 8 * i + (lane >> 2);
        const int rth = r / p.TW, rtw = r - rth * p.TW;
        const int roh = (rem / p.tiles_w) * p.TH + rth, row_w = (rem % p.tiles_w) * p.TW + rtw;
        rvalid[i] = (roh < p.Ho) && (row_w < p.Wo);
        roff[i] = img * p.os_n + roh * p.os_h + row_w * p.os_w;
      }
      uint4 rnext[4] = {};
      if (has_aux && valid && ch0 < p.Cout) {
        const uint4* r = reinterpret_cast<const uint4*>(aux + pix_off + ch0);
#pragma unroll
        for (int j = 0; j < 4; ++j) rnext[j] = r[j];
      }
      mbar_wait(tfull_bar(as), aphase);
      tc_fence_after();
#pragma unroll 1
      for (int c = 0; c < kChunks; ++c) {
        const int ch = ch0 + c * 32;
        uint4 rcur[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) rcur[j] = rnext[j];
        if (c + 1 < kChunks && has_aux && valid && ch + 32 < p.Cout) {
          const uint4* r = reinterpret_cast<const uint4*>(aux + pix_off + ch + 32);
#pragma unroll
          for (int j = 0; j < 4; ++j) rnext[j] = r[j];
        }
        uint32_t v[32];
        tmem_ld_32x32(tmem_base + (uint32_t(quad * 32) << 16) + as * BLOCK_N + half * kColsPerWG + c * 32, v);
        tmem_ld_wait();
        if (out_f32 ? (valid && ch < p.Cout) : (ch < p.Cout)) {
          float f[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
          if (p.flags & T2R_EPI_BIAS) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 b = *reinterpret_cast<const float4*>(p.bias + ch + j);
              f[j] += b.x; f[j + 1] += b.y; f[j + 2] += b.z; f[j + 3] += b.w;
            }
          }
          if (has_res && valid) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint4 q = rcur[j];
              f[8 * j + 0] += bf16_lo(q.x); f[8 * j + 1] += bf16_hi(q.x);
              f[8 * j + 2] += bf16_lo(q.y); f[8 * j + 3] += bf16_hi(q.y);
              f[8 * j + 4] += bf16_lo(q.z); f[8 * j + 5] += bf16_hi(q.z);
              f[8 * j + 6] += bf16_lo(q.w); f[8 * j + 7] += bf16_hi(q.w);
            }
          }
          if (p.flags & T2R_EPI_RELU) {
#pragma unroll
            for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
          }
          if (bnbwd) {
            // g = dz * [scale * x + shift > 0], rounded to bf16 like the stored value; column sums of g * x
            // (those of g itself come out of the staged tile below, as for the fused bn_stats)
            float xv[32];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint4 q = rcur[j];
              xv[8 * j + 0] = bf16_lo(q.x); xv[8 * j + 1] = bf16_hi(q.x);
              xv[8 * j + 2] = bf16_lo(q.y); xv[8 * j + 3] = bf16_hi(q.y);
              xv[8 * j + 4] = bf16_lo(q.z); xv[8 * j + 5] = bf16_hi(q.z);
              xv[8 * j + 6] = bf16_lo(q.w); xv[8 * j + 7] = bf16_hi(q.w);
            }
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 sc = __ldg(reinterpret_cast<const float4*>(p.bn_scale + ch + j));
              const float4 sh = __ldg(reinterpret_cast<const float4*>(p.bn_shift + ch + j));
              const float scv[4] = {sc.x, sc.y, sc.z, sc.w}, shv[4] = {sh.x, sh.y, sh.z, sh.w};
#pragma unroll
              for (int i = 0; i < 4; i += 2) {
                const float g0 = (valid && fmaf(xv[j + i], scv[i], shv[i]) > 0.f) ? f[j + i] : 0.f;
                const float g1 = (valid && fmaf(xv[j + i + 1], scv[i + 1], shv[i + 1]) > 0.f) ? f[j + i + 1] : 0.f;
                const uint32_t pk = pack_bf16(g0, g1);
                f[j + i] = bf16_lo(pk);
                f[j + i + 1] = bf16_hi(pk);
                xv[j + i] *= f[j + i];
                xv[j + i + 1] *= f[j + i + 1];
              }
            }
            const float sgx = warp_transpose_sum32(xv, lane);
            atomicAdd(stat_acc + p.Cout + ch + lane, sgx);
          }
          if (out_f32) {
            float4* o = reinterpret_cast<float4*>(static_cast<float*>(p.out) + pix_off + ch);
#pragma unroll
            for (int j = 0; j < 8; ++j)
              o[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
          } else {
            // bf16 output.  A thread owns one pixel row, so direct stores would hit 32 different
            // 32-byte sectors per instruction (16 B each, row pitch = Cout*2 B).  Stage the warp's
            // 32 rows x 64 B through a swizzled shared tile instead: every store instruction then
            // writes 8 rows x 64 contiguous bytes (16 fully written sectors).
            const uint32_t wb = store_stage_base + uint32_t(ew) * 2048u;
            const uint32_t sw = (uint32_t(lane) >> 1) & 3u;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint32_t q0 = pack_bf16(f[8 * j + 0], f[8 * j + 1]), q1 = pack_bf16(f[8 * j + 2], f[8 * j + 3]);
              uint32_t q2 = pack_bf16(f[8 * j + 4], f[8 * j + 5]), q3 = pack_bf16(f[8 * j + 6], f[8 * j + 7]);
              if (!valid) q0 = q1 = q2 = q3 = 0u;  // rows outside the image are never stored and must not count
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(wb + uint32_t(lane) * 64u + ((uint32_t(j) ^ sw) << 4)),
                           "r"(q0), "r"(q1), "r"(q2), "r"(q3)
                           : "memory");
            }
            __syncwarp();
            if (p.stats != nullptr) {
              // fused bn_stats: lane l sums column l of the staged 32 x 32 tile (the bf16 values the
              // next layer's batch norm will read), then one shared-memory atomic per statistic.
              float s1 = 0.f, s2 = 0.f;
              const uint32_t cj = uint32_t(lane) >> 3, cb = (uint32_t(lane) & 7u) * 2u;
#pragma unroll
              for (uint32_t r = 0; r < 32; ++r) {
                uint16_t h;
                asm volatile("ld.shared.u16 %0, [%1];" : "=h"(h) : "r"(wb + r * 64u + ((cj ^ ((r >> 1) & 3u)) << 4) + cb) : "memory");
                const float v = __uint_as_float(uint32_t(h) << 16);
                s1 += v;
                s2 = fmaf(v, v, s2);
              }
              atomicAdd(stat_acc + ch + lane, s1);
              if (!bnbwd) atomicAdd(stat_acc + p.Cout + ch + lane, s2);
            }
            const uint32_t jj = uint32_t(lane) & 3u;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const uint32_t r = 8u * i + (uint32_t(lane) >> 2);
              uint4 q;
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                           : "=r"(q.x), "=r"(q.y), "=r"(q.z), "=r"(q.w)
                           : "r"(wb + r * 64u + ((jj ^ ((r >> 1) & 3u)) << 4))
                           : "memory");
              if (rvalid[i])
                *reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(p.out) + roff[i] + ch + jj * 8) = q;
            }
            __syncwarp();
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(as));
      if (++as == 2) {
        as = 0;
        aphase ^= 1u;
      }
    }
    if (p.stats != nullptr) {
      asm volatile("bar.sync 1, 256;" ::: "memory");  // the 8 epilogue warps
      for (int i = threadIdx.x - 128; i < 2 * p.Cout; i += 256) {
        const float v = stat_acc[i];
        if (v != 0.f) atomicAdd(p.stats + i, double(v));
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// Zero a strided [N,Hv,Wv,C] view (C in uint4 = 8 bf16 units).
__global__ void zero_view_kernel(uint4* out, int N, int Hv, int Wv, int C8, long long os_n,
                                 long long os_h, long long os_w) {
  const long long total = (long long)N * Hv * Wv * C8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c = int(i % C8);
    long long r = i / C8;
    const int w = int(r % Wv); r /= Wv;
    const int h = int(r % Hv);
    const int n = int(r / Hv);
    out[n * os_n + h * os_h + w * os_w + c] = make_uint4(0, 0, 0, 0);
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------

// Pick the TW x TH = `pixels` rectangle that wastes the fewest padded pixels.
void pick_tile(int Ho, int Wo, int pixels, int* TW, int* TH) {
  long long best = -1;
  for (int tw = pixels; tw >= 1; tw >>= 1) {
    const int th = pixels / tw;
    if (tw > 256 || th > 256) continue;
    const long long cover = ceil_div(Wo, tw) * tw * ceil_div(Ho, th) * th;
    // prefer wider tiles on ties (longer contiguous runs per TMA row)
    if (best < 0 || cover < best) {
      best = cover;
      *TW = tw;
      *TH = th;
    }
  }
}

// Activation tensor maps for reading input coordinate (s*o + k - pad): phase (ph, pw) of a
// [N,H,W,C] bf16 tensor is the sub-image of rows ph, ph+s, ... and columns pw, pw+s, ...
int make_phase_maps(CUtensorMap* maps, const void* x, int N, int H, int W, int C, int stride,
                    int TW, int TH) {
  const char* base = static_cast<const char*>(x);
  for (int ph = 0; ph < stride; ++ph)
    for (int pw = 0; pw < stride; ++pw) {
      const int Hd = (H - ph + stride - 1) / stride;
      const int Wd = (W - pw + stride - 1) / stride;
      uint64_t dims[4] = {uint64_t(C), uint64_t(std::max(Wd, 1)), uint64_t(std::max(Hd, 1)),
                          uint64_t(N)};
      uint64_t strides[3] = {uint64_t(stride) * C * 2, uint64_t(stride) * W * C * 2,
                             uint64_t(H) * W * C * 2};
      uint32_t box[4] = {64, uint32_t(TW), uint32_t(TH), 1};
      const void* addr = base + (size_t(ph) * W + pw) * C * 2;
      if (Hd <= 0 || Wd <= 0) addr = base;  // degenerate phase: never referenced by a tap
      if (encode_tmap_bf16(&maps[ph * stride + pw], addr, 4, dims, strides, box) != 0) return -1;
    }
  // fill unused slots with a valid descriptor so prefetch is harmless
  for (int i = stride * stride; i < 4; ++i) maps[i] = maps[0];
  return 0;
}

static inline int floor_div(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }

template <int BLOCK_N, bool kPro>
static int launch_igemm_v(const IgemmParams& p, cudaStream_t stream) {
  using Cfg = IgemmCfg<BLOCK_N>;
  static bool configured = false;
  if (!configured) {
    T2R_CUDA_OK(cudaFuncSetAttribute(conv_igemm_kernel<BLOCK_N, kPro>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     Cfg::kSmemBytes));
    configured = true;
  }
  const int grid = std::min(p.total_tiles, num_sms());
  conv_igemm_kernel<BLOCK_N, kPro><<<grid, kPro ? 512 : 384, Cfg::kSmemBytes, stream>>>(p);
  T2R_LAUNCH_OK();
  return T2R_OK;
}
template <int BLOCK_N>
static int launch_igemm(const IgemmParams& p, cudaStream_t stream) {
  return (p.flags & kProBnRelu) ? launch_igemm_v<BLOCK_N, true>(p, stream) : launch_igemm_v<BLOCK_N, false>(p, stream);
}

// Tile width and epilogue flavour.  bf16 outputs with N <= 128 use the TMA epilogue
// (conv_igemm_tma.cu); 256-multiple channel counts do so too (as two 128-wide tiles) when the GEMM K
// is so small that the layer is bound by its output / residual traffic rather than by the MMA.
static int pick_block_n(int Cout, long long k_total, int flags, bool* tma) {
  static const bool no_tma = std::getenv("T2R_DISABLE_TMA_EPI") != nullptr;
  int bn = 64;
  if (Cout % 256 == 0) bn = 256;
  else if (Cout % 128 == 0) bn = 128;
  *tma = !no_tma && !(flags & T2R_EPI_OUT_F32);
  if (*tma && bn == 256) {
    if (k_total <= 256) bn = 128; else *tma = false;
  }
  return bn;
}

static int dispatch_igemm(IgemmParams& p, int block_n, bool tma, cudaStream_t stream) {
  if (tma) return conv_igemm_tma_launch(p, block_n, stream);
  p.n_tiles_n = int(ceil_div(p.Cout, block_n));
  p.total_tiles = p.N * p.tiles_w * p.tiles_h * p.n_tiles_n;
  if (p.total_tiles <= 0) return T2R_OK;
  switch (block_n) {
    case 64: return launch_igemm<64>(p, stream);
    case 128: return launch_igemm<128>(p, stream);
    default: return launch_igemm<256>(p, stream);
  }
}

static int check_desc(const T2RConvDesc* d) {
  T2R_CHECK_ARG(d != nullptr && d->struct_size == sizeof(T2RConvDesc), "bad T2RConvDesc size");
  T2R_CHECK_ARG(d->stride == 1 || d->stride == 2, "stride must be 1 or 2 (got %d)", d->stride);
  T2R_CHECK_ARG(d->KH * d->KW <= kMaxTaps && d->KH >= 1 && d->KW >= 1, "filter %dx%d unsupported",
                d->KH, d->KW);
  T2R_CHECK_ARG(d->N > 0 && d->H > 0 && d->W > 0 && d->Ho > 0 && d->Wo > 0, "empty tensor");
  T2R_CHECK_ARG(d->Cin % 64 == 0 && d->Cin > 0, "Cin=%d must be a multiple of 64", d->Cin);
  T2R_CHECK_ARG(d->Cout % 64 == 0 && d->Cout > 0, "Cout=%d must be a multiple of 64", d->Cout);
  return T2R_OK;
}

}  // namespace t2r

using namespace t2r;

extern "C" int32_t t2r_conv_same_padding(int32_t in, int32_t k, int32_t stride, int32_t* out,
                                         int32_t* pad_before) {
  T2R_CHECK_ARG(in > 0 && k > 0 && stride > 0, "bad same-padding args");
  const int o = (in + stride - 1) / stride;
  const int total = std::max((o - 1) * stride + k - in, 0);
  if (out) *out = o;
  if (pad_before) *pad_before = total / 2;
  return T2R_OK;
}

extern "C" int32_t t2r_conv2d_fprop(const T2RConvDesc* d, const void* x, const void* w,
                                    const float* bias, const void* residual, void* y,
                                    void* stream) {
  return t2r_conv2d_fprop_stats(d, x, w, bias, residual, y, nullptr, stream);
}

static int32_t fprop_impl(const T2RConvDesc* d, const void* x, const float* bn_scale, const float* bn_shift,
                          const void* w, const float* bias, const void* residual, void* y, double* stats,
                          void* stream);

extern "C" int32_t t2r_conv2d_fprop_stats(const T2RConvDesc* d, const void* x, const void* w,
                                          const float* bias, const void* residual, void* y,
                                          double* stats, void* stream) {
  return fprop_impl(d, x, nullptr, nullptr, w, bias, residual, y, stats, stream);
}

extern "C" int32_t t2r_conv2d_fprop_bnrelu(const T2RConvDesc* d, const void* x_raw, const float* bn_scale,
                                           const float* bn_shift, const void* w, const void* residual, void* y,
                                           double* stats, void* stream) {
  T2R_CHECK_ARG(d != nullptr && d->struct_size == sizeof(T2RConvDesc), "bad T2RConvDesc size");
  T2R_CHECK_ARG(bn_scale && bn_shift, "conv2d_fprop_bnrelu: null scale / shift");
  T2R_CHECK_ARG(d->KH == 1 && d->KW == 1 && d->pad_top == 0 && d->pad_left == 0,
                "conv2d_fprop_bnrelu: only 1x1 convolutions without padding fuse the batch-norm apply "
                "(zero padding would have to stay zero after the affine map)");
  T2R_CHECK_ARG(!(d->flags & (T2R_EPI_OUT_F32 | T2R_EPI_BIAS)), "conv2d_fprop_bnrelu: bf16 output without bias only");
  return fprop_impl(d, x_raw, bn_scale, bn_shift, w, nullptr, residual, y, stats, stream);
}

static int32_t fprop_impl(const T2RConvDesc* d, const void* x, const float* bn_scale, const float* bn_shift,
                          const void* w, const float* bias, const void* residual, void* y, double* stats,
                          void* stream) {
  if (int rc = check_desc(d)) return rc;
  T2R_CHECK_ARG(x && w && y, "null pointer");
  T2R_CHECK_ARG(stats == nullptr || (!(d->flags & T2R_EPI_OUT_F32) && d->Cout <= kMaxStatChannels),
                "fused bn_stats needs a bf16 output with at most %d channels", kMaxStatChannels);
  T2R_CHECK_ARG(!(d->flags & T2R_EPI_BIAS) || bias, "bias flag without bias");
  T2R_CHECK_ARG(!(d->flags & T2R_EPI_RESIDUAL) || residual, "residual flag without residual");
  IgemmParams p;
  memset(&p, 0, sizeof(p));
  pick_tile(d->Ho, d->Wo, 128, &p.TW, &p.TH);
  if (make_phase_maps(p.tmap_a, x, d->N, d->H, d->W, d->Cin, d->stride, p.TW, p.TH) != 0)
    return T2R_ERR_CUDA;
  const uint64_t Ktot = uint64_t(d->KH) * d->KW * d->Cin;
  bool tma = false;
  const int block_n = pick_block_n(d->Cout, (long long)Ktot, d->flags, &tma);
  {
    uint64_t dims[2] = {Ktot, uint64_t(d->Cout)};
    uint64_t strides[1] = {Ktot * 2};
    uint32_t box[2] = {64, uint32_t(block_n)};
    if (encode_tmap_bf16(&p.tmap_b, w, 2, dims, strides, box) != 0) return T2R_ERR_CUDA;
  }
  p.chunks_per_tap = d->Cin / 64;
  int t = 0;
  for (int kh = 0; kh < d->KH; ++kh)
    for (int kw = 0; kw < d->KW; ++kw, ++t) {
      const int ih = kh - d->pad_top, iw = kw - d->pad_left;  // input = s*o + ih
      const int ph = ((ih % d->stride) + d->stride) % d->stride;
      const int pw = ((iw % d->stride) + d->stride) % d->stride;
      p.taps[t].map = int8_t(ph * d->stride + pw);
      p.taps[t].dh = int8_t(floor_div(ih, d->stride));
      p.taps[t].dw = int8_t(floor_div(iw, d->stride));
      p.taps[t].kchunk0 = t * p.chunks_per_tap;
    }
  p.n_taps = t;
  if (conv_halo_eligible(d->stride, t, d->Cin, d->Cout)) {
    HaloRequest r;
    memset(&r, 0, sizeof(r));
    r.x = x; r.N = d->N; r.H = d->H; r.W = d->W; r.C = d->Cin;
    r.w = w; r.Ktot = Ktot;
    memcpy(r.taps, p.taps, sizeof(r.taps));
    r.n_taps = t;
    r.Ho = d->Ho; r.Wo = d->Wo; r.Cout = d->Cout;
    r.os_w = d->Cout; r.os_h = (long long)d->Wo * d->Cout; r.os_n = (long long)d->Ho * d->Wo * d->Cout;
    r.out = y; r.residual = residual; r.bias = bias; r.flags = d->flags; r.stats = stats;
    return conv_halo_launch(r, static_cast<cudaStream_t>(stream));
  }
  p.tiles_w = int(ceil_div(d->Wo, p.TW));
  p.tiles_h = int(ceil_div(d->Ho, p.TH));
  p.N = d->N; p.Ho = d->Ho; p.Wo = d->Wo; p.Cout = d->Cout;
  p.os_w = d->Cout;
  p.os_h = (long long)d->Wo * d->Cout;
  p.os_n = (long long)d->Ho * d->Wo * d->Cout;
  p.out = y; p.residual = residual; p.bias = bias; p.flags = d->flags; p.stats = stats;
  if (bn_scale != nullptr) {
    p.flags |= kProBnRelu;
    p.bn_scale = bn_scale;
    p.bn_shift = bn_shift;
  }
  return dispatch_igemm(p, block_n, tma, static_cast<cudaStream_t>(stream));
}

static int32_t dgrad_impl(const T2RConvDesc* d, const void* dy, const void* w_dgrad, void* dx, int32_t accumulate,
                          const void* bn_x, const float* bn_scale, const float* bn_shift, double* red,
                          const float* bn_coef, const void* dpass, void* stream);

extern "C" int32_t t2r_conv2d_dgrad(const T2RConvDesc* d, const void* dy, const void* w_dgrad,
                                    void* dx, int32_t accumulate, void* stream) {
  return dgrad_impl(d, dy, w_dgrad, dx, accumulate, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, stream);
}

extern "C" int32_t t2r_conv2d_dgrad_bnrelu(const T2RConvDesc* d, const void* dy, const void* w_dgrad,
                                           const void* x_raw, const float* bn_scale, const float* bn_shift, void* g,
                                           int32_t accumulate, double* red, void* stream) {
  T2R_CHECK_ARG(x_raw && bn_scale && bn_shift && red, "conv2d_dgrad_bnrelu: null pointer");
  return dgrad_impl(d, dy, w_dgrad, g, accumulate, x_raw, bn_scale, bn_shift, red, nullptr, nullptr, stream);
}

extern "C" int32_t t2r_conv2d_dgrad_bnapply_supported(const T2RConvDesc* d) {
  if (d == nullptr || d->struct_size != sizeof(T2RConvDesc)) return 0;
  if (d->KH != 1 || d->KW != 1 || d->stride != 1 || d->pad_top != 0 || d->pad_left != 0) return 0;
  if (d->Cin % 64 != 0 || d->Cout % 64 != 0 || d->Cin <= 0 || d->Cout <= 0) return 0;
  bool tma = false;
  pick_block_n(d->Cin, d->Cout, 0, &tma);
  return tma ? 1 : 0;
}

extern "C" int32_t t2r_conv2d_dgrad_bnapply(const T2RConvDesc* d, const void* dy, const void* w_dgrad,
                                            const void* x_raw, const float* bn_scale, const float* bn_shift,
                                            const float* bn_coef, const void* dpass, void* dx, void* stream) {
  if (int rc = check_desc(d)) return rc;
  T2R_CHECK_ARG(x_raw && bn_scale && bn_shift && bn_coef, "conv2d_dgrad_bnapply: null pointer");
  T2R_CHECK_ARG(t2r_conv2d_dgrad_bnapply_supported(d),
                "conv2d_dgrad_bnapply: needs a 1x1 stride-1 unpadded convolution whose data gradient runs on the "
                "TMA-epilogue kernel (Cin <= 128, or a multiple of 256 with Cout <= 256)");
  return dgrad_impl(d, dy, w_dgrad, dx, 0, x_raw, bn_scale, bn_shift, nullptr, bn_coef, dpass, stream);
}

static int32_t dgrad_impl(const T2RConvDesc* d, const void* dy, const void* w_dgrad, void* dx, int32_t accumulate,
                          const void* bn_x, const float* bn_scale, const float* bn_shift, double* red,
                          const float* bn_coef, const void* dpass, void* stream) {
  if (int rc = check_desc(d)) return rc;
  T2R_CHECK_ARG(dy && w_dgrad && dx, "null pointer");
  // Batch-norm backward fusion: the epilogues mask and reduce while they write (kEpiBnBwd) unless the launch
  // accumulates into dx (the mask would have to cover the sum) or runs on the halo kernel; those cases run the
  // plain data gradient followed by the stand-alone reduction pass over (dx, x).
  // Measured on B200 (profiles/r02_bn_fusion.md): the fused epilogue costs ~24 instructions per element where a
  // memory-bound kernel can afford ~6, e.g. 3.3 ms against 1.1 ms (data gradient) + 1.2 ms (reduction pass) on
  // 512x118x118x256, so the reduction pass below stays the default and the epilogue is opt-in (T2R_BNBWD_EPI=1).
  static const bool epi_bnbwd = std::getenv("T2R_BNBWD_EPI") != nullptr && std::getenv("T2R_BNBWD_EPI")[0] == '1';
  const bool want_bn = bn_x != nullptr && bn_coef == nullptr;
  bool fuse_bn = want_bn && epi_bnbwd && !accumulate && d->Cin <= kMaxStatChannels;
  const int s = d->stride;
  const int taps_total = d->KH * d->KW;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // dx[n,h,w,ci] = sum_{kh,kw,co} dy[n,(h+pt-kh)/s,(w+pl-kw)/s,co] * w[co,kh,kw,ci]
  // One launch per output phase (h%s, w%s): inside a phase the contributing taps are fixed and
  // the access is a stride-1 convolution over dy.
  for (int ph = 0; ph < s; ++ph)
    for (int pw = 0; pw < s; ++pw) {
      const int Hv = (d->H - ph + s - 1) / s, Wv = (d->W - pw + s - 1) / s;
      if (Hv <= 0 || Wv <= 0) continue;
      IgemmParams p;
      memset(&p, 0, sizeof(p));
      int t = 0;
      for (int kh = 0; kh < d->KH; ++kh) {
        if (((ph + d->pad_top - kh) % s + s) % s != 0) continue;
        for (int kw = 0; kw < d->KW; ++kw) {
          if (((pw + d->pad_left - kw) % s + s) % s != 0) continue;
          p.taps[t].map = 0;
          p.taps[t].dh = int8_t(floor_div(ph + d->pad_top - kh, s));
          p.taps[t].dw = int8_t(floor_div(pw + d->pad_left - kw, s));
          p.taps[t].kchunk0 = (kh * d->KW + kw) * (d->Cout / 64);
          ++t;
        }
      }
      p.n_taps = t;
      bool tma = false;
      const int block_n = pick_block_n(d->Cin, (long long)t * d->Cout, 0, &tma);
      const size_t view_off = (size_t(ph) * d->W + pw) * d->Cin * 2;
      char* out = static_cast<char*>(dx) + view_off;
      if (conv_halo_eligible(s, t, d->Cout, d->Cin)) {
        fuse_bn = false;
        HaloRequest r;
        memset(&r, 0, sizeof(r));
        r.x = dy; r.N = d->N; r.H = d->Ho; r.W = d->Wo; r.C = d->Cout;
        r.w = w_dgrad; r.Ktot = uint64_t(taps_total) * d->Cout;
        memcpy(r.taps, p.taps, sizeof(r.taps));
        r.n_taps = t;
        r.Ho = Hv; r.Wo = Wv; r.Cout = d->Cin;
        r.os_w = d->Cin; r.os_h = (long long)d->W * d->Cin; r.os_n = (long long)d->H * d->W * d->Cin;
        r.out = out; r.residual = accumulate ? out : nullptr; r.flags = accumulate ? T2R_EPI_RESIDUAL : 0;
        if (int rc = conv_halo_launch(r, st)) return rc;
        continue;
      }
      pick_tile(Hv, Wv, 128, &p.TW, &p.TH);
      if (make_phase_maps(p.tmap_a, dy, d->N, d->Ho, d->Wo, d->Cout, 1, p.TW, p.TH) != 0)
        return T2R_ERR_CUDA;
      const uint64_t Ktot = uint64_t(taps_total) * d->Cout;
      uint64_t dims[2] = {Ktot, uint64_t(d->Cin)};
      uint64_t strides[1] = {Ktot * 2};
      uint32_t box[2] = {64, uint32_t(block_n)};
      if (encode_tmap_bf16(&p.tmap_b, w_dgrad, 2, dims, strides, box) != 0) return T2R_ERR_CUDA;
      p.chunks_per_tap = d->Cout / 64;
      p.tiles_w = int(ceil_div(Wv, p.TW));
      p.tiles_h = int(ceil_div(Hv, p.TH));
      p.N = d->N; p.Ho = Hv; p.Wo = Wv; p.Cout = d->Cin;
      p.os_w = (long long)s * d->Cin;
      p.os_h = (long long)s * d->W * d->Cin;
      p.os_n = (long long)d->H * d->W * d->Cin;
      p.out = out;
      p.residual = accumulate ? out : nullptr;
      p.flags = accumulate ? T2R_EPI_RESIDUAL : 0;
      if (bn_coef != nullptr) {   // t2r_conv2d_dgrad_bnapply: one phase, one tap, TMA epilogue (checked there)
        p.flags = kEpiBnApply;
        p.bn_x = bn_x;
        p.bn_scale = bn_scale;
        p.bn_shift = bn_shift;
        p.bn_coef = bn_coef;
        p.residual = dpass;
      }
      if (fuse_bn) {
        p.flags |= kEpiBnBwd;
        p.bn_x = static_cast<const char*>(bn_x) + view_off;
        p.bn_scale = bn_scale;
        p.bn_shift = bn_shift;
        p.stats = red;
      }
      if (t == 0) {
        // No tap reaches this phase (e.g. 1x1 stride-2): the gradient there is zero.
        if (!accumulate) {
          const long long total = (long long)d->N * Hv * Wv * (d->Cin / 8);
          const int blocks = int(std::min<long long>(ceil_div(total, 256), 148 * 16));
          zero_view_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<uint4*>(out), d->N, Hv, Wv,
                                                   d->Cin / 8, p.os_n / 8, p.os_h / 8, p.os_w / 8);
          T2R_LAUNCH_OK();
        }
        continue;
      }
      if (int rc = dispatch_igemm(p, block_n, tma, st)) return rc;
    }
  if (want_bn && !fuse_bn)
    return bn_bwd_reduce_launch(dx, bn_x, (long long)d->N * d->H * d->W, d->Cin, nullptr, nullptr, bn_scale, bn_shift,
                                1, red, st);
  return T2R_OK;
}

// ------------------------------------------------------------------------------------------
// Stem convolution (Cin = 3) without im2col.
//
// The image is held as a zero-padded NHWC4 buffer x4p[N][Hp][Wp][4] (channel 3 = 0, logical pixel
// (ih, iw) at (ih + pad_top, iw + pad_left)).  For one filter row kh, the K slice of output pixel
// (oh, ow) is the 64 *contiguous* bf16 values x4p[n, s*oh + kh, s*ow : s*ow + 16, 0:4]: 16 pixels x
// 4 channels, of which the first KW pixels x 3 channels carry non-zero weights.  A TMA tensor map
// with OVERLAPPING windows (dim1 = ow with a byte stride of s*8, smaller than the 128-byte inner
// extent) delivers exactly that tile, so the tap-table kernel runs unchanged with KH "taps" of one
// 64-wide chunk each.  K is padded 147 -> 448 (7x7) / 108 -> 384 (6x6): the stem is ~3 % of the
// model's FLOPs and this removes the 10.9 GB im2col matrix and two HBM passes over it.
namespace t2r {
int make_stem_maps(CUtensorMap* maps, const void* x4p, int N, int Hp, int Wp, int KW, int stride, int Ho, int Wo,
                   int TW, int TH) {
  const char* base = static_cast<const char*>(x4p);
  (void)Ho;
  if (stem_rows_per_chunk(KW, stride) == 2) {
    // Row-pair image layout [N][Hp/2][Wp][8] (t2r_stem_pack_image): the window under output pixel
    // (oh, ow) for filter rows (2j, 2j+1) is the 128 contiguous bytes at pair row oh + j, column 2*ow.
    uint64_t dims[4] = {64, uint64_t(Wo), uint64_t(Hp / 2), uint64_t(N)};
    uint64_t strides[3] = {uint64_t(stride) * 16, uint64_t(Wp) * 16, uint64_t(Hp / 2) * Wp * 16};
    uint32_t box[4] = {64, uint32_t(TW), uint32_t(TH), 1};
    if (encode_tmap_bf16(&maps[0], base, 4, dims, strides, box) != 0) return -1;
    for (int i = 1; i < 4; ++i) maps[i] = maps[0];
    return 0;
  }
  for (int ph = 0; ph < stride; ++ph) {
    const int rows = (Hp - ph + stride - 1) / stride;
    uint64_t dims[4] = {64, uint64_t(Wo), uint64_t(std::max(rows, 1)), uint64_t(N)};
    uint64_t strides[3] = {uint64_t(stride) * 8, uint64_t(stride) * Wp * 8, uint64_t(Hp) * Wp * 8};
    uint32_t box[4] = {64, uint32_t(TW), uint32_t(TH), 1};
    if (encode_tmap_bf16(&maps[ph], base + size_t(ph) * Wp * 8, 4, dims, strides, box) != 0) return -1;
  }
  for (int i = stride; i < 4; ++i) maps[i] = maps[0];
  return 0;
}

int make_stem_taps(ConvTap* taps, int KH, int KW, int stride) {
  const int rows = stem_rows_per_chunk(KW, stride);
  const int n = (KH + rows - 1) / rows;
  for (int j = 0; j < n; ++j) {
    const int kh = j * rows;
    taps[j].map = int8_t(rows == 2 ? 0 : kh % stride);
    taps[j].dh = int8_t(kh / stride);
    taps[j].dw = 0;
    taps[j].kchunk0 = j;
  }
  return n;
}
}  // namespace t2r

extern "C" int32_t t2r_stem_conv_fprop(const T2RConvDesc* d, const void* x4p, int32_t Hp, int32_t Wp,
                                       const void* w_stem, const float* bias, void* y, void* stream) {
  T2R_CHECK_ARG(d && d->struct_size == sizeof(T2RConvDesc) && x4p && w_stem && y, "stem_conv_fprop: bad args");
  T2R_CHECK_ARG(d->Cin == 3 && d->KW <= 16 && d->KH <= kMaxTaps && d->Cout % 64 == 0 && d->stride >= 1 &&
                    d->stride <= 2, "stem_conv_fprop: unsupported geometry");
  const int rpc = stem_rows_per_chunk(d->KW, d->stride);
  const int n_chunks = (d->KH + rpc - 1) / rpc;
  T2R_CHECK_ARG(Wp % 2 == 0 && Hp % rpc == 0 && Wp >= d->stride * (d->Wo - 1) + 16 / rpc &&
                    Hp >= d->stride * (d->Ho - 1) + n_chunks * rpc,
                "stem_conv_fprop: padded image %dx%d too small", Hp, Wp);
  IgemmParams p;
  memset(&p, 0, sizeof(p));
  pick_tile(d->Ho, d->Wo, 128, &p.TW, &p.TH);
  if (make_stem_maps(p.tmap_a, x4p, d->N, Hp, Wp, d->KW, d->stride, d->Ho, d->Wo, p.TW, p.TH) < 0) return T2R_ERR_CUDA;
  const uint64_t Ktot = uint64_t(n_chunks) * 64;
  bool tma = false;
  const int block_n = pick_block_n(d->Cout, (long long)Ktot, 0, &tma);
  uint64_t dims[2] = {Ktot, uint64_t(d->Cout)};
  uint64_t strides[1] = {Ktot * 2};
  uint32_t box[2] = {64, uint32_t(block_n)};
  if (encode_tmap_bf16(&p.tmap_b, w_stem, 2, dims, strides, box) != 0) return T2R_ERR_CUDA;
  p.chunks_per_tap = 1;
  p.n_taps = make_stem_taps(p.taps, d->KH, d->KW, d->stride);
  p.tiles_w = int(ceil_div(d->Wo, p.TW));
  p.tiles_h = int(ceil_div(d->Ho, p.TH));
  p.N = d->N; p.Ho = d->Ho; p.Wo = d->Wo; p.Cout = d->Cout;
  p.os_w = d->Cout;
  p.os_h = (long long)d->Wo * d->Cout;
  p.os_n = (long long)d->Ho * d->Wo * d->Cout;
  p.out = y; p.bias = bias; p.flags = bias ? T2R_EPI_BIAS : 0;
  return dispatch_igemm(p, block_n, tma, static_cast<cudaStream_t>(stream));
}
