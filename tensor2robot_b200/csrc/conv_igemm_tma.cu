// conv_igemm_tma.cu — the tap-table implicit-GEMM convolution (see conv_igemm.cu) with a TMA epilogue.
//
// Low-K convolutions (ResNet 1x1 expansions, their data gradients) are bound by the epilogue's
// global traffic, not by the tensor core: each output tile is written (and, with the residual
// shortcut, first read) once, and a register epilogue exposes the DRAM latency of the residual loads
// and emits half-line stores.  Here the output tile lives in shared memory in the TMA box layout:
//
//   warp 3     : (residual only) TMA-loads the residual tile, same box geometry as the output, into
//                C buffer b as soon as the previous store has read it
//   epilogue   : TMEM -> registers -> (+bias) (+residual from smem) (ReLU) -> bf16 -> back to the
//                same smem bytes (+ fused bn_stats column sums) -> fence.proxy.async -> barrier ->
//                one thread per 64-channel sub-tile issues the TMA store; rows / columns outside
//                the tensor are clipped by TMA, so there is no per-row validity logic
//   C buffers  : two (tile i+1 is converted while tile i's store is still reading shared memory)
//
// BLOCK_N = 128 (warpgroup h owns 64-channel sub-tile h) or 64 (the two warpgroups split one
// sub-tile).  Main loop, warp roles and barriers are those of conv_igemm.cu.
#include <algorithm>
#include <cstdlib>

#include "conv_common.cuh"

namespace t2r {

struct IgemmTmaParams {
  IgemmParams g;
  CUtensorMap tmap_c;  // output view, box 64 x TW x TH x 1
  CUtensorMap tmap_r;  // residual, same geometry
  CUtensorMap tmap_x;  // kEpiBnApply: the batch-norm input x, same geometry
};

// kApply (kEpiBnApply): x lands in the C buffer (the output overwrites it in place) and the residual in a second
// pair of buffers; no column sums.  The GEMMs it serves have K = 64-256 (1-4 k-iterations per tile), so fewer
// operand stages make room for the extra buffers.
template <int BLOCK_N, bool kApply = false>
struct IgemmTmaCfg {
  static constexpr int kABytes = 128 * 128;
  static constexpr int kBBytes = BLOCK_N * 128;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = BLOCK_N == 64 ? 6 : (kApply ? 3 : 4);
  static constexpr int kSubTiles = BLOCK_N / 64;
  static constexpr int kCBytes = kSubTiles * 128 * 128;  // one bf16 output tile
  static constexpr int kRBytes = kApply ? 2 * kCBytes : 0;
  static constexpr int kTmemCols = 2 * BLOCK_N;
  static constexpr int kStatBytes = kApply ? 0 : 2 * kMaxStatChannels * 4;
  static constexpr int kSmemBytes = kStages * kStageBytes + 2 * kCBytes + kRBytes + kStatBytes + 256 + 1024;
  static_assert(kSmemBytes <= 232448, "shared memory");
};

__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(map),
               "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}

// kPro: see conv_igemm.cu (warps 12..15 rewrite each landed A tile as relu(bn_scale * x + bn_shift)).
// kEpiWarps: 8, or 16 for BLOCK_N = 128 without kPro.  The layers this kernel serves are bound by their output /
// residual traffic, and two consecutive tiles' epilogues run on the same warps: with 8 warps each converts two
// 32-column chunks per tile (~2 x 900 cycles of dependent TMEM load -> shared load -> convert -> shared store ->
// column sums) and the tile rate is latency bound at ~0.6 of the HBM roofline; 16 warps take one chunk each.
template <int BLOCK_N, bool kPro, int kEpiWarps, bool kApply>
__global__ void __launch_bounds__(128 + 32 * kEpiWarps + (kPro ? 128 : 0), 1)
conv_igemm_tma_kernel(const __grid_constant__ IgemmTmaParams pp) {
  static_assert(kEpiWarps == 8 || (kEpiWarps == 16 && BLOCK_N == 128 && !kPro), "16 epilogue warps: BLOCK_N 128 only");
  static_assert(!(kPro && kApply), "operand transform and batch-norm apply epilogue do not combine");
  using Cfg = IgemmTmaCfg<BLOCK_N, kApply>;
  const IgemmParams& p = pp.g;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t c_base = smem_base + Cfg::kStages * Cfg::kStageBytes;
  const uint32_t r_base = c_base + 2 * Cfg::kCBytes;   // kApply: residual tiles
  const uint32_t stat_base = r_base + Cfg::kRBytes;
  const uint32_t bar_base = stat_base + Cfg::kStatBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (Cfg::kStages + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::kStages + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::kStages + 2 + s); };
  auto cfull_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::kStages + 4 + s); };
  auto cempty_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::kStages + 6 + s); };
  const uint32_t tmem_ptr_addr = bar_base + 8u * (2 * Cfg::kStages + 8);
  auto ready_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::kStages + 9 + s); };
  volatile uint32_t* tmem_ptr_gen =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_ptr_addr - smem_u32(smem_raw)));
  float* stat_acc = reinterpret_cast<float*>(smem_raw + (stat_base - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const bool bnbwd = (p.flags & kEpiBnBwd) != 0;  // the "residual" tile is then the normalised tensor x
  const bool has_res = (p.flags & T2R_EPI_RESIDUAL) != 0 || bnbwd;
  const bool apply_res = kApply && p.residual != nullptr;
  const bool loads_c = has_res || kApply;             // warp 3 feeds the C buffers

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < 4; ++i) tma_prefetch_desc(&p.tmap_a[i]);
    tma_prefetch_desc(&p.tmap_b);
    tma_prefetch_desc(&pp.tmap_c);
    tma_prefetch_desc(&pp.tmap_r);
    if (kApply) tma_prefetch_desc(&pp.tmap_x);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < Cfg::kStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
      if (kPro) mbar_init(ready_bar(s), 4);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), kEpiWarps);
      mbar_init(cfull_bar(s), 1);
      mbar_init(cempty_bar(s), Cfg::kSubTiles);  // one arrival per store-issuing thread
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
    // Without a residual: three warps take the k-iterations round-robin.  With one: warps 0 and 2
    // do, and warp 3 only feeds residual tiles into the C buffers, so that the operand pipeline
    // never waits for an output store.
    if (lane == 0) {
      const int pid = warp == 0 ? 0 : warp - 1;
      const int n_prod = loads_c ? 2 : 3;
      if (pid < n_prod) {
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
                mbar_expect_tx(full_bar(stage), Cfg::kStageBytes);
                tma_load_4d(sa, &p.tmap_a[tap.map], full_bar(stage), c * 64, ow0 + tap.dw, oh0 + tap.dh, img);
                tma_load_2d(sa + Cfg::kABytes, &p.tmap_b, full_bar(stage), (tap.kchunk0 + c) * 64, nt * BLOCK_N);
              }
              if (++turn == n_prod) turn = 0;
              if (++stage == Cfg::kStages) {
                stage = 0;
                phase ^= 1u;
              }
            }
          }
        }
      } else {
        int cb = 0;
        uint32_t cphase = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
          const int nt = tile % p.n_tiles_n;
          const int mt = tile / p.n_tiles_n;
          const int img = mt / tiles_per_img;
          const int rem = mt - img * tiles_per_img;
          const int oh0 = (rem / p.tiles_w) * p.TH;
          const int ow0 = (rem % p.tiles_w) * p.TW;
          mbar_wait(cempty_bar(cb), cphase ^ 1u);  // the store that last used this buffer has read it
          mbar_expect_tx(cfull_bar(cb), apply_res ? 2 * Cfg::kCBytes : Cfg::kCBytes);
#pragma unroll
          for (int j = 0; j < Cfg::kSubTiles; ++j)
            tma_load_4d(c_base + cb * Cfg::kCBytes + j * 16384, kApply ? &pp.tmap_x : &pp.tmap_r, cfull_bar(cb),
                        nt * BLOCK_N + j * 64, ow0, oh0, img);
          if (apply_res)
#pragma unroll
            for (int j = 0; j < Cfg::kSubTiles; ++j)
              tma_load_4d(r_base + cb * Cfg::kCBytes + j * 16384, &pp.tmap_r, cfull_bar(cb), nt * BLOCK_N + j * 64, ow0,
                          oh0, img);
          if (++cb == 2) {
            cb = 0;
            cphase ^= 1u;
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
    // ===================== operand transform: 4 warps (see conv_igemm.cu) =====================
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
  } else if (warp >= 4 && warp < 4 + kEpiWarps) {
    // ===================== epilogue: 8 or 16 warps =====================
    // Warp w reads TMEM lanes 32 * (w % 4) .. +31 (one output pixel per thread); `part` picks the columns:
    //   BLOCK_N 128,  8 warps: part = sub-tile (64 channels, two 32-column chunks per warp)
    //   BLOCK_N 128, 16 warps: part = 32-column chunk 0..3 (sub-tile part / 2)
    //   BLOCK_N  64,  8 warps: part = 32-column half of the single sub-tile
    const int ew = warp - 4;
    const int quad = ew & 3;
    const int part = ew >> 2;
    constexpr bool kWide = kEpiWarps == 16;
    constexpr int kChunks = (BLOCK_N == 128 && !kWide) ? 2 : 1;
    const int sub = BLOCK_N == 128 ? (kWide ? part >> 1 : part) : 0;            // 64-channel sub-tile this warp writes
    const int col0 = BLOCK_N == 128 ? (kWide ? (part & 1) * 32 : 0) : part * 32;   // first column inside the sub-tile
    const int half = sub;
    const int row = quad * 32 + lane;
    const int th = row / p.TW;
    const int tw = row - th * p.TW;
    const uint32_t rsw = uint32_t(row) & 7u;
    // one thread per sub-tile issues its TMA store
    const bool elected = (quad == 0 && lane == 0) && (BLOCK_N == 128 ? (!kWide || (part & 1) == 0) : part == 0);
    int as = 0, cb = 0, pending_cb = -1;
    uint32_t aphase = 0, cphase = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const int nt = tile % p.n_tiles_n;
      const int mt = tile / p.n_tiles_n;
      const int img = mt / tiles_per_img;
      const int rem = mt - img * tiles_per_img;
      const int oh0 = (rem / p.tiles_w) * p.TH, ow0 = (rem % p.tiles_w) * p.TW;
      const bool valid = (oh0 + th < p.Ho) && (ow0 + tw < p.Wo);
      const uint32_t csub = c_base + cb * Cfg::kCBytes + sub * 16384;
      const uint32_t crow = csub + uint32_t(row) * 128u;
      const uint32_t rrow = crow + (r_base - c_base);   // kApply: the residual row beside it
      if (elected && pending_cb >= 0) {
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        mbar_arrive(cempty_bar(pending_cb));
        pending_cb = -1;
      }
      if (loads_c) mbar_wait(cfull_bar(cb), cphase);   // the residual tile has landed in the C buffer
      else mbar_wait(cempty_bar(cb), cphase ^ 1u);     // the store that last used the buffer has read it
      mbar_wait(tfull_bar(as), aphase);
      tc_fence_after();
#pragma unroll
      for (int c = 0; c < kChunks; ++c) {
        const int colc = col0 + c * 32;                       // column inside the sub-tile
        const int ch = nt * BLOCK_N + sub * 64 + colc;        // global channel
        uint32_t v[32];
        tmem_ld_32x32(tmem_base + (uint32_t(quad * 32) << 16) + as * BLOCK_N + sub * 64 + colc, v);
        tmem_ld_wait();
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
        const uint32_t chunk0 = uint32_t(colc) >> 3;          // first 16-byte chunk of these 32 columns
        if (kApply) {
          // dx = scale * [scale * x + shift > 0] * acc + kb * x + kc (+ residual); the arithmetic of
          // bn_bwd_apply_kernel (norm.cu) on the fp32 accumulator instead of the bf16-rounded g
#pragma unroll
          for (uint32_t j = 0; j < 4; ++j) {
            const uint32_t off = ((chunk0 + j) ^ rsw) << 4;
            uint4 q, r = make_uint4(0u, 0u, 0u, 0u);
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(q.x), "=r"(q.y), "=r"(q.z), "=r"(q.w)
                         : "r"(crow + off)
                         : "memory");
            if (apply_res)
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                           : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                           : "r"(rrow + off)
                           : "memory");
            const uint32_t qv[4] = {q.x, q.y, q.z, q.w}, rv[4] = {r.x, r.y, r.z, r.w};
            float sc[8], sh[8], kb[8], kc[8];
            const int c8 = ch + 8 * int(j);
            load8(p.bn_scale + c8, sc);
            load8(p.bn_shift + c8, sh);
            load8(p.bn_coef + c8, kb);
            load8(p.bn_coef + p.Cout + c8, kc);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float x = (i & 1) ? bf16_hi(qv[i >> 1]) : bf16_lo(qv[i >> 1]);
              const float dz = fmaf(x, sc[i], sh[i]) > 0.f ? f[8 * j + i] : 0.f;
              float o = fmaf(sc[i], dz, fmaf(kb[i], x, kc[i]));
              if (apply_res) o += (i & 1) ? bf16_hi(rv[i >> 1]) : bf16_lo(rv[i >> 1]);
              f[8 * j + i] = o;
            }
          }
        } else if (bnbwd) {
          // g = dz * [scale * x + shift > 0] (x = the tile warp 3 loaded), rounded to bf16 like the stored value;
          // column sums of g * x by shuffles, those of g from the staged tile below (as the fused bn_stats)
          float xv[32];
#pragma unroll
          for (uint32_t j = 0; j < 4; ++j) {
            uint4 q;
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(q.x), "=r"(q.y), "=r"(q.z), "=r"(q.w)
                         : "r"(crow + (((chunk0 + j) ^ rsw) << 4))
                         : "memory");
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
        } else if (has_res) {
#pragma unroll
          for (uint32_t j = 0; j < 4; ++j) {
            uint4 q;
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(q.x), "=r"(q.y), "=r"(q.z), "=r"(q.w)
                         : "r"(crow + (((chunk0 + j) ^ rsw) << 4))
                         : "memory");
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
#pragma unroll
        for (uint32_t j = 0; j < 4; ++j) {
          uint32_t q0 = pack_bf16(f[8 * j + 0], f[8 * j + 1]), q1 = pack_bf16(f[8 * j + 2], f[8 * j + 3]);
          uint32_t q2 = pack_bf16(f[8 * j + 4], f[8 * j + 5]), q3 = pack_bf16(f[8 * j + 6], f[8 * j + 7]);
          if (!valid) q0 = q1 = q2 = q3 = 0u;  // clipped by the TMA store; zero so that bn_stats ignores it
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(crow + (((chunk0 + j) ^ rsw) << 4)), "r"(q0),
                       "r"(q1), "r"(q2), "r"(q3)
                       : "memory");
        }
        if (p.stats != nullptr) {
          // fused bn_stats: lane l sums column l of this warp's 32 rows x 32 columns
          __syncwarp();
          float s1 = 0.f, s2 = 0.f;
          const uint32_t cj = chunk0 + (uint32_t(lane) >> 3), cbyte = (uint32_t(lane) & 7u) * 2u;
          const uint32_t wrow = csub + uint32_t(quad * 32) * 128u;
#pragma unroll
          for (uint32_t r = 0; r < 32; ++r) {
            uint16_t h;
            asm volatile("ld.shared.u16 %0, [%1];" : "=h"(h) : "r"(wrow + r * 128u + ((cj ^ (r & 7u)) << 4) + cbyte) : "memory");
            const float x = __uint_as_float(uint32_t(h) << 16);
            s1 += x;
            s2 = fmaf(x, x, s2);
          }
          atomicAdd(stat_acc + ch + lane, s1);
          if (!bnbwd) atomicAdd(stat_acc + p.Cout + ch + lane, s2);
        }
      }
      // accumulator stage is free for the MMA of tile i+2
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(as));
      // hand the finished sub-tile to TMA
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      if (BLOCK_N == 128) {   // the warps that wrote sub-tile `sub`
        asm volatile("bar.sync %0, %1;" ::"r"(1 + half), "r"(kWide ? 256 : 128) : "memory");
      } else {
        asm volatile("bar.sync 1, 256;" ::: "memory");
      }
      if (elected) {
        tma_store_4d(&pp.tmap_c, csub, nt * BLOCK_N + sub * 64, ow0, oh0, img);
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        pending_cb = cb;  // released at the top of the next tile, once the store has read the buffer
      }
      if (++as == 2) {
        as = 0;
        aphase ^= 1u;
      }
      if (++cb == 2) {
        cb = 0;
        cphase ^= 1u;
      }
    }
    if (elected) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    if (p.stats != nullptr) {
      asm volatile("bar.sync 3, %0;" ::"r"(32 * kEpiWarps) : "memory");
      for (int i = threadIdx.x - 128; i < 2 * p.Cout; i += 32 * kEpiWarps) {
        const float x = stat_acc[i];
        if (x != 0.f) atomicAdd(p.stats + i, double(x));
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

template <int BLOCK_N, bool kPro, int kEpiWarps, bool kApply = false>
static int launch_v(const IgemmTmaParams& pp, cudaStream_t stream) {
  using Cfg = IgemmTmaCfg<BLOCK_N, kApply>;
  static bool configured = false;
  if (!configured) {
    T2R_CUDA_OK(cudaFuncSetAttribute(conv_igemm_tma_kernel<BLOCK_N, kPro, kEpiWarps, kApply>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    configured = true;
  }
  const int grid = std::min(pp.g.total_tiles, num_sms());
  conv_igemm_tma_kernel<BLOCK_N, kPro, kEpiWarps, kApply>
      <<<grid, 128 + 32 * kEpiWarps + (kPro ? 128 : 0), Cfg::kSmemBytes, stream>>>(pp);
  T2R_LAUNCH_OK();
  return T2R_OK;
}
template <int BLOCK_N>
static int launch(const IgemmTmaParams& pp, cudaStream_t stream) {
  if (pp.g.flags & kEpiBnApply) return launch_v<BLOCK_N, false, 8, true>(pp, stream);
  if (pp.g.flags & kProBnRelu) return launch_v<BLOCK_N, true, 8>(pp, stream);
  return launch_v<BLOCK_N, false, 8>(pp, stream);
}
// BLOCK_N 128: T2R_TMA_EPI_WARPS=16 runs the epilogue on 16 warps (one 32-column chunk each).  Measured on the
// ResNet-50 step (gpurun_out/r02i_detail_epi{8,auto}.txt): no gain (64->256 1x1 at 118x118: 2.03 -> 1.99 ms; step
// 142.6 -> 143.5 ms), so 8 stays the default - the low-K layers are not bound by the epilogue's latency.
template <>
int launch<128>(const IgemmTmaParams& pp, cudaStream_t stream) {
  if (pp.g.flags & kEpiBnApply) return launch_v<128, false, 8, true>(pp, stream);
  if (pp.g.flags & kProBnRelu) return launch_v<128, true, 8>(pp, stream);
  static const char* mode = std::getenv("T2R_TMA_EPI_WARPS");
  const int k_iters = pp.g.n_taps * pp.g.chunks_per_tap;
  const bool wide = mode != nullptr && (mode[0] == 'a' ? k_iters <= 8 : (mode[0] == '1' && mode[1] == '6'));
  return wide ? launch_v<128, false, 16>(pp, stream) : launch_v<128, false, 8>(pp, stream);
}

int conv_igemm_tma_launch(const IgemmParams& p, int block_n, cudaStream_t stream) {
  IgemmTmaParams pp;
  pp.g = p;
  pp.g.n_tiles_n = int(ceil_div(p.Cout, block_n));
  pp.g.total_tiles = p.N * p.tiles_w * p.tiles_h * pp.g.n_tiles_n;
  if (pp.g.total_tiles <= 0) return T2R_OK;
  uint64_t dims[4] = {uint64_t(p.Cout), uint64_t(p.Wo), uint64_t(p.Ho), uint64_t(p.N)};
  uint64_t strides[3] = {uint64_t(p.os_w) * 2, uint64_t(p.os_h) * 2, uint64_t(p.os_n) * 2};
  uint32_t box[4] = {64, uint32_t(p.TW), uint32_t(p.TH), 1};
  if (encode_tmap_bf16(&pp.tmap_c, p.out, 4, dims, strides, box) != 0) return T2R_ERR_CUDA;
  const void* aux = (p.flags & kEpiBnBwd) ? p.bn_x : p.residual;
  if (encode_tmap_bf16(&pp.tmap_r, aux ? aux : p.out, 4, dims, strides, box) != 0) return T2R_ERR_CUDA;
  pp.tmap_x = pp.tmap_r;
  if ((p.flags & kEpiBnApply) && encode_tmap_bf16(&pp.tmap_x, p.bn_x, 4, dims, strides, box) != 0) return T2R_ERR_CUDA;
  return block_n == 128 ? launch<128>(pp, stream) : launch<64>(pp, stream);
}

}  // namespace t2r
