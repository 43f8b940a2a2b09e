// test_bn_bwd_gemm.cu — stand-alone GPU harness (no Python, no torch) for the batch-norm backward through a 1x1
// consumer's GEMMs: t2r_conv2d_wgrad_bnsums -> t2r_bn_backward_gemm_finalize -> t2r_conv2d_dgrad_bnapply against
// naive CPU loops in double.  Usage: ./test_bn_bwd_gemm [filter-substring]; exit code = number of failures.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <functional>
#include <string>
#include <vector>

#include "../../include/t2r_b200.h"

static int g_fail = 0, g_pass = 0;
static const char* g_filter = nullptr;

#define CK(expr)                                                                   \
  do {                                                                             \
    cudaError_t _e = (expr);                                                       \
    if (_e != cudaSuccess) {                                                       \
      printf("[FATAL] %s -> %s (%s:%d)\n", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      printf("SUMMARY pass=%d fail=%d (aborted)\n", g_pass, g_fail + 1);          \
      exit(100);                                                                   \
    }                                                                              \
  } while (0)
#define T2R(expr)                                                                  \
  do {                                                                             \
    int _rc = (expr);                                                              \
    if (_rc != 0) {                                                                \
      printf("[FAIL] %s rc=%d: %s\n", #expr, _rc, t2r_last_error());               \
      ++g_fail;                                                                    \
      return;                                                                      \
    }                                                                              \
  } while (0)

static uint32_t rng_state = 12345;
static float frand() {  // uniform [-1,1)
  rng_state = rng_state * 1664525u + 1013904223u;
  return float(rng_state >> 8) * (2.0f / 16777216.0f) - 1.0f;
}
static float bf16r(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

template <class T>
struct Dev {
  T* p = nullptr;
  size_t n = 0;
  explicit Dev(size_t n_) : n(n_) { CK(cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T))); CK(cudaMemset(p, 0, std::max<size_t>(n,1) * sizeof(T))); }
  ~Dev() { cudaFree(p); }
  void up(const std::vector<T>& h) { CK(cudaMemcpy(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice)); }
  std::vector<T> down() const { std::vector<T> h(n); CK(cudaMemcpy(h.data(), p, n * sizeof(T), cudaMemcpyDeviceToHost)); return h; }
};

static std::vector<__nv_bfloat16> to_bf16(const std::vector<float>& v) {
  std::vector<__nv_bfloat16> o(v.size());
  for (size_t i = 0; i < v.size(); ++i) o[i] = __float2bfloat16_rn(v[i]);
  return o;
}
static std::vector<float> from_bf16(const std::vector<__nv_bfloat16>& v) {
  std::vector<float> o(v.size());
  for (size_t i = 0; i < v.size(); ++i) o[i] = __bfloat162float(v[i]);
  return o;
}
static std::vector<float> randv(size_t n, float scale = 1.f, bool round_bf16 = true) {
  std::vector<float> v(n);
  for (auto& x : v) { x = frand() * scale; if (round_bf16) x = bf16r(x); }
  return v;
}

static void report(const std::string& name, const std::vector<float>& got, const std::vector<float>& ref,
                   float rtol, float atol) {
  double maxerr = 0, maxref = 0;
  size_t bad = 0, first_bad = 0;
  for (size_t i = 0; i < ref.size(); ++i) {
    const double e = fabs(double(got[i]) - double(ref[i]));
    if (!(e <= atol + rtol * fabs(ref[i]))) { if (!bad) first_bad = i; ++bad; }
    if (e > maxerr || e != e) maxerr = e;
    if (fabs(ref[i]) > maxref) maxref = fabs(ref[i]);
  }
  if (bad) {
    printf("[FAIL] %-44s bad=%zu/%zu maxerr=%.4g maxref=%.4g first_bad=%zu got=%.6g ref=%.6g\n", name.c_str(), bad,
           ref.size(), maxerr, maxref, first_bad, got[first_bad], ref[first_bad]);
    ++g_fail;
  } else {
    printf("[PASS] %-44s n=%zu maxerr=%.4g maxref=%.4g\n", name.c_str(), ref.size(), maxerr, maxref);
    ++g_pass;
  }
  fflush(stdout);
}

static void sync_check(const char* what) {
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    printf("[FATAL] %s: %s\nSUMMARY pass=%d fail=%d (aborted)\n", what, cudaGetErrorString(e), g_pass, g_fail + 1);
    exit(100);
  }
}

struct ConvCase {
  const char* name;
  int N, H, W, Cin, Cout, KH, KW, stride, pt, pl, Ho, Wo, flags;
};

static T2RConvDesc mkdesc(const ConvCase& c) {
  T2RConvDesc d;
  memset(&d, 0, sizeof(d));
  d.struct_size = sizeof(d);
  d.N = c.N; d.H = c.H; d.W = c.W; d.Cin = c.Cin; d.Cout = c.Cout; d.KH = c.KH; d.KW = c.KW;
  d.stride = c.stride; d.pad_top = c.pt; d.pad_left = c.pl; d.Ho = c.Ho; d.Wo = c.Wo; d.flags = c.flags;
  return d;
}

// ------------------------------------------------------------------------------------------
// batch-norm backward through a 1x1 consumer's GEMMs: t2r_conv2d_wgrad_bnsums -> t2r_bn_backward_gemm_finalize ->
// t2r_conv2d_dgrad_bnapply against CPU loops in double (dw, dgamma, dbeta, dx)
// ------------------------------------------------------------------------------------------
static void test_bnbwd_gemm(const ConvCase& c, bool with_dpass) {
  std::string name = std::string("bn_bwd_gemm ") + c.name + (with_dpass ? " +dpass" : "");
  if (g_filter && !strstr(name.c_str(), g_filter)) return;
  const T2RConvDesc d = mkdesc(c);
  const int C = c.Cin, K = c.Cout;
  const long long rows = (long long)c.N * c.H * c.W;
  const size_t nx = size_t(rows) * C, ny = size_t(rows) * K, nw = size_t(K) * C;
  std::vector<float> x = randv(nx, 2.f), w = randv(nw, 1.0f / sqrtf(float(C)), false), dy = randv(ny), dp = randv(nx),
                     scale = randv(C, 1.f, false), shift = randv(C, 1.f, false), mean = randv(C, 0.5f, false),
                     invstd = randv(C, 1.f, false);
  for (auto& v : scale) v = 0.75f + 0.5f * v;
  scale[1] = -scale[1];          // negative gamma
  shift[2] = -100.f;             // a channel the ReLU masks everywhere
  for (auto& v : invstd) v = 1.f + 0.5f * v;
  Dev<__nv_bfloat16> dx_(nx), ddy(ny), ddp(nx), dout(nx), dwf(nw), dwd(nw);
  Dev<float> dw32(nw), dsc(C), dsh(C), dmean(C), dinv(C), dwg(nw), dgam(C), dbet(C), coef(2 * C);
  Dev<double> sums(2 * C);
  dx_.up(to_bf16(x)); ddy.up(to_bf16(dy)); ddp.up(to_bf16(dp)); dw32.up(w); dsc.up(scale); dsh.up(shift);
  dmean.up(mean); dinv.up(invstd);
  T2R(t2r_pack_weights(dw32.p, dwf.p, dwd.p, K, 1, C, nullptr));
  if (!t2r_conv2d_dgrad_bnapply_supported(&d)) {
    printf("[FAIL] %-44s dgrad_bnapply_supported() == 0\n", name.c_str());
    ++g_fail;
    return;
  }
  T2R(t2r_conv2d_wgrad_bnsums(&d, dx_.p, dsc.p, dsh.p, ddy.p, dwd.p, dwg.p, sums.p, nullptr));
  T2R(t2r_bn_backward_gemm_finalize(sums.p, rows, C, dmean.p, dinv.p, dsc.p, dgam.p, dbet.p, coef.p, nullptr));
  T2R(t2r_conv2d_dgrad_bnapply(&d, ddy.p, dwd.p, dx_.p, dsc.p, dsh.p, coef.p, with_dpass ? ddp.p : nullptr, dout.p,
                               nullptr));
  sync_check(name.c_str());
  std::vector<float> wb(nw);   // the bf16 weights both GEMMs multiply with
  for (size_t i = 0; i < nw; ++i) wb[i] = bf16r(w[i]);
  std::vector<double> dwr(nw, 0.0), gr(nx), db(C, 0.0), sgx(C, 0.0);
  for (long long r = 0; r < rows; ++r)
    for (int ch = 0; ch < C; ++ch) {
      const float xv = x[r * C + ch];
      const bool on = fmaf(xv, scale[ch], shift[ch]) > 0.f;
      const double z = on ? double(xv) * scale[ch] + shift[ch] : 0.0;
      double dz = 0.0;
      for (int n = 0; n < K; ++n) {
        dz += double(dy[r * K + n]) * wb[size_t(n) * C + ch];
        dwr[size_t(n) * C + ch] += double(dy[r * K + n]) * z;
      }
      gr[r * C + ch] = on ? dz : 0.0;
      db[ch] += gr[r * C + ch];
      sgx[ch] += gr[r * C + ch] * xv;
    }
  std::vector<float> dwf_ref(nw), dg_ref(C), db_ref(C), dx_ref(nx);
  double wmax = 0, gmax = 0, xmax = 0;
  std::vector<double> kb(C), kc(C);
  for (int ch = 0; ch < C; ++ch) {
    const double dg = invstd[ch] * (sgx[ch] - double(mean[ch]) * db[ch]);
    dg_ref[ch] = float(dg);
    db_ref[ch] = float(db[ch]);
    gmax = fmax(gmax, fmax(fabs(dg), fabs(db[ch])));
    const double t = double(scale[ch]) * dg * invstd[ch] / double(rows);
    kb[ch] = -t;
    kc[ch] = t * mean[ch] - double(scale[ch]) * db[ch] / double(rows);
  }
  for (size_t i = 0; i < nw; ++i) { dwf_ref[i] = float(dwr[i]); wmax = fmax(wmax, fabs(dwr[i])); }
  for (size_t i = 0; i < nx; ++i) {
    const int ch = int(i % C);
    double v = scale[ch] * gr[i] + kb[ch] * x[i] + kc[ch];
    if (with_dpass) v += dp[i];
    dx_ref[i] = float(v);
    xmax = fmax(xmax, fabs(v));
  }
  report(name + " dw", dwg.down(), dwf_ref, 1e-3f, float(1e-4 * wmax + 1e-6));
  report(name + " dgamma", dgam.down(), dg_ref, 1e-3f, float(1e-4 * gmax + 1e-6));
  report(name + " dbeta", dbet.down(), db_ref, 1e-3f, float(1e-4 * gmax + 1e-6));
  report(name + " dx", from_bf16(dout.down()), dx_ref, 8e-3f, float(2e-3 * xmax));
}

static void tests_bnbwd_gemm() {
  const ConvCase cases[] = {
      {"1x1 19x17 64->256", 2, 19, 17, 64, 256, 1, 1, 1, 0, 0, 19, 17, 0},       // one group; dgrad tma<64>
      {"1x1 19x17 256->64", 2, 19, 17, 256, 64, 1, 1, 1, 0, 0, 19, 17, 0},       // four groups; dgrad tma<128> x2
      {"1x1 30x30 512->128", 1, 30, 30, 512, 128, 1, 1, 1, 0, 0, 30, 30, 0},
      {"1x1 7x13 1024->256", 2, 7, 13, 1024, 256, 1, 1, 1, 0, 0, 7, 13, 0},      // wgrad<256>, two group sets
  };
  test_bnbwd_gemm(cases[0], false);
  test_bnbwd_gemm(cases[1], true);
  test_bnbwd_gemm(cases[2], true);
  test_bnbwd_gemm(cases[3], true);
  test_bnbwd_gemm(cases[3], false);
}

int main(int argc, char** argv) {
  if (argc > 1) g_filter = argv[1];
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, 0));
  printf("device: %s sm_%d%d, %d SMs, lib version %d\n", prop.name, prop.major, prop.minor, prop.multiProcessorCount,
         t2r_version());
  tests_bnbwd_gemm();
  printf("SUMMARY pass=%d fail=%d\n", g_pass, g_fail);
  return g_fail;
}
