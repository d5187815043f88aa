// Stand-alone probe for the tcgen05 convolution kernels (kalle_audio_b200/csrc/conv_umma2.cuh, conv_ru2.cuh).
// Each invocation runs ONE case so a trap in one case cannot poison the others:
//   umma_probe <case> <variant>     variant 3: automatic tiling
//                                   variant 4: a grid of 3 CTAs, so every CTA loops over many tiles
//                                   variant 5: 128-row tiles at most 128 channels wide
//                                   variant 6: operand swap disabled (time rows on the M side)
//   umma_probe perf <idx> <version> <epilogue>   timing of full-size layers (no CPU check); version 2: automatic
//                                   tiling, 3: the table's MT / NT, 4: operand swap disabled
//   umma_probe ru <dilation> <B> <T> [perf]       the fused ResidualUnit against the CPU loops (or timed)
// The check is a double-precision channels-last convolution over the same bf16-rounded operands.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <random>
#include <vector>

#include "../kalle_audio_b200/csrc/conv_umma_host.cuh"

using namespace kvae;

#define CK(x)                                                                          \
  do {                                                                                 \
    cudaError_t e_ = (x);                                                              \
    if (e_ != cudaSuccess) {                                                           \
      printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__);  \
      exit(2);                                                                         \
    }                                                                                  \
  } while (0)

static float bf16r(float f) { return __bfloat162float(__float2bfloat16(f)); }

struct Case {
  const char* name;
  ConvGeom g;
  int B, T;
  int MT, NT;
  bool epi;  // exercise bias + residual + raw + snake outputs
};

static const Case kCases[] = {
    {"k1_c64_128_T128", {kConv, 64, 128, 1, 1, 1, 0}, 1, 128, 1, 128, false},
    {"k1_c256_256_T300", {kConv, 256, 256, 1, 1, 1, 0}, 2, 300, 2, 256, false},
    {"k7d1_c128", {kConv, 128, 128, 7, 1, 1, 3}, 2, 1000, 2, 128, false},
    {"k7d3_c128", {kConv, 128, 128, 7, 1, 3, 9}, 2, 1000, 2, 128, false},
    {"k7d9_c256", {kConv, 256, 256, 7, 1, 9, 27}, 1, 700, 2, 128, true},
    {"convT_s8_k16", {kConvT, 256, 128, 16, 8, 1, 4}, 2, 150, 2, 128, false},
    {"convT_s5_k11", {kConvT, 128, 64, 11, 5, 1, 3}, 1, 333, 2, 64, true},
    {"convT_s2_k4", {kConvT, 128, 128, 4, 2, 1, 1}, 1, 257, 2, 128, false},
    {"down_s4_k8", {kConv, 128, 256, 8, 4, 1, 2}, 2, 1024, 2, 256, false},
    {"down_s5_k10", {kConv, 64, 128, 10, 5, 1, 3}, 1, 1500, 1, 128, true},
    {"down_s8_k16", {kConv, 128, 128, 16, 8, 1, 4}, 1, 4096, 2, 128, false},
    {"k3_c512_128", {kConv, 512, 128, 3, 1, 1, 1}, 1, 216, 1, 128, false},
    {"k7_c64_2048", {kConv, 64, 2048, 7, 1, 1, 3}, 1, 216, 2, 256, true},
};
static const int kNumCases = sizeof(kCases) / sizeof(kCases[0]);

// packed weights [k][co][ci]
static void cpu_conv(const Case& c, const std::vector<float>& x, const std::vector<float>& w,
                     std::vector<double>& y, int T_out) {
  const ConvGeom& g = c.g;
  y.assign((size_t)c.B * T_out * g.Cout, 0.0);
  for (int b = 0; b < c.B; ++b)
    for (int k = 0; k < g.K; ++k) {
      if (g.kind == kConv) {
        for (int t = 0; t < T_out; ++t) {
          int ti = t * g.stride + k * g.dilation - g.pad;
          if (ti < 0 || ti >= c.T) continue;
          const float* xr = &x[((size_t)b * c.T + ti) * g.Cin];
          for (int co = 0; co < g.Cout; ++co) {
            const float* wr = &w[((size_t)k * g.Cout + co) * g.Cin];
            double s = 0;
            for (int ci = 0; ci < g.Cin; ++ci) s += (double)xr[ci] * wr[ci];
            y[((size_t)b * T_out + t) * g.Cout + co] += s;
          }
        }
      } else {
        for (int ti = 0; ti < c.T; ++ti) {
          int t = ti * g.stride - g.pad + k;
          if (t < 0 || t >= T_out) continue;
          const float* xr = &x[((size_t)b * c.T + ti) * g.Cin];
          for (int co = 0; co < g.Cout; ++co) {
            const float* wr = &w[((size_t)k * g.Cout + co) * g.Cin];
            double s = 0;
            for (int ci = 0; ci < g.Cin; ++ci) s += (double)xr[ci] * wr[ci];
            y[((size_t)b * T_out + t) * g.Cout + co] += s;
          }
        }
      }
    }
}

static int run_case(int idx, int variant) {
  const Case& c = kCases[idx];
  const ConvGeom& g = c.g;
  const int T_out = g.out_len(c.T);
  std::mt19937 rng(1234 + idx);
  std::normal_distribution<float> nd(0.f, 1.f);
  std::vector<float> x((size_t)c.B * c.T * g.Cin), w((size_t)g.K * g.Cout * g.Cin);
  for (auto& v : x) v = bf16r(nd(rng));
  const float ws = 1.0f / std::sqrt((float)(g.Cin * (g.kind == kConv ? g.K : (g.K + g.stride - 1) / g.stride)));
  for (auto& v : w) v = bf16r(nd(rng) * ws);
  std::vector<float> bias(g.Cout), sa(g.Cout), sib(g.Cout), res((size_t)c.B * T_out * g.Cout);
  for (int i = 0; i < g.Cout; ++i) {
    bias[i] = nd(rng) * 0.1f;
    sa[i] = std::exp(nd(rng) * 0.3f);
    sib[i] = 1.0f / (std::exp(nd(rng) * 0.3f) + 1e-9f);
  }
  for (auto& v : res) v = nd(rng);
  std::vector<double> ref;
  cpu_conv(c, x, w, ref, T_out);

  std::vector<__nv_bfloat16> xb(x.size()), wb(w.size());
  for (size_t i = 0; i < x.size(); ++i) xb[i] = __float2bfloat16(x[i]);
  for (size_t i = 0; i < w.size(); ++i) wb[i] = __float2bfloat16(w[i]);
  __nv_bfloat16 *dx, *dw, *dact;
  float *dbias, *dsa, *dsib, *dres, *draw;
  const size_t nout = (size_t)c.B * T_out * g.Cout;
  CK(cudaMalloc(&dx, xb.size() * 2));
  CK(cudaMalloc(&dw, wb.size() * 2));
  CK(cudaMalloc(&dact, nout * 2));
  CK(cudaMalloc(&draw, nout * 4));
  CK(cudaMalloc(&dres, nout * 4));
  CK(cudaMalloc(&dbias, g.Cout * 4));
  CK(cudaMalloc(&dsa, g.Cout * 4));
  CK(cudaMalloc(&dsib, g.Cout * 4));
  CK(cudaMemcpy(dx, xb.data(), xb.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dw, wb.data(), wb.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dres, res.data(), nout * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dbias, bias.data(), g.Cout * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dsa, sa.data(), g.Cout * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dsib, sib.data(), g.Cout * 4, cudaMemcpyHostToDevice));
  CK(cudaMemset(draw, 0xff, nout * 4));
  CK(cudaMemset(dact, 0xff, nout * 2));

  ConvEpilogue ep;
  ep.out_raw = draw;
  ep.out_raw_f32 = 1;
  if (c.epi) {
    ep.bias = dbias;
    ep.residual = dres;
    ep.residual_f32 = 1;
    ep.out_act = dact;
    ep.snake_a = dsa;
    ep.snake_inv_b = dsib;
  }
  std::string err;
  ConvTuning2 tune2;
  if (variant == 4) tune2.max_ctas = 3;
  if (variant == 5) { tune2.MT = 1; tune2.NT = c.NT > 128 ? 128 : c.NT; }
  if (variant == 6) tune2.swap = 0;   // time rows on the M side even for 128-channel tiles
  ConvLaunch2 L2;
  if (!prepare_conv_umma2(g, dx, c.B, c.T, dw, ep, tune2, L2, err)) {
    printf("CASE %d %s variant %d: prepare failed: %s\n", idx, c.name, variant, err.c_str());
    return 3;
  }
  printf("CASE %d %s variant %d: grid %d smem %zu MT %d NT %d acc %d RB %d nbox %d SA %d SB %d tmem %d tiles %d\n",
         idx, c.name, variant, L2.grid, L2.smem, L2.p.MT, L2.p.NT, L2.p.acc_stages, L2.p.RB, L2.p.nbox, L2.p.SA,
         L2.p.SB, L2.p.tmem_cols, L2.p.total_tiles);
  fflush(stdout);
  CK(launch_conv_umma2(L2, 0));
  CK(cudaDeviceSynchronize());
  std::vector<float> raw(nout);
  std::vector<__nv_bfloat16> act(nout);
  CK(cudaMemcpy(raw.data(), draw, nout * 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(act.data(), dact, nout * 2, cudaMemcpyDeviceToHost));
  double max_err = 0, max_ref = 0, max_err_act = 0;
  size_t bad = 0, first_bad = (size_t)-1;
  for (size_t i = 0; i < nout; ++i) {
    double r = ref[i];
    if (c.epi) r += bias[i % g.Cout] + res[i];
    double e = std::fabs((double)raw[i] - r);
    if (!(e <= 1e30)) e = 1e30;  // NaN
    max_err = std::max(max_err, e);
    max_ref = std::max(max_ref, std::fabs(r));
    if (e > 2e-2) { if (!bad) first_bad = i; ++bad; }
    if (c.epi) {
      double s = std::sin(r * sa[i % g.Cout]);
      double a = r + sib[i % g.Cout] * s * s;
      double ea = std::fabs((double)__bfloat162float(act[i]) - a);
      if (!(ea <= 1e30)) ea = 1e30;
      max_err_act = std::max(max_err_act, ea / (1.0 + std::fabs(a)));
    }
  }
  const bool ok = bad == 0 && (!c.epi || max_err_act < 1e-2);
  printf("RESULT case %d %s variant %d: %s max_err %.3e max_ref %.3e bad %zu/%zu act_rel_err %.3e\n", idx,
         c.name, variant, ok ? "PASS" : "FAIL", max_err, max_ref, bad, nout, max_err_act);
  if (bad) {
    size_t i = first_bad;
    size_t co = i % g.Cout, t = (i / g.Cout) % T_out, b = i / ((size_t)g.Cout * T_out);
    printf("  first bad at b=%zu t=%zu co=%zu got %.5f want %.5f\n", b, t, co, raw[i],
           ref[i] + (c.epi ? bias[co] + res[i] : 0.0));
    // error map over (t mod 16) to expose row-shift / swizzle mistakes
    std::vector<size_t> by_row(16, 0);
    for (size_t j = 0; j < nout; ++j) {
      double r = ref[j] + (c.epi ? bias[j % g.Cout] + res[j] : 0.0);
      if (!(std::fabs((double)raw[j] - r) <= 2e-2)) by_row[(j / g.Cout) % T_out % 16]++;
    }
    printf("  bad count by t%%16:");
    for (int j = 0; j < 16; ++j) printf(" %zu", by_row[j]);
    printf("\n");
  }
  return ok ? 0 : 1;
}

struct Perf {
  const char* name;
  ConvGeom g;
  int B, T, MT, NT;
};
static const Perf kPerf[] = {
    {"sao_s5_k7_c128", {kConv, 128, 128, 7, 1, 1, 3}, 4, 442368, 2, 128},
    {"sao_s5_k1_c128", {kConv, 128, 128, 1, 1, 1, 0}, 4, 442368, 2, 128},
    {"sao_s4_k7_c256", {kConv, 256, 256, 7, 1, 3, 9}, 4, 221184, 2, 256},
    {"sao_s4_k7_c256_nt128", {kConv, 256, 256, 7, 1, 3, 9}, 4, 221184, 2, 128},
    {"sao_s3_k7_c512", {kConv, 512, 512, 7, 1, 9, 27}, 4, 55296, 2, 256},
    {"sao_s1_k7_c2048", {kConv, 2048, 2048, 7, 1, 1, 3}, 16, 1728, 2, 256},
    {"sao_convT_s8_1024_512", {kConvT, 1024, 512, 16, 8, 1, 4}, 16, 1728, 2, 256},
    {"sao_convT_s2_128_128", {kConvT, 128, 128, 4, 2, 1, 1}, 4, 221184, 2, 128},
};
static const int kNumPerf = sizeof(kPerf) / sizeof(kPerf[0]);

static int run_perf(int idx, int ver, int epi) {
  const Perf& c = kPerf[idx];
  const ConvGeom& g = c.g;
  const int T_out = g.out_len(c.T);
  const size_t nin = (size_t)c.B * c.T * g.Cin, nw = (size_t)g.K * g.Cout * g.Cin,
               nout = (size_t)c.B * T_out * g.Cout;
  __nv_bfloat16 *dx, *dw, *dact;
  CK(cudaMalloc(&dx, nin * 2));
  CK(cudaMalloc(&dw, nw * 2));
  CK(cudaMalloc(&dact, nout * 2));
  {  // realistic operand values (power draw and clocks depend on the data)
    std::vector<__nv_bfloat16> h(1 << 20);
    std::mt19937 rng(7);
    std::normal_distribution<float> nd(0.f, 1.f);
    for (auto& v : h) v = __float2bfloat16(nd(rng));
    for (size_t o = 0; o < nin; o += h.size())
      CK(cudaMemcpy(dx + o, h.data(), std::min(h.size(), nin - o) * 2, cudaMemcpyHostToDevice));
    for (auto& v : h) v = __float2bfloat16(nd(rng) * 0.03f);
    for (size_t o = 0; o < nw; o += h.size())
      CK(cudaMemcpy(dw + o, h.data(), std::min(h.size(), nw - o) * 2, cudaMemcpyHostToDevice));
  }
  float *dbias, *dsa, *dsib, *dres = nullptr, *draw = nullptr;
  CK(cudaMalloc(&dbias, g.Cout * 4));
  CK(cudaMalloc(&dsa, g.Cout * 4));
  CK(cudaMalloc(&dsib, g.Cout * 4));
  {
    std::vector<float> ones(g.Cout, 1.0f), zeros(g.Cout, 0.01f);
    CK(cudaMemcpy(dbias, zeros.data(), g.Cout * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dsa, ones.data(), g.Cout * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dsib, ones.data(), g.Cout * 4, cudaMemcpyHostToDevice));
  }
  ConvEpilogue ep;
  ep.out_act = dact;
  if (epi >= 1) { ep.bias = dbias; ep.snake_a = dsa; ep.snake_inv_b = dsib; }
  if (epi >= 2) {
    CK(cudaMalloc(&dres, nout * 4));
    CK(cudaMalloc(&draw, nout * 4));
    CK(cudaMemset(dres, 0, nout * 4));
    ep.residual = dres; ep.residual_f32 = 1; ep.out_raw = draw; ep.out_raw_f32 = 1;
  }
  std::string err;
  ConvLaunch2 L2;
  ConvTuning2 tune2;
  if (ver == 3) { tune2.MT = c.MT; tune2.NT = c.NT; }
  if (ver == 4) tune2.swap = 0;
  if (!prepare_conv_umma2(g, dx, c.B, c.T, dw, ep, tune2, L2, err)) {
    printf("PERF %s: prepare failed: %s\n", c.name, err.c_str());
    return 3;
  }
  auto launch = [&]() { return launch_conv_umma2(L2, 0); };
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  for (int i = 0; i < 3; ++i) CK(launch());
  CK(cudaDeviceSynchronize());
  const int iters = 10;
  CK(cudaEventRecord(e0));
  for (int i = 0; i < iters; ++i) CK(launch());
  CK(cudaEventRecord(e1));
  CK(cudaDeviceSynchronize());
  float ms;
  CK(cudaEventElapsedTime(&ms, e0, e1));
  ms /= iters;
  const double taps_eff = (g.kind == kConv) ? (double)g.K * T_out : (double)g.K * c.T;
  const double flops = 2.0 * c.B * taps_eff * g.Cin * g.Cout;
  const double bytes = (nin + nout) * 2.0 + (epi >= 2 ? nout * 8.0 : 0.0);
  printf("PERF v%d epi%d %s: %.3f ms  %.1f TFLOP/s  %.1f GB/s  MT %d NT %d swap %d acc %d grid %d smem %zu SA %d SB %d\n",
         ver, epi, c.name, ms, flops / ms * 1e-9, bytes / ms * 1e-6, L2.p.MT, L2.p.NT, L2.p.swap, L2.p.acc_stages,
         L2.grid, L2.smem, L2.p.SA, L2.p.SB);
  return 0;
}

// Fused ResidualUnit check: x' = x + W1 * bf16(snake2(W7 (*) a + b7)) + b1 ; a' = bf16(snake_n(x'))
static int run_ru(int dilation, int B, int T, int perf) {
  const int C = 128;
  std::mt19937 rng(99 + dilation);
  std::normal_distribution<float> nd(0.f, 1.f);
  const size_t n = (size_t)B * T * C;
  std::vector<float> a(n), x(n), w7((size_t)7 * C * C), w1((size_t)C * C), b7(C), b1(C), s2a(C), s2ib(C), sna(C), snib(C);
  if (perf) {   // timing only: a 1 Mi-element random block repeated (host RNG over 10^8 elements costs GPU-box minutes)
    const size_t blk = std::min<size_t>(n, (size_t)1 << 20);
    for (size_t i = 0; i < blk; ++i) { a[i] = bf16r(nd(rng)); x[i] = nd(rng); }
    for (size_t i = blk; i < n; ++i) { a[i] = a[i - blk]; x[i] = x[i - blk]; }
  } else {
    for (auto& v : a) v = bf16r(nd(rng));
    for (auto& v : x) v = nd(rng);
  }
  for (auto& v : w7) v = bf16r(nd(rng) / std::sqrt(7.f * C));
  for (auto& v : w1) v = bf16r(nd(rng) / std::sqrt((float)C));
  for (int i = 0; i < C; ++i) {
    b7[i] = nd(rng) * 0.1f; b1[i] = nd(rng) * 0.1f;
    s2a[i] = std::exp(nd(rng) * 0.3f); s2ib[i] = 1.f / (std::exp(nd(rng) * 0.3f) + 1e-9f);
    sna[i] = std::exp(nd(rng) * 0.3f); snib[i] = 1.f / (std::exp(nd(rng) * 0.3f) + 1e-9f);
  }
  std::vector<__nv_bfloat16> ab(n), w7b(w7.size()), w1b(w1.size());
  for (size_t i = 0; i < n; ++i) ab[i] = __float2bfloat16(a[i]);
  for (size_t i = 0; i < w7.size(); ++i) w7b[i] = __float2bfloat16(w7[i]);
  for (size_t i = 0; i < w1.size(); ++i) w1b[i] = __float2bfloat16(w1[i]);
  __nv_bfloat16 *da, *dw7, *dw1, *dact;
  __half *dx, *draw;                       // the fused kernel reads / writes the fp16 residual stream
  float *db7, *db1, *ds2a, *ds2ib, *dsna, *dsnib;
  std::vector<__half> xh(n);
  for (size_t i = 0; i < n; ++i) { xh[i] = __float2half(x[i]); x[i] = __half2float(xh[i]); }
  CK(cudaMalloc(&da, n * 2)); CK(cudaMalloc(&dw7, w7.size() * 2)); CK(cudaMalloc(&dw1, w1.size() * 2));
  CK(cudaMalloc(&dact, n * 2)); CK(cudaMalloc(&dx, n * 2)); CK(cudaMalloc(&draw, n * 2));
  CK(cudaMalloc(&db7, C * 4)); CK(cudaMalloc(&db1, C * 4)); CK(cudaMalloc(&ds2a, C * 4)); CK(cudaMalloc(&ds2ib, C * 4));
  CK(cudaMalloc(&dsna, C * 4)); CK(cudaMalloc(&dsnib, C * 4));
  CK(cudaMemcpy(da, ab.data(), n * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dw7, w7b.data(), w7.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dw1, w1b.data(), w1.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dx, xh.data(), n * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(db7, b7.data(), C * 4, cudaMemcpyHostToDevice)); CK(cudaMemcpy(db1, b1.data(), C * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(ds2a, s2a.data(), C * 4, cudaMemcpyHostToDevice)); CK(cudaMemcpy(ds2ib, s2ib.data(), C * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dsna, sna.data(), C * 4, cudaMemcpyHostToDevice)); CK(cudaMemcpy(dsnib, snib.data(), C * 4, cudaMemcpyHostToDevice));
  CK(cudaMemset(draw, 0xff, n * 2)); CK(cudaMemset(dact, 0xff, n * 2));
  RuArgs ra;
  ra.a = da; ra.x = dx; ra.w7 = dw7; ra.w1 = dw1; ra.bias7 = db7; ra.s2_a = ds2a; ra.s2_inv_b = ds2ib; ra.bias1 = db1;
  ra.out_raw = draw; ra.out_act = dact; ra.sn_a = dsna; ra.sn_inv_b = dsnib;
  ra.stream_f16 = 1;
  RuLaunch L;
  std::string err;
  if (!prepare_conv_ru(ra, B, T, dilation, L, err)) { printf("RU d=%d: prepare failed: %s\n", dilation, err.c_str()); return 3; }
  printf("RU d=%d B=%d T=%d: grid %d smem %zu RB %d nbox %d SA %d SB %d tiles %d\n", dilation, B, T, L.grid, L.smem, L.p.RB,
         L.p.nbox, L.p.SA, L.p.SB, L.p.total_tiles);
  fflush(stdout);
  CK(launch_conv_ru(L, 0));
  CK(cudaDeviceSynchronize());
  if (perf) {
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    for (int i = 0; i < 3; ++i) CK(launch_conv_ru(L, 0));
    CK(cudaEventRecord(e0));
    for (int i = 0; i < 10; ++i) CK(launch_conv_ru(L, 0));
    CK(cudaEventRecord(e1));
    CK(cudaDeviceSynchronize());
    float ms; CK(cudaEventElapsedTime(&ms, e0, e1)); ms /= 10;
    const double flops = 2.0 * B * T * C * C * 8.0, bytes = (double)n * (2 + 2 + 2 + 2);
    printf("PERF fused RU d=%d B=%d T=%d: %.3f ms  %.1f TFLOP/s  %.1f GB/s\n", dilation, B, T, ms, flops / ms * 1e-9, bytes / ms * 1e-6);
    return 0;
  }
  std::vector<float> raw(n);
  std::vector<__half> rawh(n);
  std::vector<__nv_bfloat16> act(n);
  CK(cudaMemcpy(rawh.data(), draw, n * 2, cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < n; ++i) raw[i] = __half2float(rawh[i]);
  CK(cudaMemcpy(act.data(), dact, n * 2, cudaMemcpyDeviceToHost));
  double max_err = 0, max_err_act = 0, max_ref = 0; size_t bad = 0, first_bad = (size_t)-1;
  std::vector<float> h((size_t)T * C);
  for (int b = 0; b < B; ++b) {
    for (int t = 0; t < T; ++t)
      for (int co = 0; co < C; ++co) {
        double s = b7[co];
        for (int k = 0; k < 7; ++k) {
          const int ti = t + (k - 3) * dilation;
          if (ti < 0 || ti >= T) continue;
          const float* ar = &a[((size_t)b * T + ti) * C];
          const float* wr = &w7[((size_t)k * C + co) * C];
          for (int ci = 0; ci < C; ++ci) s += (double)ar[ci] * wr[ci];
        }
        const double sn = std::sin(s * s2a[co]);
        h[(size_t)t * C + co] = bf16r((float)(s + s2ib[co] * sn * sn));
      }
    for (int t = 0; t < T; ++t)
      for (int co = 0; co < C; ++co) {
        double s = b1[co] + x[((size_t)b * T + t) * C + co];
        const float* wr = &w1[(size_t)co * C];
        for (int ci = 0; ci < C; ++ci) s += (double)h[(size_t)t * C + ci] * wr[ci];
        const size_t i = ((size_t)b * T + t) * C + co;
        double e = std::fabs((double)raw[i] - s);
        if (!(e <= 1e30)) e = 1e30;
        max_err = std::max(max_err, e); max_ref = std::max(max_ref, std::fabs(s));
        if (e > 3e-2) { if (!bad) first_bad = i; ++bad; }
        const double sn = std::sin(s * sna[co]);
        const double av = s + snib[co] * sn * sn;
        double ea = std::fabs((double)__bfloat162float(act[i]) - av) / (1.0 + std::fabs(av));
        if (!(ea <= 1e30)) ea = 1e30;
        max_err_act = std::max(max_err_act, ea);
      }
  }
  const bool ok = bad == 0 && max_err_act < 3e-2;
  printf("RESULT fused RU d=%d B=%d T=%d: %s max_err %.3e max_ref %.3e bad %zu/%zu act_rel_err %.3e\n", dilation, B, T,
         ok ? "PASS" : "FAIL", max_err, max_ref, bad, n, max_err_act);
  if (bad) printf("  first bad at b=%zu t=%zu c=%zu got %.5f\n", first_bad / ((size_t)T * C), (first_bad / C) % T, first_bad % C, raw[first_bad]);
  return ok ? 0 : 1;
}

int main(int argc, char** argv) {
  if (argc >= 5 && std::string(argv[1]) == "ru")
    return run_ru(atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), argc >= 6 ? atoi(argv[5]) : 0);
  if (argc >= 3 && std::string(argv[1]) == "perf") {
    int idx = atoi(argv[2]);
    if (idx < 0 || idx >= kNumPerf) return 4;
    const int ver = argc >= 4 ? atoi(argv[3]) : 2, epi = argc >= 5 ? atoi(argv[4]) : 0;
    if (ver < 2 || ver > 4) return 4;
    return run_perf(idx, ver, epi);
  }
  if (argc >= 2 && std::string(argv[1]) == "count") {
    printf("%d %d\n", kNumCases, kNumPerf);
    return 0;
  }
  if (argc < 3) {
    printf("usage: umma_probe <case 0..%d> <variant 3..6> | perf <0..%d> [2..4] [0..2] | ru <dil> <B> <T> [1] | count\n",
           kNumCases - 1, kNumPerf - 1);
    return 4;
  }
  int idx = atoi(argv[1]), variant = atoi(argv[2]);
  if (idx < 0 || idx >= kNumCases || variant < 3 || variant > 6) return 4;
  return run_case(idx, variant);
}
