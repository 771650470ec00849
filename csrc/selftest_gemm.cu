// Standalone GPU self-test + micro-benchmark of otb_gemm_bf16 through the public C ABI.
// Not part of the product path: a developer tool for quick timings on a B200.  The parity tests of record are
// tests/test_gemm_gpu.py (every kernel family, layout and epilogue class against an fp64 reference with a derived
// tolerance).  Reference here = fp64 accumulation on the host over the bf16-rounded inputs, with fixed tolerances.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../include/otter_b200.h"

#define CK(x)                                                                      \
  do {                                                                             \
    cudaError_t e = (x);                                                           \
    if (e != cudaSuccess) {                                                        \
      printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); \
      exit(2);                                                                     \
    }                                                                              \
  } while (0)

static uint32_t rng_state = 12345;
static float frand() {
  rng_state = rng_state * 1664525u + 1013904223u;
  return ((rng_state >> 8) & 0xFFFF) / 65536.0f - 0.5f;
}
static float bf(float x) { return __bfloat162float(__float2bfloat16(x)); }
static double gelu(double x) { return 0.5 * x * (1.0 + erf(x * 0.7071067811865476)); }
static double gelu_grad(double x) {
  return 0.5 * (1.0 + erf(x * 0.7071067811865476)) + x * 0.3989422804014327 * exp(-0.5 * x * x);
}

struct Case {
  int M, N, K, a_mn, b_mn, mode;  // mode: 0 plain bf16 out, 1 bias+gelu+aux_out, 2 gate(tanh)+residual, 3 dgelu aux_in,
                                  //       4 fp32 out accumulate, 5 quick-gelu + bias, 6 fp32 out (no accumulate), 7 bias + residual
};

static int run_case(const Case& c) {
  const int M = c.M, N = c.N, K = c.K;
  // logical A[m][k], B[n][k]
  std::vector<float> A((size_t)M * K), B((size_t)N * K);
  for (auto& v : A) v = bf(frand());
  for (auto& v : B) v = bf(frand());
  // physical layouts
  std::vector<__nv_bfloat16> hA((size_t)M * K), hB((size_t)N * K);
  for (int m = 0; m < M; ++m)
    for (int k = 0; k < K; ++k) {
      size_t idx = c.a_mn ? (size_t)k * M + m : (size_t)m * K + k;
      hA[idx] = __float2bfloat16(A[(size_t)m * K + k]);
    }
  for (int n = 0; n < N; ++n)
    for (int k = 0; k < K; ++k) {
      size_t idx = c.b_mn ? (size_t)k * N + n : (size_t)n * K + k;
      hB[idx] = __float2bfloat16(B[(size_t)n * K + k]);
    }
  std::vector<float> bias(N), resid((size_t)M * N), auxin((size_t)M * N), out0((size_t)M * N);
  for (auto& v : bias) v = frand();
  for (auto& v : resid) v = bf(frand());
  for (auto& v : auxin) v = bf(4.f * frand());
  for (auto& v : out0) v = frand();
  std::vector<__nv_bfloat16> hres((size_t)M * N), haux((size_t)M * N);
  for (size_t i = 0; i < hres.size(); ++i) {
    hres[i] = __float2bfloat16(resid[i]);
    haux[i] = __float2bfloat16(auxin[i]);
  }
  const float gate = 0.5f;

  __nv_bfloat16 *dA, *dB, *dres, *dauxin, *dauxout, *dout_bf;
  float *dbias, *dgate, *dout_f;
  CK(cudaMalloc(&dA, hA.size() * 2));
  CK(cudaMalloc(&dB, hB.size() * 2));
  CK(cudaMalloc(&dres, hres.size() * 2));
  CK(cudaMalloc(&dauxin, haux.size() * 2));
  CK(cudaMalloc(&dauxout, (size_t)M * N * 2));
  CK(cudaMalloc(&dout_bf, (size_t)M * N * 2));
  CK(cudaMalloc(&dout_f, (size_t)M * N * 4));
  CK(cudaMalloc(&dbias, N * 4));
  CK(cudaMalloc(&dgate, 4));
  CK(cudaMemcpy(dA, hA.data(), hA.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dB, hB.data(), hB.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dres, hres.data(), hres.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dauxin, haux.data(), haux.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dbias, bias.data(), N * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dgate, &gate, 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dout_f, out0.data(), (size_t)M * N * 4, cudaMemcpyHostToDevice));
  CK(cudaMemset(dout_bf, 0xFF, (size_t)M * N * 2));
  CK(cudaMemset(dauxout, 0xFF, (size_t)M * N * 2));

  otb_gemm_epilogue e;
  memset(&e, 0, sizeof(e));
  e.alpha = 1.0f;
  e.ld_out = e.ld_aux_in = e.ld_aux_out = e.ld_res = N;
  e.out = dout_bf;
  switch (c.mode) {
    case 1: e.bias = dbias; e.act = 1; e.aux_out = dauxout; break;
    case 2: e.scale_ptr = dgate; e.scale_tanh = 1; e.residual = dres; break;
    case 3: e.aux_in = dauxin; e.alpha = 0.25f; break;
    case 4: e.out = dout_f; e.out_fp32 = 1; e.accumulate = 1; break;
    case 5: e.bias = dbias; e.act = 2; break;
    case 6: e.out = dout_f; e.out_fp32 = 1; break;
    case 7: e.bias = dbias; e.residual = dres; break;
    default: break;
  }
  int rc = otb_gemm_bf16(dA, c.a_mn, c.a_mn ? M : K, dB, c.b_mn, c.b_mn ? N : K, M, N, K, &e, nullptr);
  if (rc) {
    printf("  otb_gemm_bf16 rc=%d: %s\n", rc, otb_last_error());
    return 1;
  }
  cudaError_t err = cudaDeviceSynchronize();
  if (err != cudaSuccess) {
    printf("  kernel failed: %s\n", cudaGetErrorString(err));
    exit(3);
  }
  std::vector<__nv_bfloat16> gout((size_t)M * N), gaux((size_t)M * N);
  std::vector<float> goutf((size_t)M * N);
  CK(cudaMemcpy(gout.data(), dout_bf, gout.size() * 2, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(gaux.data(), dauxout, gaux.size() * 2, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(goutf.data(), dout_f, goutf.size() * 4, cudaMemcpyDeviceToHost));

  double max_err = 0, max_ref = 0, max_aux_err = 0;
  size_t bad = 0;
  // Big problems are verified on a subset of rows (all columns): the first / last rows, every row next to a 128-row
  // tile boundary, and a stride of the rest — the host reference is a scalar triple loop.
  const bool sample_rows = (double)M * N * K > 3e9;
  for (int m = 0; m < M; ++m) {
    if (sample_rows) {
      const int r = m % 128;
      if (!(m < 4 || m >= M - 4 || r < 2 || r >= 126 || m % 61 == 0)) continue;
    }
    for (int n = 0; n < N; ++n) {
      double acc = 0;
      const float* a = &A[(size_t)m * K];
      const float* b = &B[(size_t)n * K];
      for (int k = 0; k < K; ++k) acc += (double)a[k] * b[k];
      double v = acc, pre = acc;
      size_t i = (size_t)m * N + n;
      switch (c.mode) {
        case 1: pre = acc + bias[n]; v = gelu(pre); break;
        case 2: v = acc * tanh((double)gate) + resid[i]; break;
        case 3: v = acc * gelu_grad(auxin[i]) * 0.25; break;
        case 4: v = acc + out0[i]; break;
        case 5: { double z = acc + bias[n]; v = z / (1.0 + exp(-1.702 * z)); } break;
        case 7: v = acc + bias[n] + resid[i]; break;
        default: break;
      }
      double got = (c.mode == 4 || c.mode == 6) ? (double)goutf[i] : (double)__bfloat162float(gout[i]);
      double tol = (c.mode == 4 || c.mode == 6) ? 1e-3 : (fabs(v) * 8e-3 + 2e-3);
      double err = fabs(got - v);
      if (!(err <= tol)) {
        if (bad < 5) printf("    mismatch m=%d n=%d got=%f ref=%f\n", m, n, got, v);
        ++bad;
      }
      if (err > max_err) max_err = err;
      if (fabs(v) > max_ref) max_ref = fabs(v);
      if (c.mode == 1) {
        double ae = fabs((double)__bfloat162float(gaux[i]) - pre);
        if (ae > max_aux_err) max_aux_err = ae;
        if (!(ae <= fabs(pre) * 8e-3 + 2e-3)) ++bad;
      }
    }
  }
  printf("  M=%d N=%d K=%d a_mn=%d b_mn=%d mode=%d : max_err=%.3e (max|ref|=%.3f aux_err=%.3e) bad=%zu %s\n", M, N, K,
         c.a_mn, c.b_mn, c.mode, max_err, max_ref, max_aux_err, bad, bad ? "FAIL" : "ok");
  cudaFree(dA); cudaFree(dB); cudaFree(dres); cudaFree(dauxin); cudaFree(dauxout); cudaFree(dout_bf);
  cudaFree(dout_f); cudaFree(dbias); cudaFree(dgate);
  return bad ? 1 : 0;
}

static void bench(int M, int N, int K, int a_mn, int b_mn, int mode, const char* name) {
  __nv_bfloat16 *dA, *dB, *dO, *dAux;
  float* dOf;
  CK(cudaMalloc(&dA, (size_t)M * K * 2));
  CK(cudaMalloc(&dB, (size_t)N * K * 2));
  CK(cudaMalloc(&dO, (size_t)M * N * 2));
  CK(cudaMalloc(&dAux, (size_t)M * N * 2));
  CK(cudaMalloc(&dOf, (size_t)M * N * 4));
  CK(cudaMemset(dA, 0x11, (size_t)M * K * 2));
  CK(cudaMemset(dB, 0x11, (size_t)N * K * 2));
  CK(cudaMemset(dOf, 0, (size_t)M * N * 4));
  otb_gemm_epilogue e;
  memset(&e, 0, sizeof(e));
  e.alpha = 1.0f;
  e.ld_out = e.ld_aux_in = e.ld_aux_out = e.ld_res = N;
  e.out = dO;
  float* dBias;
  CK(cudaMalloc(&dBias, (size_t)N * 4));
  CK(cudaMemset(dBias, 0, (size_t)N * 4));
  if (mode == 1) { e.act = 1; e.aux_out = dAux; }
  if (mode == 3) { e.aux_in = dAux; }
  if (mode == 4) { e.out = dOf; e.out_fp32 = 1; }
  if (mode == 5) { e.bias = dBias; e.act = 2; }
  if (mode == 6) { e.out = dOf; e.out_fp32 = 1; e.accumulate = 1; }
  if (mode == 7) { e.bias = dBias; e.residual = dAux; }
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  for (int i = 0; i < 3; ++i) otb_gemm_bf16(dA, a_mn, a_mn ? M : K, dB, b_mn, b_mn ? N : K, M, N, K, &e, nullptr);
  CK(cudaDeviceSynchronize());
  const int iters = 20;
  CK(cudaEventRecord(e0));
  for (int i = 0; i < iters; ++i) otb_gemm_bf16(dA, a_mn, a_mn ? M : K, dB, b_mn, b_mn ? N : K, M, N, K, &e, nullptr);
  CK(cudaEventRecord(e1));
  CK(cudaEventSynchronize(e1));
  float ms;
  CK(cudaEventElapsedTime(&ms, e0, e1));
  ms /= iters;
  printf("  bench %-28s M=%5d N=%5d K=%5d a_mn=%d b_mn=%d mode=%d : %.3f ms  %.1f TFLOP/s\n", name, M, N, K, a_mn, b_mn,
         mode, ms, 2.0 * M * N * K / ms / 1e9);
  cudaFree(dA); cudaFree(dB); cudaFree(dO); cudaFree(dAux); cudaFree(dOf); cudaFree(dBias);
}

int main(int argc, char** argv) {
  int fails = 0;
  printf("otb gemm selftest: version %d arch %d\n", otb_version(), otb_compiled_arch());
  const Case cases[] = {
      {128, 256, 64, 0, 0, 0},   {128, 128, 64, 0, 0, 0},    {256, 512, 256, 0, 0, 0},  {200, 136, 200, 0, 0, 0},
      {1000, 1024, 512, 0, 0, 1}, {512, 4096, 512, 0, 0, 2},  {512, 2048, 256, 0, 0, 3}, {384, 1024, 320, 0, 0, 5},
      {128, 256, 64, 0, 1, 0},   {256, 512, 256, 0, 1, 0},   {200, 136, 200, 0, 1, 0},  {1000, 1024, 512, 0, 1, 3},
      {128, 256, 64, 1, 1, 0},   {256, 512, 256, 1, 1, 4},   {1024, 512, 1000, 1, 1, 4}, {2048, 4096, 300, 1, 1, 0},
      {4096, 4096, 1024, 0, 0, 0},
      // CTA-pair multicast path (>= 148 tiles): odd row-tile count, all three layouts, heavy epilogues
      {2056, 4096, 1024, 0, 0, 5}, {2048, 16384, 512, 0, 1, 3}, {16384, 4096, 256, 1, 1, 4}, {2200, 4096, 320, 0, 0, 2},
      {2048, 16384, 320, 0, 0, 1}, {4096, 2560, 192, 1, 1, 0},
      // output-path coverage for the TMA-store epilogue: fp32 store with ragged M/N, bias + residual, N tail inside a box
      {200, 136, 200, 1, 1, 6},  {1000, 1032, 128, 0, 0, 7},  {2056, 1024, 256, 0, 0, 7}, {520, 4136, 128, 0, 1, 6},
      {300, 40, 64, 0, 0, 7},    {2056, 3072, 128, 0, 0, 5},
  };
  bool no_cases = false;
  for (int i = 1; i < argc; ++i) no_cases |= (strcmp(argv[i], "--no-cases") == 0);   // profiling runs: only --shape / --bench
  if (!no_cases)
    for (const Case& c : cases) fails += run_case(c);
  bool do_bench = false;
  for (int i = 1; i < argc; ++i) do_bench |= (strcmp(argv[i], "--bench") == 0);
  if (do_bench) {
    bench(2048, 16384, 4096, 0, 0, 1, "gated ffn up (gelu+aux)");
    bench(2048, 4096, 16384, 0, 0, 0, "gated ffn down");
    bench(2048, 16384, 4096, 0, 1, 0, "dgrad via MN-major W");
    bench(16384, 4096, 2048, 1, 1, 4, "wgrad fp32 out");
    bench(2056, 4096, 1024, 0, 0, 0, "clip fc1");
    bench(2048, 512, 4096, 0, 0, 0, "to_q");
    bench(8192, 8192, 8192, 0, 0, 0, "square 8k");
    // CLIP tower shapes (M = 8 x 257) with their real epilogues, and K = 64 problems = epilogue cost alone
    bench(2056, 3072, 1024, 0, 0, 5, "clip qkv (bias)");
    bench(2056, 4096, 1024, 0, 0, 5, "clip fc1 (bias+qgelu)");
    bench(2056, 1024, 4096, 0, 0, 7, "clip fc2 (bias+res)");
    bench(2056, 1024, 1024, 0, 0, 7, "clip out_proj (bias+res)");
    bench(2048, 16384, 64, 0, 0, 0, "epilogue only: plain");
    bench(2048, 16384, 64, 0, 0, 1, "epilogue only: gelu+aux");
    bench(2048, 16384, 64, 0, 0, 3, "epilogue only: dgelu");
    bench(2048, 16384, 64, 0, 0, 7, "epilogue only: bias+res");
    bench(16384, 4096, 64, 1, 1, 4, "epilogue only: fp32 store");
    bench(16384, 4096, 64, 1, 1, 6, "epilogue only: fp32 accum");
  }
  // --shape M N K a_mn b_mn mode   (repeatable): time one custom problem
  for (int i = 1; i + 6 < argc + 0; ++i)
    if (strcmp(argv[i], "--shape") == 0)
      bench(atoi(argv[i + 1]), atoi(argv[i + 2]), atoi(argv[i + 3]), atoi(argv[i + 4]), atoi(argv[i + 5]),
            atoi(argv[i + 6]), "custom");
  printf("selftest %s (%d failing cases), launches=%lld\n", fails ? "FAILED" : "PASSED", fails, otb_launch_count());
  return fails ? 1 : 0;
}
