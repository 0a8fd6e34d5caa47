// Stand-alone check of the tcgen05 GEMM against the fp32 FFMA GEMM on random data (GPU box only):
//   build/selftest_gemm      -> prints max |tc - simt| per shape and a timing, exit code 0 if all close
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "common.cuh"

using namespace vsr;

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA %s: %s\n", #x, cudaGetErrorString(e)); exit(2); } } while (0)
#define VK(x) do { int r = (x); if (r != 0) { printf("VSR %s: %s\n", #x, vsr_last_error()); exit(3); } } while (0)

static float* dev_rand(size_t n, float scale, unsigned seed) {
  std::vector<float> h(n);
  srand(seed);
  for (size_t i = 0; i < n; ++i) h[i] = scale * ((rand() / (float)RAND_MAX) * 2.f - 1.f);
  float* d; CK(cudaMalloc(&d, n * 4)); CK(cudaMemcpy(d, h.data(), n * 4, cudaMemcpyHostToDevice));
  return d;
}
// f8 = false: fp16 hi + fp16 residual (f16x3); true: fp16 hi + e4m3 hi8 / lo8 (f16+f8x2)
static void make_pair(F16Pair* b, const float* f, int rows, int ld, int box, bool weight, bool f8) {
  CK(cudaMalloc(&b->hi, (size_t)rows * ld * 2));
  b->rows = rows; b->ld = ld; b->box_rows = box; b->n_valid = rows;
  VK(make_tmap_f16(b->map_hi, b->hi, rows, ld, ld, box));
  VK(make_tmap_f16(b->map32_hi, b->hi, rows, ld, ld, box, 32));
  if (!f8) {
    CK(cudaMalloc(&b->lo, (size_t)rows * ld * 2));
    VK(make_tmap_f16(b->map_lo, b->lo, rows, ld, ld, box));
    VK(make_tmap_f16(b->map32_lo, b->lo, rows, ld, ld, box, 32));
  } else {
    CK(cudaMalloc(&b->hi8, (size_t)rows * ld)); CK(cudaMalloc(&b->lo8, (size_t)rows * ld));
    VK(make_tmap_u8(b->map8_hi, b->hi8, rows, ld, ld, box));
    VK(make_tmap_u8(b->map8_lo, b->lo8, rows, ld, ld, box));
    VK(make_tmap_u8(b->map8_32_hi, b->hi8, rows, ld, ld, box, 32));
    VK(make_tmap_u8(b->map8_32_lo, b->lo8, rows, ld, ld, box, 32));
  }
  b->act_scale = (!weight && f8) ? ACT_SCALE_F8 : 1.f;
  if (weight) CK(cudaMalloc(&b->scale, 2 * sizeof(float)));     // weights: power-of-two scaled split
  VK(launch_split_pair(f, *b, (size_t)rows * ld, 0, weight));
  b->kb = getenv("VSRDEC_KB") && atoi(getenv("VSRDEC_KB")) == 32 ? 32 : 64;
}

static bool g_time = true;
static bool g_f8 = false;
static bool g_pair = false;      // CTA-pair kernel (needs M >= 1024; BN = pair tile width)
static bool g_vocab = false;     // vocabulary-head epilogue (logits + chunk records; the logits are checked)
static int run_case(int M, int N, int nseg, const int* ks, bool extras, int BN, float wscale = 0.05f) {
  const int Mp = (M + 127) / 128 * 128;
  int K = 0; for (int s = 0; s < nseg; ++s) K += ks[s];
  float* W = dev_rand((size_t)N * K, wscale, 1);
  F16Pair wb{}; make_pair(&wb, W, N, K, g_pair ? 128 : BN, true, g_f8);
  if (g_pair) VK(make_pair_maps(&wb, BN / 2));
  GemmArgs g{};
  g.nseg = nseg;
  F16Pair ab[3];
  for (int s = 0; s < nseg; ++s) {
    float* A = dev_rand((size_t)Mp * ks[s], 1.0f, 10 + s);
    ab[s] = F16Pair{};
    make_pair(&ab[s], A, Mp, ks[s], 128, false, g_f8);
    g.seg[s] = {A, ks[s], ks[s], ks[s], &ab[s]};
  }
  g.w = W; g.ldw = K; g.wb = &wb; g.f8 = g_f8; g.allow_pair = g_pair;
  float *bias = nullptr, *radd = nullptr, *cadd = nullptr;
  if (extras) {
    bias = dev_rand(N, 1.f, 5); radd = dev_rand((size_t)(Mp / 5 + 1) * N, 1.f, 6); cadd = dev_rand((size_t)Mp * (N + 64), 1.f, 7);
    g.bias = bias; g.rowadd = radd; g.ld_rowadd = N; g.row_div = 5; g.rowadd_mul = 1; g.cadd = cadd + 64; g.ld_cadd = N + 64;
  }
  float* vpart = nullptr;
  if (g_vocab) {
    bias = dev_rand(N, 1.f, 5); g.bias = bias;
    CK(cudaMalloc(&vpart, (size_t)Mp * (N / 16) * 2 * sizeof(float)));
  }
  float *C1, *C2;
  CK(cudaMalloc(&C1, (size_t)Mp * N * 4)); CK(cudaMalloc(&C2, (size_t)Mp * N * 4));
  CK(cudaMemset(C1, 0, (size_t)Mp * N * 4)); CK(cudaMemset(C2, 0, (size_t)Mp * N * 4));
  g.M = M; g.N = N; g.ldc = N;
  g.c = C1; VK(launch_gemm_simt(g, 0));
  if (g_vocab) { g.cell.mode = 3; g.cell.vocab_part = vpart; }
  g.c = C2; VK(launch_gemm_tc(g, nullptr, 0));
  CK(cudaDeviceSynchronize());
  std::vector<float> h1((size_t)M * N), h2((size_t)M * N);
  CK(cudaMemcpy(h1.data(), C1, h1.size() * 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(h2.data(), C2, h2.size() * 4, cudaMemcpyDeviceToHost));
  double maxerr = 0, maxref = 0;
  for (size_t i = 0; i < h1.size(); ++i) { maxerr = fmax(maxerr, fabs((double)h1[i] - h2[i])); maxref = fmax(maxref, fabs((double)h1[i])); }
  if (!g_time) {
    const bool ok1 = maxerr <= (g_f8 ? 4e-3 : 2e-4) * (wscale / 0.05) * fmax(1.0, maxref);
    printf("%s M=%d N=%d K=%d BN=%d maxerr=%.3e %s\n", g_pair ? "pair" : "1cta", M, N, K, BN, maxerr, ok1 ? "OK" : "MISMATCH");
    return ok1 ? 0 : 1;
  }
  // timing of both
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  float ms_tc = 0, ms_simt = 0;
  for (int rep = 0; rep < 2; ++rep) {
    cudaEventRecord(e0); for (int i = 0; i < 10; ++i) { g.c = C2; VK(launch_gemm_tc(g, nullptr, 0)); } cudaEventRecord(e1); CK(cudaEventSynchronize(e1));
    cudaEventElapsedTime(&ms_tc, e0, e1);
  }
#ifdef VSR_DBG_CLK
  if (g_pair) {
    char label[96];
    snprintf(label, sizeof(label), "M=%d N=%d K=%d BN=%d%s", M, N, K, BN, g_vocab ? " vocab" : "");
    tc_dbg_clk_report(label);
  }
#endif
  cudaEventRecord(e0); for (int i = 0; i < 3; ++i) { g.c = C1; VK(launch_gemm_simt(g, 0)); } cudaEventRecord(e1); CK(cudaEventSynchronize(e1));
  cudaEventElapsedTime(&ms_simt, e0, e1);
  const double flops = 2.0 * M * N * K;
  // f16x3 carries ~22 bits; f16+f8x2 ~2^-15 per product term (measured ~1e-5 of the output scale)
  const bool ok = maxerr <= (g_f8 ? 4e-3 : 2e-4) * (wscale / 0.05) * fmax(1.0, maxref);
  printf("%s M=%4d N=%5d K=%4d segs=%d extras=%d BN=%d : max|tc-simt|=%.3e (max|ref|=%.2f) %s | tc %.1f us (%.1f TF/s algorithmic) simt %.1f us\n",
         g_pair ? (g_f8 ? "pair f16+f8x2" : "pair f16x3   ") : (g_f8 ? "f16+f8x2" : "f16x3   "), M, N, K, nseg, (int)extras, BN, maxerr, maxref, ok ? "OK" : "MISMATCH", ms_tc * 100, flops / (ms_tc * 1e-4) / 1e12,
         ms_simt * 1000 / 3);
  fflush(stdout);
  return ok ? 0 : 1;
}

int main(int argc, char** argv) {
  int bad = 0;
  if (argc > 1 && strcmp(argv[1], "prof") == 0) {   // the per-step shapes once each (for ncu)
    const int ka[] = {1024, 1024, 1024}, kb[] = {1024}, kd[] = {2048, 1024};
    g_time = false;
    run_case(500, 6144, 3, ka, true, 128);    // A
    run_case(500, 5632, 1, kb, true, 128);    // B2
    run_case(500, 4096, 2, kd, true, 128);    // D
    run_case(500, 10240, 1, kb, true, 128);   // E
    run_case(500, 6144, 3, ka, true, 256);    // A, BN=256
    return 0;
  }
  const int k1[] = {64}, k2[] = {1024}, k3[] = {1024, 1024, 1024}, k4[] = {2048, 1024}, k5[] = {64, 64, 64};
  if (argc > 1 && strcmp(argv[1], "epi") == 0) {   // CTA-pair kernel at the 1000-caption step shapes (B-, D-, vocabulary-like):
    g_pair = true; g_f8 = true;                     // timing; with -DVSR_DBG_CLK also the per-tile clock64 phases of the last launch
    const int k6[] = {2048, 1024, 1024};
    bad += run_case(5000, 4096, 1, k2, false, 256);
    bad += run_case(5000, 4096, 3, k6, false, 256);
    g_vocab = true;
    bad += run_case(5000, 10368, 1, k2, false, 192);
    return bad ? 1 : 0;
  }
  if (argc > 1 && strcmp(argv[1], "quick") == 0) {   // one launch per kernel variant, no timing loops (compute-sanitizer)
    g_time = false;
    for (int pass = 0; pass < 2; ++pass) {
      g_f8 = pass == 1;
      g_pair = false;
      bad += run_case(300, 512, 1, k2, true, 128);
      bad += run_case(300, 768, 3, k5, true, 256);
      g_pair = true;
      bad += run_case(1100, 512, 1, k2, true, 256);
      bad += run_case(1100, 768, 3, k5, true, 192);
    }
    printf("%s\n", bad ? "SELFTEST FAILED" : "SELFTEST PASSED");
    return bad ? 1 : 0;
  }
  const int bns[2] = {256, 128};
  for (int pass = 0; pass < 4; ++pass) {
    const int BN = bns[pass & 1];
    g_f8 = pass >= 2;
    bad += run_case(128, 256, 1, k1, false, BN);
    bad += run_case(100, 256, 3, k5, true, BN);
    bad += run_case(500, 512, 1, k2, false, BN);
    bad += run_case(500, 2560, 1, k2, true, BN);
    bad += run_case(500, 6144, 3, k3, true, BN);
    bad += run_case(500, 4096, 2, k4, true, BN);
    bad += run_case(500, 10240, 1, k2, true, BN);
    bad += run_case(100, 6144, 3, k3, true, BN);
    bad += run_case(500, 4096, 2, k4, false, BN, 5e-5f);    // tiny weights: the scaled split keeps ~22 bits
    bad += run_case(500, 4096, 2, k4, false, BN, 50.f);     // large weights
  }
  g_pair = true;
  for (int pass = 0; pass < 2; ++pass) {
    g_f8 = pass == 1;
    bad += run_case(2000, 4096, 2, k4, true, 256);
    bad += run_case(2000, 2560, 1, k2, true, 256);
    bad += run_case(1900, 6144, 3, k3, true, 192);      // odd number of 128-row tiles: the last pair is half empty
    bad += run_case(1024, 512, 1, k2, false, 256);
    bad += run_case(4000, 4096, 2, k4, true, 256);
  }
  printf("%s\n", bad ? "SELFTEST FAILED" : "SELFTEST PASSED");
  return bad ? 1 : 0;
}
