// scores_probe.cu -- k_scores_tc2 checked against an f64 CPU evaluation of
//   score = sigmoid(sigmoid(qa + Kp + (q * H) Wp) W2 + b2) . kv + bk        (r4_scores_tc.cuh)
// on random inputs, then timed on an observation-pass-sized launch (sequence 0 unshared, sequence 1 shared, as in Slate)
// for several CTA shares of the shared sequence, and broken down per role and phase by the instrumented build (DBG).
// Build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -o tools/build/scores_probe tools/scores_probe.cu
// Run:   tools/build/scores_probe [rows=4096] [check_rows=300] [reps=20]
#include "../rl4rs_b200/csrc/r4_scores_tc.cuh"
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <vector>
#include <random>

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(1); } } while (0)
using namespace r4tc;

template <class T> T* up(const std::vector<T>& v) { T* d; CK(cudaMalloc(&d, v.size() * sizeof(T))); CK(cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice)); return d; }

int main(int argc, char** argv) {
  const int R = argc > 1 ? atoi(argv[1]) : 4096, RC = argc > 2 ? atoi(argv[2]) : 300, reps = argc > 3 ? atoi(argv[3]) : 20;
  int pct = 100;                                   // CTA share of the shared sequence (scores_grid_split)
  std::mt19937 g(7);
  std::normal_distribution<float> nd(0.f, 1.f);
  auto rnd = [&](size_t n, float sc) { std::vector<float> v(n); for (auto& x : v) x = sc * nd(g); return v; };
  // sequence 0: one cached (H, Kp) per row; sequence 1: one shared cached row
  std::vector<float> H0 = rnd((size_t)R * 64 * 128, 0.5f), K0 = rnd((size_t)R * 64 * 64, 0.7f);   // K: [row][key][j] on the host
  std::vector<float> H1 = rnd((size_t)64 * 128, 0.5f), K1 = rnd((size_t)64 * 64, 0.7f);
  std::vector<float> q = rnd((size_t)R * 128, 0.6f), qa0 = rnd((size_t)R * 64, 0.8f), qa1 = rnd((size_t)R * 64, 0.8f);
  std::vector<float> Wp[2] = {rnd(128 * 64, 0.25f), rnd(128 * 64, 0.25f)}, W2[2] = {rnd(64 * 16, 0.4f), rnd(64 * 16, 0.4f)};
  std::vector<float> b2[2] = {rnd(16, 0.3f), rnd(16, 0.3f)}, kv[2] = {rnd(16, 0.8f), rnd(16, 0.8f)};
  const float bk[2] = {0.1f, -0.2f};
  const int rt = (R + 127) / 128;
  ScoreTcParams p{};
  float* out[2];
  for (int i = 0; i < 2; ++i) {
    std::vector<uint8_t> img(S_IMG_BYTES);
    build_scores_image2(Wp[i].data(), W2[i].data(), img.data());
    ScoreTcSeq& s = p.s[i];
    const std::vector<float>& Kh = i ? K1 : K0;
    std::vector<float> Kq(Kh.size());               // device layout: [row][j / 4][key][j % 4] (kq_index)
    for (size_t n = 0; n < Kh.size() / (64 * 64); ++n)
      for (int key = 0; key < 64; ++key)
        for (int j = 0; j < 64; ++j) Kq[kq_index(n, 16, j / 4, 64, key) + j % 4] = Kh[(n * 64 + key) * 64 + j];
    s.qa = up(i ? qa1 : qa0); s.H = up(i ? H1 : H0); s.Kp = up(Kq); s.WpImg = up(img);
    s.Wqd = nullptr; s.b1 = nullptr; s.W2 = up(W2[i]); s.b2 = up(b2[i]); s.kv = up(kv[i]); s.bk = bk[i]; s.shared = i;
    CK(cudaMalloc(&out[i], (size_t)rt * 64 * 128 * 4)); CK(cudaMemset(out[i], 0xff, (size_t)rt * 64 * 128 * 4));
  }
  p.q = up(q); p.row0 = 0; p.div = 1;
  CK(cudaFuncSetAttribute(k_scores_tc2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, S2_SMEM_BYTES));
  CK(cudaFuncSetAttribute(k_scores_tc2<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, S2_SMEM_BYTES));
  auto launch = [&](int rows) {
    p.R = rows;
    for (int i = 0; i < 2; ++i) p.s[i].scoresT = out[i];
    const int ctas = std::min(2 * ((rows + 1) / 2), 148);
    k_scores_tc2<false><<<ctas, S2_THREADS, S2_SMEM_BYTES>>>(p, scores_grid_split(ctas, (rows + 1) / 2, 0, 1, pct));
  };
  // ---- correctness on RC rows (odd counts exercise the half-filled last tile), then on all R rows for the first / last rows
  int bad_total = 0;
  for (int rows : {RC, 1, R}) {
    launch(rows); CK(cudaGetLastError()); CK(cudaDeviceSynchronize());
    std::vector<float> o[2];
    for (int i = 0; i < 2; ++i) { o[i].resize((size_t)rt * 64 * 128); CK(cudaMemcpy(o[i].data(), out[i], o[i].size() * 4, cudaMemcpyDeviceToHost)); }
    double worst = 0;
    int bad = 0;
    const int step = rows > 600 ? rows / 300 : 1;
    for (int r = 0; r < rows; r += (r + step < rows || r == rows - 1) ? step : (rows - 1 - r)) {
      for (int i = 0; i < 2; ++i)
        for (int key = 0; key < 64; ++key) {
          const float* h = (i ? H1.data() : H0.data() + (size_t)r * 64 * 128) + key * 128;
          const float* kp = (i ? K1.data() : K0.data() + (size_t)r * 64 * 64) + key * 64;
          const float* qa = (i ? qa1 : qa0).data() + (size_t)r * 64;
          double z2[16];
          for (int n = 0; n < 16; ++n) z2[n] = b2[i][n];
          for (int j = 0; j < 64; ++j) {
            double a = (double)qa[j] + kp[j];
            for (int k = 0; k < 128; ++k) a += (double)q[(size_t)r * 128 + k] * h[k] * Wp[i][k * 64 + j];
            const double z1 = 1.0 / (1.0 + exp(-a));
            for (int n = 0; n < 16; ++n) z2[n] += z1 * W2[i][j * 16 + n];
          }
          double sc = bk[i];
          for (int n = 0; n < 16; ++n) sc += kv[i][n] / (1.0 + exp(-z2[n]));
          const size_t idx = ((size_t)(r >> 7) * 64 + key) * 128 + (r & 127);
          const double err = fabs((double)o[i][idx] - sc);
          if (!(err <= 2e-5 * (1.0 + fabs(sc)))) ++bad;
          if (err > worst || err != err) worst = err;
        }
      if (r == rows - 1) break;
    }
    printf("rows %5d: k_scores_tc2 worst |err| %.3g (%d bad)\n", rows, worst, bad);
    bad_total += bad;
  }
  printf("%s\n", bad_total ? "FAIL" : "PASS");
  // ---- timing
  cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  for (int cfg = 0; cfg < 6; ++cfg) {
    const int pcts[6] = {100, 85, 75, 65, 55, 45};
    pct = pcts[cfg];
    for (int i = 0; i < 3; ++i) launch(R);
    CK(cudaEventRecord(e0));
    for (int i = 0; i < reps; ++i) launch(R);
    CK(cudaEventRecord(e1)); CK(cudaEventSynchronize(e1));
    float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
    printf("timing k_scores_tc2 (shared-sequence share %3d%%): %.1f us per launch of %d rows (%d tiles per sequence)\n", pct, 1e3 * ms / reps, R, (R + 1) / 2);
  }
  pct = 100;
  // ---- where the time of a tile goes (CTA (0, 0) = unshared sequence, instrumented build of the kernel)
  {
    long long* dd; CK(cudaMalloc(&dd, 32 * 8)); CK(cudaMemset(dd, 0, 32 * 8));
    p.R = R;
    for (int i = 0; i < 2; ++i) p.s[i].scoresT = out[i];
    const int grid = std::min(2 * ((R + 1) / 2), 148), n0 = scores_grid_split(grid, (R + 1) / 2, 0, 1, 100);
    cudaEvent_t a0, a1; CK(cudaEventCreate(&a0)); CK(cudaEventCreate(&a1));
    k_scores_tc2<true><<<grid, S2_THREADS, S2_SMEM_BYTES>>>(p, n0, dd);
    CK(cudaEventRecord(a0));
    k_scores_tc2<true><<<grid, S2_THREADS, S2_SMEM_BYTES>>>(p, n0, dd);
    CK(cudaEventRecord(a1)); CK(cudaDeviceSynchronize());
    float ms; CK(cudaEventElapsedTime(&ms, a0, a1));
    long long hh[32]; CK(cudaMemcpy(hh, dd, sizeof(hh), cudaMemcpyDeviceToHost));
    const double nt = ((R + 1) / 2 + n0 - 1) / n0;
    printf("instrumented launch %.1f us, %.0f tiles per CTA; cycles per tile:\n", 1e3 * ms, nt);
    for (int sq = 0; sq < 2; ++sq) {
      const long long* h = hh + 16 * sq;
      printf(" sequence %d (%s)\n", sq, sq ? "shared rows, L2-resident" : "one cached row per feature row, from HBM");
      printf("  producer : bar.sync %.0f | wait A free %.0f | convert %.0f\n", h[0] / nt, h[1] / nt, h[2] / nt);
      printf("  mma      : wait A full %.0f | wait acc free %.0f | issue L1 %.0f | wait A2 full %.0f | issue L2 %.0f\n", h[4] / nt, h[5] / nt, h[6] / nt, h[7] / nt, h[8] / nt);
      printf("  epilogue : wait acc %.0f | z1 + pack %.0f | wait A2 free + st %.0f | tail %.0f\n", h[10] / nt, h[11] / nt, h[12] / nt, h[13] / nt);
    }
  }
  return bad_total ? 1 : 0;
}
