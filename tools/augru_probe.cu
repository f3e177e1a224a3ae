// augru_probe.cu -- standalone check + timing of the AUGRU pair kernels (default: k_augru_pair2, -DPP: k_augru_pp)
// against a CPU (f64) recurrence.
// Build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -o tools/build/augru_probe tools/augru_probe.cu
#include "../rl4rs_b200/csrc/r4_augru_pp.cuh"
#ifdef PP
#define KERNEL k_augru_pp
#define KSMEM PP_SMEM_BYTES
#else
#define KERNEL k_augru_pair2
#define KSMEM P_SMEM_BYTES
#define CLUSTER 2
#endif
#define KTHREADS NTHREADS
#define GRIDX(t) (2 * (t))
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <vector>
#include <algorithm>
using namespace r4tc;
#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(1); } } while (0)

static float frand(float a) { return a * ((rand() % 20001) - 10000) / 10000.f; }

void build_image(const std::vector<float>& Wg, const std::vector<float>& Wc, std::vector<uint8_t>& img) {
  img.assign(W_IMAGE_BYTES, 0);
  build_pair_image(Wg.data(), Wc.data(), img.data());
}

int main(int argc, char** argv) {
  int R = argc > 1 ? atoi(argv[1]) : 300;
  int div = argc > 2 ? atoi(argv[2]) : 1;
  int timing_tiles = argc > 3 ? atoi(argv[3]) : 148;
  srand(3);
  int ncache = (R + div - 1) / div;
  std::vector<float> Wg(256 * 512), Wc(256 * 256);
  for (auto& w : Wg) w = frand(0.17f);
  for (auto& w : Wc) w = frand(0.17f);
  std::vector<float> X((size_t)ncache * 64 * 768), sc((size_t)R * 64);
  for (size_t i = 0; i < X.size(); ++i) X[i] = frand(1.0f) + ((i % 768) < 512 ? 1.0f : 0.f);
  for (auto& s : sc) s = 0.5f + frand(0.5f);
  int ctiles = (ncache + TM - 1) / TM, rtiles = (R + TM - 1) / TM;
  std::vector<float> XT((size_t)ctiles * 64 * 768 * TM, 0.f), sT((size_t)rtiles * 64 * TM, 0.f);
  for (int c = 0; c < ncache; ++c) for (int t = 0; t < 64; ++t) for (int col = 0; col < 768; ++col)
    XT[(((size_t)(c / TM) * 64 + t) * 768 + (col & ~3)) * TM + (c % TM) * 4 + (col & 3)] = X[((size_t)c * 64 + t) * 768 + col];   // quad layout (r4_gemm_tc.cuh: xt_index)
  for (int r = 0; r < R; ++r) for (int t = 0; t < 64; ++t) sT[((size_t)(r / TM) * 64 + t) * TM + r % TM] = sc[(size_t)r * 64 + t];
  std::vector<uint8_t> img; build_image(Wg, Wc, img);
  // CPU reference (f64)
  std::vector<double> href((size_t)R * 256, 0.0);
  for (int r = 0; r < R; ++r) {
    int c = r / div;
    std::vector<double> h(256, 0.0), g(512), rh(256), cc(256);
    for (int t = 0; t < 64; ++t) {
      const float* x = &X[((size_t)c * 64 + t) * 768];
      for (int n = 0; n < 512; ++n) { double s = x[n]; for (int k = 0; k < 256; ++k) s += h[k] * Wg[(size_t)k * 512 + n]; g[n] = 1.0 / (1.0 + exp(-s)); }
      for (int k = 0; k < 256; ++k) rh[k] = g[k] * h[k];
      for (int n = 0; n < 256; ++n) { double s = x[512 + n]; for (int k = 0; k < 256; ++k) s += rh[k] * Wc[(size_t)k * 256 + n]; cc[n] = tanh(s); }
      double om = 1.0 - sc[(size_t)r * 64 + t];
      for (int n = 0; n < 256; ++n) { double u = om * g[256 + n]; h[n] = u * h[n] + (1 - u) * cc[n]; }
    }
    for (int n = 0; n < 256; ++n) href[(size_t)r * 256 + n] = h[n];
  }
  float *dXT, *dsT, *dout; uint8_t* dimg;
  CK(cudaMalloc(&dXT, XT.size() * 4)); CK(cudaMalloc(&dsT, sT.size() * 4)); CK(cudaMalloc(&dout, (size_t)R * 256 * 4)); CK(cudaMalloc(&dimg, img.size()));
  CK(cudaMemcpy(dXT, XT.data(), XT.size() * 4, cudaMemcpyHostToDevice)); CK(cudaMemcpy(dsT, sT.data(), sT.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dimg, img.data(), img.size(), cudaMemcpyHostToDevice));
  CK(cudaMemset(dout, 0, (size_t)R * 256 * 4));
  CK(cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, KSMEM));
  CUtensorMap tmap;
  { int trc = make_pair_tensor_map(dimg, &tmap); if (trc) { printf("make_pair_tensor_map failed: %d\n", trc); return 1; } }
#ifdef CLUSTER
#define LAUNCH(grid, prm) do { AugruPairParams pp_; pp_.b = (prm); pp_.tmap[0] = tmap; pp_.tmap[1] = tmap; \
    cudaLaunchConfig_t lc_ = {}; dim3 g_ = (grid); g_.x = (g_.x + CLUSTER - 1) / CLUSTER * CLUSTER; lc_.gridDim = g_; lc_.blockDim = dim3(KTHREADS); \
    lc_.dynamicSmemBytes = KSMEM; cudaLaunchAttribute at_[1]; at_[0].id = cudaLaunchAttributeClusterDimension; \
    at_[0].val.clusterDim.x = CLUSTER; at_[0].val.clusterDim.y = 1; at_[0].val.clusterDim.z = 1; lc_.attrs = at_; lc_.numAttrs = 1; \
    CK(cudaLaunchKernelEx(&lc_, KERNEL, pp_)); } while (0)
#else
#define LAUNCH(grid, prm) do { AugruPairParams pp_; pp_.b = (prm); pp_.tmap[0] = tmap; pp_.tmap[1] = tmap; KERNEL<<<grid, KTHREADS, KSMEM>>>(pp_); } while (0)
#endif
  AugruTcParams p{};
  p.s[0] = {dXT, dimg, dsT, dout, 0}; p.s[1] = p.s[0];
#ifdef PP
  float* dout1; CK(cudaMalloc(&dout1, (size_t)R * 256 * 4)); CK(cudaMemset(dout1, 0, (size_t)R * 256 * 4));
  p.s[1].out = dout1;          // the second recurrence of the pair: same inputs, its own output
#endif
  p.R = R; p.row0 = 0; p.div = div; p.out_ld = 256;
  LAUNCH(dim3(GRIDX(rtiles), 1), p);
  CK(cudaGetLastError()); CK(cudaDeviceSynchronize());
  std::vector<float> hout((size_t)R * 256);
  CK(cudaMemcpy(hout.data(), dout, hout.size() * 4, cudaMemcpyDeviceToHost));
  double rms = 0, worst = 0; for (auto v : href) rms += v * v; rms = sqrt(rms / href.size());
  int wi = 0;
  for (size_t i = 0; i < href.size(); ++i) { double e = fabs(hout[i] - href[i]); if (e > worst) { worst = e; wi = (int)i; } }
  printf("R=%d div=%d: rms(h)=%.4f  max abs err %.3g (%.3g of rms) at row %d col %d: got %f ref %f -> %s\n", R, div, rms, worst,
         worst / rms, wi / 256, wi % 256, hout[wi], href[wi], worst / rms < 1e-4 ? "PASS" : "FAIL");
#ifdef PP
  {
    std::vector<float> h1((size_t)R * 256);
    CK(cudaMemcpy(h1.data(), dout1, h1.size() * 4, cudaMemcpyDeviceToHost));
    double w1 = 0; for (size_t i = 0; i < href.size(); ++i) w1 = std::max(w1, (double)fabs(h1[i] - href[i]));
    printf("   second recurrence: max abs err %.3g (%.3g of rms) -> %s; bitwise equal to the first: %s\n", w1, w1 / rms,
           w1 / rms < 1e-4 ? "PASS" : "FAIL", memcmp(h1.data(), hout.data(), h1.size() * 4) == 0 ? "yes" : "NO");
  }
#endif
  // timing: `timing_tiles` tiles sharing cache row tile 0 (div large -> all rows read cached sequence 0.. via shared)
  if (timing_tiles > 0) {
    int RT = timing_tiles * TM;
    float *dsT2, *dout2;
    CK(cudaMalloc(&dsT2, (size_t)timing_tiles * 64 * TM * 4)); CK(cudaMalloc(&dout2, (size_t)RT * 256 * 4));
    CK(cudaMemset(dsT2, 0, (size_t)timing_tiles * 64 * TM * 4));
    AugruTcParams q = p; q.s[0].scoresT = dsT2; q.s[0].out = dout2; q.s[0].shared = 1; q.R = RT;
    if (argc > 4 && atoi(argv[4])) {          // every tile streams its own inputs from HBM (as in the product)
      float* dXTbig; size_t nb = (size_t)timing_tiles * 64 * 768 * TM * 4;
      CK(cudaMalloc(&dXTbig, nb)); CK(cudaMemset(dXTbig, 0, nb));
      q.s[0].XT = dXTbig; q.s[0].shared = 0; q.div = 1; q.row0 = 0;
      printf("unshared inputs: %.2f GB per launch\n", nb / 1e9);
    }
    q.s[1] = q.s[0];
#ifdef PP
    { float* dout3; CK(cudaMalloc(&dout3, (size_t)RT * 256 * 4)); q.s[1].out = dout3; }
#endif
    long long* ddbg; CK(cudaMalloc(&ddbg, 64 * 16 * 8)); CK(cudaMemset(ddbg, 0, 64 * 16 * 8));
    q.dbg = ddbg;
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    for (int it = 0; it < 3; ++it) {
      cudaEventRecord(e0);
      LAUNCH(dim3(GRIDX(timing_tiles), 1), q);
      cudaEventRecord(e1); CK(cudaDeviceSynchronize());
      float ms; cudaEventElapsedTime(&ms, e0, e1);
      double flops = (double)RT * 64 * 2.0 * (256 * 512 + 256 * 256);
#ifdef PP
      flops *= 2;              // two recurrences per tile
#endif
      if (it == 2) {
        long long hd[64 * 16]; CK(cudaMemcpy(hd, ddbg, sizeof(hd), cudaMemcpyDeviceToHost));
#ifndef PP
        for (int t = 10; t < 13; ++t) {
          long long* d = hd + t * 16;
          printf("  step %d MMA thread: wait h %lld | issue r %lld | issue u %lld | wait rh %lld | issue c %lld | total %lld (waits: operand quarters %lld, ring stages %lld)\n", t, d[1] - d[0],
                 d[2] - d[1], d[3] - d[2], d[4] - d[3], d[5] - d[4], hd[(t + 1) * 16] - d[0], d[6], d[7]);
          printf("      epilogue thread 0: wait r %lld | R %lld | wait u %lld | U %lld | wait c %lld | C %lld\n", d[9] - d[8], d[10] - d[9],
                 d[11] - d[10], d[12] - d[11], d[13] - d[12], d[14] - d[13]);
        }
#else
        if (hd[16 * 10]) for (int t = 10; t < 13; ++t) {
          long long* d = hd + t * 16;
          printf("  step %d: waitU %lld | U %lld | waitR %lld | R %lld | waitC %lld | C %lld | total %lld\n", t, d[1] - d[0], d[2] - d[1],
                 d[3] - d[2], d[4] - d[3], d[5] - d[4], d[6] - d[5], hd[(t + 1) * 16] - d[0]);
          printf("      R detail: 2 chunks %lld | publish %lld | 2 chunks %lld | publish %lld\n", d[8] - d[3], d[9] - d[8], d[10] - d[9], d[11] - d[10]);
        }
#endif
      }
      printf("timing: %d tiles (%d rows) %.3f ms -> %.1f TFLOP/s fp32-equivalent, %.0f cycles/step @1.965GHz\n", timing_tiles, RT, ms,
             flops / ms / 1e9, ms * 1e-3 * 1.965e9 / 64 / ((GRIDX(timing_tiles) + 147) / 148));
    }
  }
  return 0;
}

