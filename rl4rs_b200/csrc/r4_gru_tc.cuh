// r4_gru_tc.cuh -- K7 on tcgen05: the interest-extractor GRU (TF1 GRUCell via deepctr DynamicGRU,
// nets/utils.py:120), hidden 128, 64 steps, h0 = 0, every step's output kept (H feeds the attention and the AUGRU).
//
//   r = sigmoid(Xr_t + h Wr)   u = sigmoid(Xu_t + h Wu)   c = tanh(Xc_t + (r*h) Wc)   h <- u h + (1-u) c
//
// Same machinery as the AUGRU kernels (bf16 hi/lo split x3 products, fp32 accumulators in TMEM, fp32 state in
// registers, cp.async.bulk weight ring) but with hidden 128 everything fits without aliasing:
//   TMEM  r | u | c = 3 x 128 columns;  shared: h operand 64 KB + SEPARATE r*h operand 64 KB + 4 x 8 KB ring,
// so the u-GEMM runs while the epilogue converts r*h, and sigmoid(u) is written back in place during the c-GEMM.
// One CTA = 128 sequences.  Warp roles: 8 epilogue warps (thread = row x 64-column half), MMA issuer, TMA producer.
#pragma once
#include "r4_tc_common.cuh"

namespace r4tc {

constexpr int GH = 128;                          // GRU hidden
constexpr int G1_A_BYTES = TM * GH * 2;          // 32 KB per split
constexpr int G1_A_SBO = (GH / 8) * 128;         // 2048
constexpr int G1_STAGE = GH * KB * 2;            // [128 n x 32 k] = 8 KB
constexpr int G1_NST = 4;
constexpr int G1_NKB = GH / KB;                  // 4
constexpr int G1_STAGES_PER_STEP = 3 * G1_NKB * 2;   // r, u, c x 4 K blocks x (hi, lo) = 24
constexpr int G1_IMAGE_BYTES = G1_STAGES_PER_STEP * G1_STAGE;   // 196608
constexpr int G1_SMEM_BYTES = 4 * G1_A_BYTES + G1_NST * G1_STAGE + 1024;
constexpr int G1_XT_COLS = 3 * GH;               // transposed input halves [r | u | c]
constexpr int G1_T_R = 0, G1_T_U = 128, G1_T_C = 256;

// host: Wg [128 k][256 = r|u], Wc [128 k][128] (the h halves of the TF1 GRUCell kernels) -> stream image r, u, c
inline void build_gru_image(const float* Wg, const float* Wc, uint8_t* img) {
  for (int mat = 0; mat < 3; ++mat)
    for (int kb = 0; kb < G1_NKB; ++kb)
      for (int sp = 0; sp < 2; ++sp) {
        uint8_t* st = img + (size_t)((mat * G1_NKB + kb) * 2 + sp) * G1_STAGE;
        for (int n = 0; n < GH; ++n)
          for (int kk = 0; kk < KB; ++kk) {
            int k = kb * KB + kk;
            float w = mat == 0 ? Wg[(size_t)k * 2 * GH + n] : (mat == 1 ? Wg[(size_t)k * 2 * GH + GH + n] : Wc[(size_t)k * GH + n]);
            uint16_t hi = host_bf16_bits(w);
            uint16_t v = sp == 0 ? hi : host_bf16_bits(w - host_bf16_val(hi));
            memcpy(st + (n / 8) * B_SBO + (kk / 8) * LBO + (n % 8) * 16 + (kk % 8) * 2, &v, 2);
          }
      }
}

struct GruTcParams {
  const float* XT;        // [ceil(n/128), steps, 384 / 4, 128, 4]  input halves (+bias), lane-major tiles, quad layout
  const uint8_t* Wimg;    // G1_IMAGE_BYTES
  float* H;               // [n, steps, 128] outputs of every step, or nullptr
  int n;
  int steps = STEPS;      // recurrence length (<= 64): 64 for the behaviour sequences, 21 for the `lstm` simulator's category GRU
  int hard = 0;           // 1: Keras v1 GRU gates, hard sigmoid clip(0.2 x + 0.5, 0, 1) (nets/utils.py:34,92); 0: TF1 GRUCell
  float* Hlast = nullptr; // [n, ld_last] the LAST state only (the `lstm` simulator), or nullptr
  int ld_last = GH;
};

// gate non-linearity of the r / u gates
__device__ __forceinline__ float gru_gate(float x, int hard) {
  return hard ? fminf(fmaxf(fmaf(0.2f, x, 0.5f), 0.0f), 1.0f) : fast_sigmoid(x);
}

__global__ void __launch_bounds__(NTHREADS, 1) k_gru_tc(GruTcParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sHhi = smem;
  uint8_t* sHlo = smem + G1_A_BYTES;
  uint8_t* sRhi = smem + 2 * G1_A_BYTES;
  uint8_t* sRlo = smem + 3 * G1_A_BYTES;
  uint8_t* sB = smem + 4 * G1_A_BYTES;
  __shared__ uint64_t bar_full[G1_NST], bar_empty[G1_NST], bar_h, bar_r, bar_u, bar_rh, bar_c;
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int m0 = blockIdx.x * TM;

  if (tid == 0) {
    for (int i = 0; i < G1_NST; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], 1); }
    mbar_init(&bar_h, 256); mbar_init(&bar_rh, 256);
    mbar_init(&bar_r, 1); mbar_init(&bar_u, 1); mbar_init(&bar_c, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 8) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = tmem_base_s;

  if (warp >= 8) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (warp == 9) {
      if (lane == 0) {
        int stage = 0; uint32_t phase = 0;
        for (int t = 0; t < p.steps; ++t) {
          const uint8_t* src = p.Wimg;
          for (int i = 0; i < G1_STAGES_PER_STEP; ++i, src += G1_STAGE) {
            mbar_wait(&bar_empty[stage], phase ^ 1);
            mbar_expect_tx(&bar_full[stage], G1_STAGE);
            bulk_g2s(sB + stage * G1_STAGE, src, G1_STAGE, &bar_full[stage]);
            if (++stage == G1_NST) { stage = 0; phase ^= 1; }
          }
        }
      }
    } else if (warp == 8) {
      if (lane == 0) {
        constexpr uint32_t idesc = make_idesc(TM, GH);
        const uint32_t bBase = smem_u32(sB);
        int stage = 0; uint32_t phase = 0;
        auto gemm = [&](uint32_t dcol, uint32_t aHi, uint32_t aLo) {
          for (int kb = 0; kb < G1_NKB; ++kb) {
            mbar_wait(&bar_full[stage], phase);
            tc_fence_after();
            {
              uint32_t b = bBase + stage * G1_STAGE;
#pragma unroll
              for (int j = 0; j < KB / 16; ++j) {
                uint64_t db = make_desc(b + j * 2 * LBO, LBO, B_SBO);
                uint32_t koff = (kb * (KB / 16) + j) * 2 * LBO;
                mma_bf16(tbase + dcol, make_desc(aHi + koff, LBO, G1_A_SBO), db, idesc, (kb | j) ? 1u : 0u);
                mma_bf16(tbase + dcol, make_desc(aLo + koff, LBO, G1_A_SBO), db, idesc, 1u);
              }
            }
            umma_commit(&bar_empty[stage]);
            if (++stage == G1_NST) { stage = 0; phase ^= 1; }
            mbar_wait(&bar_full[stage], phase);
            tc_fence_after();
            {
              uint32_t b = bBase + stage * G1_STAGE;
#pragma unroll
              for (int j = 0; j < KB / 16; ++j) {
                uint64_t db = make_desc(b + j * 2 * LBO, LBO, B_SBO);
                uint32_t koff = (kb * (KB / 16) + j) * 2 * LBO;
                mma_bf16(tbase + dcol, make_desc(aHi + koff, LBO, G1_A_SBO), db, idesc, 1u);
              }
            }
            umma_commit(&bar_empty[stage]);
            if (++stage == G1_NST) { stage = 0; phase ^= 1; }
          }
        };
        const uint32_t hHi = smem_u32(sHhi), hLo = smem_u32(sHlo), rHi = smem_u32(sRhi), rLo = smem_u32(sRlo);
        for (int t = 0; t < p.steps; ++t) {
          const uint32_t par = t & 1;
          mbar_wait(&bar_h, par);
          tc_fence_after();
          gemm(G1_T_R, hHi, hLo);
          umma_commit(&bar_r);
          gemm(G1_T_U, hHi, hLo);          // overlaps the epilogue's r*h conversion (separate operand buffer)
          umma_commit(&bar_u);
          mbar_wait(&bar_rh, par);
          tc_fence_after();
          gemm(G1_T_C, rHi, rLo);
          umma_commit(&bar_c);
        }
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    const int q = warp & 3, half = warp >> 2;
    const int row = q * 32 + lane;
    const int c0 = half * 64;
    int n = m0 + row;
    const bool valid = n < p.n;
    if (!valid) n = p.n - 1;
    const float* xt = p.XT + ((size_t)(n / TM) * p.steps) * G1_XT_COLS * TM;
    const int ln4 = (n % TM) * 4;
    float* hout = p.H ? p.H + (size_t)n * p.steps * GH + c0 : nullptr;
    const int hard = p.hard;
    const uint32_t tlane = tbase + ((uint32_t)(q * 32) << 16);
    const uint32_t a_row_off = (uint32_t)(row / 8) * G1_A_SBO + (uint32_t)(row % 8) * 16;
    float h[64];
#pragma unroll
    for (int i = 0; i < 64; ++i) h[i] = 0.f;
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      uint32_t off = a_row_off + (uint32_t)((c0 + g * 8) / 8) * LBO;
      *reinterpret_cast<uint4*>(sHhi + off) = make_uint4(0, 0, 0, 0);
      *reinterpret_cast<uint4*>(sHlo + off) = make_uint4(0, 0, 0, 0);
    }
    proxy_fence();
    mbar_arrive(&bar_h);

    for (int t = 0; t < p.steps; ++t) {
      const uint32_t par = t & 1;
      const float* xs = xt + (size_t)t * G1_XT_COLS * TM;
#define R4_LOADX(dst, colbase) load_x16(dst, xs, (colbase), ln4)
      // ---- phase R: r*h -> its own operand buffer ----
      {
        float x[2][16], a[2][16];
        R4_LOADX(x[0], c0);
        mbar_wait(&bar_r, par);
        tc_fence_after();
        tmem_ld16(tlane + G1_T_R + c0, a[0]);
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          const int cur = ch & 1, nxt = cur ^ 1;
          tmem_wait_ld();
          if (ch < 3) { R4_LOADX(x[nxt], c0 + (ch + 1) * 16); tmem_ld16(tlane + G1_T_R + c0 + (ch + 1) * 16, a[nxt]); }
#pragma unroll
          for (int j = 0; j < 16; ++j) a[cur][j] = gru_gate(a[cur][j] + x[cur][j], hard) * h[ch * 16 + j];
#pragma unroll
          for (int g = 0; g < 2; ++g) {
            uint4 hi, lo;
            split8(a[cur] + g * 8, hi, lo);
            uint32_t off = a_row_off + (uint32_t)((c0 + ch * 16 + g * 8) / 8) * LBO;
            *reinterpret_cast<uint4*>(sRhi + off) = hi;
            *reinterpret_cast<uint4*>(sRlo + off) = lo;
          }
        }
      }
      tc_fence_before();
      proxy_fence();
      mbar_arrive(&bar_rh);
      // ---- phase U (during the c-GEMM): u = sigmoid(acc_u + Xu) -> back into TMEM (in place) ----
      {
        float x[2][16], a[2][16];
        R4_LOADX(x[0], GH + c0);
        mbar_wait(&bar_u, par);
        tc_fence_after();
        tmem_ld16(tlane + G1_T_U + c0, a[0]);
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          const int cur = ch & 1, nxt = cur ^ 1;
          tmem_wait_ld();
          if (ch < 3) { R4_LOADX(x[nxt], GH + c0 + (ch + 1) * 16); tmem_ld16(tlane + G1_T_U + c0 + (ch + 1) * 16, a[nxt]); }
#pragma unroll
          for (int j = 0; j < 16; ++j) a[cur][j] = gru_gate(a[cur][j] + x[cur][j], hard);
          tmem_st16(tlane + G1_T_U + c0 + ch * 16, a[cur]);
        }
        tmem_wait_st();
      }
      // ---- phase C: c = tanh(acc_c + Xc); h <- u h + (1-u) c -> operand buffer + H[t] ----
      {
        float x[2][16], a[2][16], u[2][16];
        R4_LOADX(x[0], 2 * GH + c0);
        mbar_wait(&bar_c, par);
        tc_fence_after();
        tmem_ld16(tlane + G1_T_C + c0, a[0]);
        tmem_ld16(tlane + G1_T_U + c0, u[0]);
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          const int cur = ch & 1, nxt = cur ^ 1;
          tmem_wait_ld();
          if (ch < 3) {
            R4_LOADX(x[nxt], 2 * GH + c0 + (ch + 1) * 16);
            tmem_ld16(tlane + G1_T_C + c0 + (ch + 1) * 16, a[nxt]);
            tmem_ld16(tlane + G1_T_U + c0 + (ch + 1) * 16, u[nxt]);
          }
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            float c = fast_tanh(a[cur][j] + x[cur][j]);
            float hn = fmaf(u[cur][j], h[ch * 16 + j] - c, c);
            h[ch * 16 + j] = hn;
            a[cur][j] = hn;
          }
#pragma unroll
          for (int g = 0; g < 2; ++g) {
            uint4 hi, lo;
            split8(a[cur] + g * 8, hi, lo);
            uint32_t off = a_row_off + (uint32_t)((c0 + ch * 16 + g * 8) / 8) * LBO;
            *reinterpret_cast<uint4*>(sHhi + off) = hi;
            *reinterpret_cast<uint4*>(sHlo + off) = lo;
          }
          if (valid && hout) {
            float* o = hout + (size_t)t * GH + ch * 16;
#pragma unroll
            for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(a[cur][j], a[cur][j + 1], a[cur][j + 2], a[cur][j + 3]);
          }
        }
      }
#undef R4_LOADX
      tc_fence_before();
      proxy_fence();
      mbar_arrive(&bar_h);
    }
    if (valid && p.Hlast) {
      float* o = p.Hlast + (size_t)n * p.ld_last + c0;
#pragma unroll
      for (int i = 0; i < 64; i += 4) *reinterpret_cast<float4*>(o + i) = make_float4(h[i], h[i + 1], h[i + 2], h[i + 3]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tbase), "r"(512));
}

}  // namespace r4tc
