// r4_gemm_tc.cuh -- fp32-parity dense layers on tcgen05 (Keras Dense: nets/utils.py:50-53,
// dien.py:35; the input projections of GRU-1 / AUGRU / attention; the Embedding gather fused in).
//
//   C[M,N] = act(A[M,K] . W[K,N] + bias)      A, C, bias fp32 in HBM; W pre-tiled bf16 hi/lo image
//
// Numerics: fp32-exact in practice.  Every operand is split THREE ways, x = hi + mid + lo (bf16 each,
// 24 significand bits together), and the six products whose magnitude exceeds 2^-24 of the result are
// issued (hh, hm, mh, hl, lh, mm), fp32 accumulation in TMEM.  These layers are a few % of the step, so
// the 2x tensor work over the 2-way split of the recurrence buys parity margin for free.
// Persistent CTAs (one per SM) walk the 128-row x (<=256)-column tiles.
// Warp roles: 0-7 A producers (cp.async fp32 rows -> bf16 hi/mid/lo core matrices), 8 MMA issuer, 9 TMA producer
// for W, 12-15 epilogue (TMEM -> bias/act -> global) on the second of two TMEM accumulators, 10-11 idle.
// Operand ring: 2 stages x (A hi/mid/lo 24 KB + W hi/mid/lo <=48 KB), K block = 32; raw A ring: 4 x 16 KB.
#pragma once
#include "r4_tc_common.cuh"

namespace r4tc {

constexpr int G_BM = 128, G_BK = 32, G_NST = 2, G_BNMAX = 256, G_SPLIT = 3, G_RAW = 3, G_OUTB = 3;
constexpr int G_A_STAGE = G_BM * G_BK * 2;                 // 8 KB per split
constexpr int G_B_STAGE = G_BNMAX * G_BK * 2;              // 16 KB per split (max)
constexpr int G_STAGE_BYTES = G_SPLIT * G_A_STAGE + G_SPLIT * G_B_STAGE;   // 72 KB
constexpr int G_RAW_BYTES = G_BM * G_BK * 4;                // 16 KB: one K block of fp32 A rows as they arrive (cp.async)
constexpr int G_OUT_BYTES = 16 * G_BM * 4;                  // 8 KB: 16 output columns x 128 rows, staged for one bulk store
constexpr int G_SMEM_BYTES = G_NST * G_STAGE_BYTES + G_RAW * G_RAW_BYTES + G_OUTB * G_OUT_BYTES + 1024;
constexpr int G_THREADS = 512;
constexpr int G_W_MMA = 8, G_W_TMA = 9, G_W_EPI = 12, G_EPI_T0 = G_W_EPI * 32;   // warps 0-7 produce A, 10-11 idle
constexpr int G_A_SBO = (G_BK / 8) * 128;                  // 512
constexpr int G_B_SBO = (G_BK / 8) * 128;                  // 512

// host-side description of a pre-tiled weight
struct GemmImage {
  const uint8_t* img = nullptr;   // device
  int K = 0, N = 0, kblocks = 0;  // kblocks = ceil(K/32) (zero padded)
};

// image layout: n-tile nt (256 columns, last one narrower), K block kb, split {hi, lo}: [bn x 32] core matrices
// bnt = n-tile width the image is cut for (<= 256, multiple of 16): 256 by default; 128 for a GEMM whose m-tiles alone
// would leave most SMs idle (the observation head: 32 m-tiles at batch 4096).
inline size_t gemm_image_bytes(int K, int N, int bnt = G_BNMAX) {
  int kb = (K + G_BK - 1) / G_BK;
  size_t tot = 0;
  for (int n0 = 0; n0 < N; n0 += bnt) tot += (size_t)kb * G_SPLIT * std::min(bnt, N - n0) * G_BK * 2;
  return tot;
}
inline void build_gemm_image(const float* W /*[K][N]*/, int K, int N, uint8_t* img, int bnt = G_BNMAX) {
  int kbn = (K + G_BK - 1) / G_BK;
  size_t off = 0;
  for (int n0 = 0; n0 < N; n0 += bnt) {
    int bn = std::min(bnt, N - n0);
    for (int kb = 0; kb < kbn; ++kb)
      for (int sp = 0; sp < G_SPLIT; ++sp) {
        uint8_t* st = img + off;
        for (int n = 0; n < bn; ++n)
          for (int kk = 0; kk < G_BK; ++kk) {
            int k = kb * G_BK + kk;
            float w = k < K ? W[(size_t)k * N + n0 + n] : 0.f;
            uint16_t hi = host_bf16_bits(w);
            float r1 = w - host_bf16_val(hi);
            uint16_t mid = host_bf16_bits(r1);
            uint16_t lo = host_bf16_bits(r1 - host_bf16_val(mid));
            uint16_t v = sp == 0 ? hi : (sp == 1 ? mid : lo);
            memcpy(st + (n / 8) * G_B_SBO + (kk / 8) * LBO + (n % 8) * 16 + (kk % 8) * 2, &v, 2);
          }
        off += (size_t)bn * G_BK * 2;
      }
  }
}

// element (tile-step base, column, lane) of a lane-major tile, in floats; ld = columns per step
__host__ __device__ __forceinline__ size_t xt_index(size_t tile_step, int ld, int col, int lane) {
  return (tile_step * ld + (size_t)(col & ~3)) * TM + (size_t)lane * 4 + (col & 3);
}

// float index of column quad `quad` (4 consecutive columns) of (sequence nabs, step t) in the key-half cache Kp: layout
// [sequence][column quad][step][4].  The scores kernels read it with lane = step (key): the 32 lanes of a warp read 512
// contiguous bytes per 128-bit load.  (Round 2, ncu on k_scores_tc: with the row-major [sequence][step][64] layout every
// lane read its own 256-byte row -- 32 L1 wavefronts per warp load, 2 k of the kernel's 4.5 k global-load wavefronts per
// tile, with the LSU data pipe at 70 % the unit that set the tile time.)
__host__ __device__ __forceinline__ size_t kq_index(size_t nabs, int nquads, int quad, int steps, int t) {
  return ((nabs * nquads + quad) * steps + t) * 4;
}

struct GemmTcParams {
  const float* A; int lda; const int32_t* gather;
  const uint8_t* Wimg; const float* bias; float* C; int ldc;
  int M, N, K, act;     // act: 0 none, 1 ELU
  // "sequence" mode (tm_ns > 0): the M = tm_ns * 64 rows are (sequence n, step t) pairs enumerated t-major
  // (m = t * tm_ns + n; source row n * 64 + t), and the result is written in the lane-major tile layout the
  // recurrent kernels read: columns < ldT -> outT[((nabs/128) * 64 + t) * ldT + col) * 128 + nabs % 128],
  // columns >= ldT -> outK in the quad layout [nabs][(col - ldT) / 4][t][4] (kq_index), nabs = cr_base + n.  Consecutive threads are
  // consecutive sequences of one step, so both reads and transposed writes stay coalesced.
  // Inside a tile-step the columns are grouped in QUADS, [col / 4][lane][col % 4] (xt_index below): a recurrent
  // kernel's thread (= lane) reads 4 consecutive columns with ONE 128-bit load (ncu, round 2: with one 32-bit load per
  // column the AUGRU epilogue spent 18 % of its cycles in lg_throttle, 192 LDGs per thread and step).
  int tm_ns, cr_base, ldT; float* outT; float* outK;
  int tm_steps = STEPS;       // steps per sequence in sequence mode (64; 21 for the `lstm` simulator's category GRU)
  int bnt = G_BNMAX;          // n-tile width of the weight image (build_gemm_image)
  // Second, GATHERED part of the A operand (the observation head: K = 768 + 21 x 128): for k >= k2_start, A[m][k] is
  // A2[gather2[m * g2_n + j] * 128 + (k - k2_start) % 128] with j = (k - k2_start) / 128 -- the Flatten() of the category
  // embeddings (nets/utils.py:24) read straight from the embedding table (L2-resident, 51 MB) instead of from a
  // 10.7 KB-per-row copy that k_cat_attn used to write and this kernel used to read back.  k2_start % 32 == 0.
  const float* A2 = nullptr; const int32_t* gather2 = nullptr; int k2_start = 0, g2_n = 0;
  // Split-K (ksplit > 1): tile t = (output tile t / ksplit, K part t % ksplit); every part writes its raw accumulators
  // to part[ks][M][N] and k_splitk_finish adds them in part order (deterministic), then bias + activation.  For GEMMs with
  // fewer output tiles than SMs and a long K (the observation head: 64 tiles x 108 K blocks at 4096 rows).
  int ksplit = 1; float* part = nullptr;
  long long* dbg = nullptr;   // development probe (tools/gemm_probe.cu): per-role wait/busy cycles of CTA 0
};

// K blocks [kb0, kb1) of part `ks`: boundaries on multiples of 4 K blocks, so a part never starts inside a 128-wide
// gathered slot (k2_start / 32 is a multiple of 4)
__device__ __forceinline__ void gemm_kpart(int kbn, int ksplit, int ks, int& kb0, int& kb1) {
  if (ksplit <= 1) { kb0 = 0; kb1 = kbn; return; }
  const int b0 = ks == 0 ? 0 : min(kbn, (int)(((long long)kbn * ks / ksplit + 2) / 4 * 4));
  const int b1 = ks + 1 >= ksplit ? kbn : min(kbn, (int)(((long long)kbn * (ks + 1) / ksplit + 2) / 4 * 4));
  kb0 = b0; kb1 = b1;
}

// out = act(sum_ks part[ks] + bias): the second, deterministic pass of a split-K GEMM.  One thread = 4 columns.
__global__ void k_splitk_finish(int M, int N, int ksplit, const float* __restrict__ part, const float* __restrict__ bias, int act,
                                float* __restrict__ C, int ldc) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int n4 = N / 4;
  if (i >= (size_t)M * n4) return;
  const int m = (int)(i / n4), n = (int)(i % n4) * 4;
  float4 a = *reinterpret_cast<const float4*>(part + (size_t)m * N + n);
  for (int ks = 1; ks < ksplit; ++ks) {
    const float4 b = *reinterpret_cast<const float4*>(part + ((size_t)ks * M + m) * N + n);
    a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
  }
  if (bias) { a.x += __ldg(bias + n); a.y += __ldg(bias + n + 1); a.z += __ldg(bias + n + 2); a.w += __ldg(bias + n + 3); }
  if (act == 1) {
    a.x = a.x > 0.f ? a.x : expm1f(a.x); a.y = a.y > 0.f ? a.y : expm1f(a.y);
    a.z = a.z > 0.f ? a.z : expm1f(a.z); a.w = a.w > 0.f ? a.w : expm1f(a.w);
  }
  *reinterpret_cast<float4*>(C + (size_t)m * ldc + n) = a;
}

__device__ __forceinline__ void cp_async16(void* dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" :: "r"(smem_u32(dst)), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory"); }

// Persistent: gridDim.x CTAs walk the (m-tile, n-tile) list (n inner, so the CTAs working on one m-tile at the same
// time share its A rows in L2).  The four pipelines -- A staging (cp.async, G_RAW K blocks in flight per thread),
// W stream (TMA), MMA, epilogue -- run across tile boundaries; two 256-column TMEM accumulators let the epilogue of
// tile i overlap the main loop of tile i+1.
__global__ void __launch_bounds__(G_THREADS, 1) k_gemm_tc(GemmTcParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* raw = smem + G_NST * G_STAGE_BYTES;
  uint8_t* outb = raw + G_RAW * G_RAW_BYTES;
  __shared__ uint64_t bar_a[G_NST], bar_b[G_NST], bar_empty[G_NST], acc_full[2], acc_empty[2];
  __shared__ uint32_t tmem_base_s;
  __shared__ __align__(16) float bias_s[2][G_BNMAX];          // bias of the tile in each accumulator's epilogue
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int kbn = (p.K + G_BK - 1) / G_BK;
  const int ntn = (p.N + p.bnt - 1) / p.bnt, mtn = (p.M + G_BM - 1) / G_BM, ksp = max(p.ksplit, 1), ntiles = mtn * ntn * ksp;

  if (tid == 0) {
    for (int i = 0; i < G_NST; ++i) { mbar_init(&bar_a[i], 256); mbar_init(&bar_b[i], 1); mbar_init(&bar_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == G_W_MMA) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = tmem_base_s;

  if (warp == G_W_TMA) {
    // ===== W stream =====
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int nt = (tile / ksp) % ntn;
        int kb0, kb1; gemm_kpart(kbn, ksp, tile % ksp, kb0, kb1);
        const uint32_t bsb = (uint32_t)min(p.bnt, p.N - nt * p.bnt) * G_BK * 2;
        // start of this n-tile in the image: the tiles before it are full width
        const uint8_t* wtile = p.Wimg + (size_t)nt * kbn * G_SPLIT * p.bnt * G_BK * 2;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&bar_empty[stage], phase ^ 1);
          uint8_t* dst = smem + stage * G_STAGE_BYTES + G_SPLIT * G_A_STAGE;
          mbar_expect_tx(&bar_b[stage], G_SPLIT * bsb);
#pragma unroll
          for (int sp = 0; sp < G_SPLIT; ++sp)
            bulk_g2s(dst + sp * G_B_STAGE, wtile + ((size_t)kb * G_SPLIT + sp) * bsb, bsb, &bar_b[stage]);
          if (++stage == G_NST) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == G_W_MMA) {
    // ===== MMA issuer =====
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      int li = 0;
      long long w_acc = 0, w_a = 0, w_b = 0, t_begin = clock64();
      const bool probe = p.dbg && blockIdx.x == 0;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++li) {
        const int nt = (tile / ksp) % ntn;
        int kb0, kb1; gemm_kpart(kbn, ksp, tile % ksp, kb0, kb1);
        const uint32_t idesc = make_idesc(G_BM, min(p.bnt, p.N - nt * p.bnt));
        const uint32_t acc = tbase + (uint32_t)(li & 1) * G_BNMAX;
        long long c0 = probe ? clock64() : 0;
        mbar_wait(&acc_empty[li & 1], (uint32_t)((li >> 1) & 1) ^ 1u);   // the epilogue has drained this accumulator
        if (probe) w_acc += clock64() - c0;
        tc_fence_after();
        for (int kb = kb0; kb < kb1; ++kb) {
          if (probe) {
            long long c1 = clock64(); mbar_wait(&bar_a[stage], phase);
            long long c2 = clock64(); mbar_wait(&bar_b[stage], phase);
            w_a += c2 - c1; w_b += clock64() - c2;
          } else { mbar_wait(&bar_a[stage], phase); mbar_wait(&bar_b[stage], phase); }
          tc_fence_after();
          uint32_t sa = smem_u32(smem + stage * G_STAGE_BYTES);
          uint32_t sb = sa + G_SPLIT * G_A_STAGE;
#pragma unroll
          for (int j = 0; j < G_BK / 16; ++j) {
            uint64_t a[3], b[3];
#pragma unroll
            for (int sp = 0; sp < 3; ++sp) {
              a[sp] = make_desc(sa + sp * G_A_STAGE + j * 2 * LBO, LBO, G_A_SBO);
              b[sp] = make_desc(sb + sp * G_B_STAGE + j * 2 * LBO, LBO, G_B_SBO);
            }
            // smallest products first so they are not absorbed by a large partial sum
            mma_bf16(acc, a[1], b[1], idesc, (kb > kb0 || j) ? 1u : 0u);   // mid*mid
            mma_bf16(acc, a[0], b[2], idesc, 1u);                   // hi*lo
            mma_bf16(acc, a[2], b[0], idesc, 1u);                   // lo*hi
            mma_bf16(acc, a[0], b[1], idesc, 1u);                   // hi*mid
            mma_bf16(acc, a[1], b[0], idesc, 1u);                   // mid*hi
            mma_bf16(acc, a[0], b[0], idesc, 1u);                   // hi*hi
          }
          umma_commit(&bar_empty[stage]);
          if (++stage == G_NST) { stage = 0; phase ^= 1; }
        }
        umma_commit(&acc_full[li & 1]);
      }
      if (probe) { p.dbg[0] = clock64() - t_begin; p.dbg[1] = w_acc; p.dbg[2] = w_a; p.dbg[3] = w_b; p.dbg[4] = li; }
    }
  } else if (warp < 8) {
    // ===== A producers: thread (r8 = tid/4, kc = tid%4) stages and converts 8 consecutive K values of 4 rows per
    // K block.  The fp32 rows come in through cp.async into a private 32-byte slot per (row, kc); G_RAW - 1 K blocks
    // are in flight while one is converted (a register-staged single prefetch left the GEMMs latency-bound).
    const int kc = tid & 3, r8 = tid >> 2;      // 64 row slots x 2 passes
    const float* arow[2] = {p.A, p.A};
    const int32_t* grow[2] = {p.gather2, p.gather2};
    int id_cur[2] = {0, 0}, id_next[2] = {0, 0};   // gathered part: table row of the current / next 128-wide slot of each row
    int is_tile = blockIdx.x, is_kb0 = 0, is_kb1 = kbn;
    if (is_tile < ntiles) gemm_kpart(kbn, ksp, is_tile % ksp, is_kb0, is_kb1);
    int is_kb = is_kb0;
    auto issue = [&](int slot) {
      if (is_tile < ntiles) {
        if (is_kb == is_kb0) {
          const int m0 = (is_tile / ksp / ntn) * G_BM;
#pragma unroll
          for (int it = 0; it < 2; ++it) {
            int m = m0 + it * 64 + r8;
            if (m >= p.M) m = p.M - 1;
            if (p.tm_ns > 0) m = (m % p.tm_ns) * p.tm_steps + (m / p.tm_ns);
            size_t src = p.gather ? (size_t)__ldg(p.gather + m) : (size_t)m;
            arow[it] = p.A + src * p.lda + kc * 8;
            if (p.A2) {        // slot 0: needed k2_start / 32 K blocks later; a K part that starts inside the gathered region: its own slot
              grow[it] = p.gather2 + (size_t)m * p.g2_n;
              id_next[it] = __ldg(grow[it] + max(0, (is_kb0 * G_BK - p.k2_start) >> 7));
            }
          }
        }
        const bool part2 = p.A2 && is_kb * G_BK >= p.k2_start;
        const int k2 = is_kb * G_BK - p.k2_start;              // offset inside the gathered part (multiple of 32)
        if (part2 && (k2 & 127) == 0) {                        // entering slot j: its id was requested 4 K blocks ago; request j + 1
          const int j = k2 >> 7;
#pragma unroll
          for (int it = 0; it < 2; ++it) {
            id_cur[it] = id_next[it];
            if (j + 1 < p.g2_n) id_next[it] = __ldg(grow[it] + j + 1);
          }
        }
        const bool kok = is_kb * G_BK + kc * 8 + 8 <= p.K;   // K % 8 == 0 is required; beyond K: zero fill
        const uint32_t nb = kok ? 16u : 0u;
#pragma unroll
        for (int it = 0; it < 2; ++it) {
          uint8_t* dst = raw + slot * G_RAW_BYTES + (it * 64 + r8) * (G_BK * 4) + kc * 32;
          const float* src = kok ? arow[it] + is_kb * G_BK : arow[it];
          if (part2 && kok) src = p.A2 + (size_t)id_cur[it] * 128 + (k2 & 127) + kc * 8;
          cp_async16(dst, src, nb);
          cp_async16(dst + 16, src + 4, nb);
        }
        if (++is_kb == is_kb1) {
          is_tile += gridDim.x;
          if (is_tile < ntiles) gemm_kpart(kbn, ksp, is_tile % ksp, is_kb0, is_kb1);
          is_kb = is_kb0;
        }
      }
      cp_async_commit();
    };
#pragma unroll
    for (int d = 0; d < G_RAW - 1; ++d) issue(d);
    int stage = 0; uint32_t phase = 0;
    int slot = 0;
    long long w_cp = 0, w_empty = 0;
    const bool probe = p.dbg && blockIdx.x == 0 && tid == 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      int ckb0, ckb1; gemm_kpart(kbn, ksp, tile % ksp, ckb0, ckb1);
      for (int kb = ckb0; kb < ckb1; ++kb) {
        issue(slot == 0 ? G_RAW - 1 : slot - 1);          // the slot converted in the previous iteration
        long long c0 = probe ? clock64() : 0;
        cp_async_wait<G_RAW - 1>();
        long long c1 = probe ? clock64() : 0;
        mbar_wait(&bar_empty[stage], phase ^ 1);
        if (probe) { w_cp += c1 - c0; w_empty += clock64() - c1; }
        uint8_t* sa = smem + stage * G_STAGE_BYTES;
#pragma unroll
        for (int it = 0; it < 2; ++it) {
          const int row = it * 64 + r8;
          const uint8_t* rs = raw + slot * G_RAW_BYTES + row * (G_BK * 4) + kc * 32;
          float v[8];
          *reinterpret_cast<float4*>(v) = *reinterpret_cast<const float4*>(rs);
          *reinterpret_cast<float4*>(v + 4) = *reinterpret_cast<const float4*>(rs + 16);
          uint4 hi, mid, lo;
          float r1[8];
          split8(v, hi, mid);                             // hi and bf16(x - hi)
          {
            const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&hi);
            const __nv_bfloat162* m2 = reinterpret_cast<const __nv_bfloat162*>(&mid);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              r1[2 * j] = (v[2 * j] - __bfloat162float(h2[j].x)) - __bfloat162float(m2[j].x);
              r1[2 * j + 1] = (v[2 * j + 1] - __bfloat162float(h2[j].y)) - __bfloat162float(m2[j].y);
            }
            uint32_t l[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              __nv_bfloat162 ll = __floats2bfloat162_rn(r1[2 * j], r1[2 * j + 1]);
              l[j] = *reinterpret_cast<uint32_t*>(&ll);
            }
            lo = make_uint4(l[0], l[1], l[2], l[3]);
          }
          uint32_t off = (uint32_t)(row / 8) * G_A_SBO + (uint32_t)kc * LBO + (uint32_t)(row % 8) * 16;
          *reinterpret_cast<uint4*>(sa + off) = hi;
          *reinterpret_cast<uint4*>(sa + G_A_STAGE + off) = mid;
          *reinterpret_cast<uint4*>(sa + 2 * G_A_STAGE + off) = lo;
        }
        proxy_fence();
        mbar_arrive(&bar_a[stage]);
        if (++stage == G_NST) { stage = 0; phase ^= 1; }
        if (++slot == G_RAW) slot = 0;
      }
    }
    cp_async_wait<0>();
    if (probe) { p.dbg[5] = w_cp; p.dbg[6] = w_empty; }
  } else if (warp >= G_W_EPI) {
    // ===== epilogue: thread = row =====
    const int q = warp - G_W_EPI;
    const int row = q * 32 + lane;
    int li = 0, nchunk = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++li) {
      const int bt = tile / ksp, ks = tile % ksp;
      const int m0 = (bt / ntn) * G_BM, n0 = (bt % ntn) * p.bnt;
      const int bn = min(p.bnt, p.N - n0);
      const int m = m0 + row;
      const uint32_t tlane = tbase + (uint32_t)(li & 1) * G_BNMAX + ((uint32_t)(q * 32) << 16);
      const bool probe = p.dbg && blockIdx.x == 0 && tid == G_EPI_T0;
      for (int i = tid - G_EPI_T0; i < bn; i += 128) bias_s[li & 1][i] = p.bias ? __ldg(p.bias + n0 + i) : 0.f;
      asm volatile("bar.sync 1, 128;" ::: "memory");
      long long c0 = probe ? clock64() : 0;
      mbar_wait(&acc_full[li & 1], (uint32_t)((li >> 1) & 1));
      long long c1 = probe ? clock64() : 0;
      tc_fence_after();
      // Sequence mode, aligned tile: its 128 rows are 128 consecutive sequences of ONE step, so 16 output columns are
      // one contiguous 8 KB block of the lane-major layout: stage them in shared memory ([column][row], conflict-free)
      // and let the bulk-copy engine write the block -- one instruction by one thread instead of 16 x 128-byte warp
      // stores per warp, and no store traffic in the epilogue warps' instruction stream.
      const bool blk = p.tm_ns > 0 && (p.tm_ns % G_BM) == 0 && (p.cr_base % G_BM) == 0 && m0 + G_BM <= p.M;
      for (int c = 0; c < bn; c += 16) {
        float a[16];
        long long e0 = probe ? clock64() : 0;
        tmem_ld16(tlane + c, a);
        tmem_wait_ld();
        long long e1 = probe ? clock64() : 0;
        if (ksp > 1) {          // split-K: raw partial sums, bias + activation in k_splitk_finish
          if (m < p.M) {
            float* o = p.part + ((size_t)ks * p.M + m) * p.N + n0 + c;
#pragma unroll
            for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(a[j], a[j + 1], a[j + 2], a[j + 3]);
          }
          continue;
        }
        // bias + activation for the whole chunk first, branch-free: with the bias load, the ELU branch and the store
        // interleaved per element the chunk was a chain of 16 exposed latencies (~2.4k cycles; ncu source page in
        // profiles/) and the epilogue, not the MMAs, set the time of the sequence-mode GEMMs.
        {
          const float4* b4 = reinterpret_cast<const float4*>(bias_s[li & 1] + c);
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) {
            const float4 bq = b4[q4];
            a[4 * q4] += bq.x; a[4 * q4 + 1] += bq.y; a[4 * q4 + 2] += bq.z; a[4 * q4 + 3] += bq.w;
          }
        }
        if (p.act == 1) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float en = expm1f(fminf(a[j], 0.f));
            a[j] = a[j] > 0.f ? a[j] : en;
          }
        }
        if (blk && n0 + c + 16 <= p.ldT) {
          float* ob = reinterpret_cast<float*>(outb + (nchunk % G_OUTB) * G_OUT_BYTES);
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4)      // [column quad][row][4]: the quad layout of the lane-major tiles
            *reinterpret_cast<float4*>(ob + j4 * G_BM * 4 + row * 4) = make_float4(a[4 * j4], a[4 * j4 + 1], a[4 * j4 + 2], a[4 * j4 + 3]);
          long long e2 = probe ? clock64() : 0;
          proxy_fence();
          long long e3 = probe ? clock64() : 0;
          // the buffer the NEXT chunk will use must have been read out by its previous bulk store
          if (tid == G_EPI_T0) asm volatile("cp.async.bulk.wait_group.read %0;" :: "n"(G_OUTB - 2) : "memory");
          asm volatile("bar.sync 1, 128;" ::: "memory");
          if (tid == G_EPI_T0) {
            const int t = m0 / p.tm_ns, nb = (p.cr_base + m0 % p.tm_ns) / G_BM;
            float* dst = p.outT + (((size_t)nb * p.tm_steps + t) * p.ldT + (n0 + c)) * TM;
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" :: "l"(dst), "r"(smem_u32(ob)), "r"(G_OUT_BYTES) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
          if (probe) { long long e4 = clock64(); p.dbg[9] += e1 - e0; p.dbg[10] += e2 - e1; p.dbg[11] += e3 - e2; p.dbg[12] += e4 - e3; }
          ++nchunk;
        } else if (m < p.M && p.tm_ns > 0) {
          const int t = m / p.tm_ns, nabs = p.cr_base + m % p.tm_ns;
          if (n0 + c >= p.ldT) {            // ldT % 16 == 0: a 16-column chunk lies on one side.  outK in the quad layout (kq_index)
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4)
              *reinterpret_cast<float4*>(p.outK + kq_index(nabs, (p.N - p.ldT) / 4, (n0 + c - p.ldT) / 4 + j4, p.tm_steps, t)) =
                  make_float4(a[4 * j4], a[4 * j4 + 1], a[4 * j4 + 2], a[4 * j4 + 3]);
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const int col = n0 + c + j;
              if (col < p.ldT) p.outT[xt_index((size_t)(nabs / TM) * p.tm_steps + t, p.ldT, col, nabs % TM)] = a[j];
            }
          }
        } else if (m < p.M) {
          float* o = p.C + (size_t)m * p.ldc + n0 + c;
#pragma unroll
          for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(a[j], a[j + 1], a[j + 2], a[j + 3]);
        }
      }
      tc_fence_before();
      mbar_arrive(&acc_empty[li & 1]);
      if (probe) { p.dbg[7] += c1 - c0; p.dbg[8] += clock64() - c1; }
    }
    if (tid == G_EPI_T0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // staging buffers are read out before exit
  }
  tc_fence_before();
  __syncthreads();
  if (warp == G_W_MMA) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tbase), "r"(512));
}

}  // namespace r4tc
