// r4_scores_tc.cuh -- K8 on tcgen05: DIN local-activation scores (deepctr AttentionSequencePoolingLayer
// (att_hidden_units=(64,16), return_score=True, weight_normalization=False); nets/utils.py:114-115,121-122).
//
//   q      = mean_j E_s[cat[-10:]]                                     (query, per feature row)
//   z1_t   = sigmoid(q (Wq+Wd) + b1 + k_t (Wk-Wd) + (q * k_t) Wp)       k_t = GRU-1 output t (cached H)
//   z2_t   = sigmoid(z1_t W2 + b2);   score_t = z2_t . kv + b           (raw, unbounded)
//
// k_query computes q and the query half q (Wq+Wd) + b1 per feature row; k_scores_tc2 does the rest, both attention
// layers on the tensor pipe, and writes the scores in the lane-major tile layout the AUGRU kernels read.
#pragma once
#include "r4_tc_common.cuh"
#include "r4_gemm_tc.cuh"

namespace r4tc {

constexpr int S_K = 128, S_N = 64, S_KEYS = 64, AH2_N = 16;
// A operand (built by the producer warps): K-adjacent core matrices 160 B apart instead of 128.  With LBO = 128 the K
// chunks of a row hit the same banks: a producer quarter-warp that stored (2 rows x 4 K chunks) replayed every 128-bit
// operand store 4x and ran the kernel at 84 % of the L1/shared pipe on those replays (ncu, round 2).  With 160 the bank
// group of (row, kc) is (row + 2 kc) mod 8: distinct.
constexpr int S_A_LBO = 160;
constexpr int S_A_SBO = (S_K / 8) * S_A_LBO;       // 2560: 8-row groups of the A operand
constexpr int S_A_SPLIT = (TM / 8) * S_A_SBO;      // 40 KB per split
constexpr int S_A_STAGE = 2 * S_A_SPLIT;           // hi + lo = 80 KB
constexpr int S_B_SPLIT = S_N * S_K * 2;           // 16 KB per split
constexpr int S_B_BYTES = 3 * S_B_SPLIT;           // 48 KB, resident
constexpr int S_SBO = (S_K / 8) * 128;             // 2048: 8-row groups (B: the weight image)
// cached key half k_t (Wk - Wd): Kp [n_cached][16 column quads][64 keys][4] (r4_gemm_tc.cuh: kq_index)

// host: Wp [128 k][64 n] fp32 -> 3 splits of [64 n x 128 k] K-major core matrices
inline void build_scores_image(const float* Wp, uint8_t* img) {
  for (int sp = 0; sp < 3; ++sp)
    for (int n = 0; n < S_N; ++n)
      for (int k = 0; k < S_K; ++k) {
        float w = Wp[(size_t)k * S_N + n];
        uint16_t hi = host_bf16_bits(w);
        float r1 = w - host_bf16_val(hi);
        uint16_t mid = host_bf16_bits(r1);
        uint16_t lo = host_bf16_bits(r1 - host_bf16_val(mid));
        uint16_t v = sp == 0 ? hi : (sp == 1 ? mid : lo);
        memcpy(img + (size_t)sp * S_B_SPLIT + (n / 8) * S_SBO + (k / 8) * LBO + (n % 8) * 16 + (k % 8) * 2, &v, 2);
      }
}

struct ScoreTcSeq {
  const float* qa;       // [R, 64]  q (Wq+Wd) + b1, from k_query
  const float* H;        // [n_cached, 64, 128]
  const float* Kp;       // [n_cached, 64, 64]   k_t (Wk - Wd)
  const uint8_t* WpImg;  // S_B_BYTES
  const float* Wqd;      // [128, 64]
  const float* b1;       // [64]
  const float* W2;       // [64, 16]
  const float* b2;       // [16]
  const float* kv;       // [16]
  float bk;
  float* scoresT;        // [ceil(R/128), 64, 128]
  int shared;
};
struct ScoreTcParams {
  ScoreTcSeq s[2];
  const float* q;        // [R, 128]  mean of the 10 slate embeddings, from k_query
  int R, row0, div;
};

// q = reduce_mean(E_s[cat[-10:]]) and qa_i = q (Wq_i + Wd_i) + b1_i for both sequences (nets/utils.py:114-115 and
// the query half of :121-122).  8 rows per CTA, 128 threads.  Keeping this out of k_scores_tc2 takes two dependent
// HBM round trips (category ids -> embedding rows) and a 128-long serial FMA chain off its per-tile critical path.
__global__ void __launch_bounds__(128) k_query(int R, const int32_t* __restrict__ cat, const float* __restrict__ emb_seq,
                                               const float* __restrict__ Wqd0, const float* __restrict__ b10,
                                               const float* __restrict__ Wqd1, const float* __restrict__ b11,
                                               float* __restrict__ q_out, float* __restrict__ qa0, float* __restrict__ qa1) {
  __shared__ float q_s[8][S_K];
  const int tid = threadIdx.x, r0 = blockIdx.x * 8;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    int r = min(r0 + i, R - 1);
    const int32_t* crow = cat + (size_t)r * 21;
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < 10; ++j) acc += __ldg(emb_seq + (size_t)crow[11 + j] * S_K + tid);
    acc = acc / 10.0f;
    q_s[i][tid] = acc;
    if (r0 + i < R) q_out[(size_t)(r0 + i) * S_K + tid] = acc;
  }
  __syncthreads();
  const int sq = tid >> 6, j = tid & 63;
  const float* W = sq ? Wqd1 : Wqd0;
  float acc[8];
  const float b = __ldg((sq ? b11 : b10) + j);
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = b;
  // 16 weight loads in flight per thread (with 4 the 128-long loop was 32 exposed L2 round trips; the kernel sits between
  // k_assemble and k_scores_tc2 on the critical path of every pass)
  for (int k0 = 0; k0 < S_K; k0 += 16) {
    float w[16];
#pragma unroll
    for (int u = 0; u < 16; ++u) w[u] = __ldg(W + (k0 + u) * S_N + j);
#pragma unroll
    for (int u = 0; u < 16; ++u)
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] = fmaf(q_s[i][k0 + u], w[u], acc[i]);
  }
  float* o = sq ? qa1 : qa0;
#pragma unroll
  for (int i = 0; i < 8; ++i) if (r0 + i < R) o[(size_t)(r0 + i) * S_N + j] = acc[i];
}

// packed fp32 pairs (sm_100+): each lane rounds like the scalar instruction
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
  float2 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(reinterpret_cast<uint64_t&>(d)) : "l"(reinterpret_cast<uint64_t&>(a)), "l"(reinterpret_cast<uint64_t&>(b)));
  return d;
}
__device__ __forceinline__ float2 fsub2(float2 a, float2 b) {
  float2 d;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(reinterpret_cast<uint64_t&>(d)) : "l"(reinterpret_cast<uint64_t&>(a)), "l"(reinterpret_cast<uint64_t&>(b)));
  return d;
}
// x = hi + lo with hi = bf16(x) (round to nearest) and lo = bf16(x - hi), for a pair: the bf16 pair words (low half = .x)
__device__ __forceinline__ void split2(float2 x, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(x.x, x.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  const float2 hf = make_float2(__uint_as_float(hi << 16), __uint_as_float(hi & 0xffff0000u));
  const float2 r = fsub2(x, hf);
  const __nv_bfloat162 l = __floats2bfloat162_rn(r.x, r.y);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(nthreads) : "memory");
}

// ------------------------------------------------------------------------------------------------
// k_scores_tc2 -- both attention layers on the tensor pipe.
//
// Layer 1: the only GEMM-shaped term, (q*k_t) Wp, is a [64 keys x 128] x [128 x 64] product per (row, sequence).  Two
// feature rows are stacked into one UMMA tile (M = 128 key rows, N = 64, K = 128).  Persistent CTAs loop over tiles;
// producer warps build A = q*H as bf16 hi/lo core matrices in shared memory (double buffered), one lane issues 5 MMAs per
// K16 slice (A hi/lo x Wp hi/mid/lo: 2-way x 3-way split, smallest products first), fp32 accumulation in TMEM.
// Layer 2 (64 -> 16) is a second GEMM  [128 rows x 64] x [64 x 16]  instead of FMAs in the epilogue.  With the FMA form
// each epilogue warp was ONE dependency chain of ~800 instructions per tile (256 FFMA2 + 128 LDS.128 of W2 rows + 32
// sigmoids; ncu, round 2, profiles/r02_k_scores_tc_ncu.txt: 11.6 cycles per issued instruction, the largest stall the
// shared-memory scoreboard), and that chain, not HBM, set the tile period: 158.8 us per 4096-row pass against 90.8 us
// for this form.  The epilogue threads only produce z1 = sigmoid(first layer) and hand it to the MMA warp:
//   * A operand IN TENSOR MEMORY (tcgen05.mma ... [d], [a], b-desc: lane = row, 32-bit column c of a K16 slice = the bf16
//     pair (k = 2c, 2c + 1); layout confirmed by tools/ts_probe.cu): a thread packs its 16 activations as bf16 hi / lo
//     pairs and writes them with two tcgen05.st into its own TMEM lane -- no shared memory, no proxy fence, and the four
//     warps of a lane quarter (16 hidden units each) simply fill different columns;
//   * B operand = W2 as bf16 hi / mid / lo K-major core matrices (6 KB, appended to the Wp image), 5 MMAs per K16 slice in
//     the order of the first layer: same 2-way x 3-way split, fp32 accumulation in TMEM;
//   * the second-layer tail (16 sigmoids . kv) of tile i runs after the thread has produced z1 of tile i + 1, so nobody
//     waits for the MMA warp in steady state; the MMA warp issues layer 1 of tile i + 1 before layer 2 of tile i.
// Loads roll one tile ahead in both roles: a register that has been consumed is refilled with the next tile's value at
// once (H and q for the producers, the cached key half and q(Wq+Wd)+b1 for the epilogue), no extra registers.
// TMEM (512 columns): [0,128) two first-layer accumulators, [128,256) two A2 buffers (32 hi + 32 lo columns each),
// [256,288) two second-layer accumulators.
// ------------------------------------------------------------------------------------------------
constexpr int S_W2_SPLIT = AH2_N * S_N * 2;        // 2 KB per split: [16 n x 64 k] K-major core matrices
constexpr int S_W2_BYTES = 3 * S_W2_SPLIT;         // 6 KB, resident behind the Wp image
constexpr int S_W2_SBO = (S_N / 8) * 128;          // 1024: 8-row groups of the W2 image
constexpr int S_IMG_BYTES = S_B_BYTES + S_W2_BYTES;    // what build_scores_image2 writes and the loader warp copies
constexpr int S2_SMEM_BYTES = 2 * S_A_STAGE + S_IMG_BYTES + 1024;
constexpr int S2_TC_A2 = 2 * S_N;                  // TMEM columns
constexpr int S2_TC_D2 = S2_TC_A2 + 2 * S_N;

// host: Wp image followed by W2 [64 k][16 n] fp32 -> 3 splits of [16 n x 64 k] K-major core matrices
inline void build_scores_image2(const float* Wp, const float* W2, uint8_t* img) {
  build_scores_image(Wp, img);
  uint8_t* w2 = img + S_B_BYTES;
  for (int sp = 0; sp < 3; ++sp)
    for (int n = 0; n < AH2_N; ++n)
      for (int k = 0; k < S_N; ++k) {
        float w = W2[(size_t)k * AH2_N + n];
        uint16_t hi = host_bf16_bits(w);
        float r1 = w - host_bf16_val(hi);
        uint16_t mid = host_bf16_bits(r1);
        uint16_t lo = host_bf16_bits(r1 - host_bf16_val(mid));
        uint16_t v = sp == 0 ? hi : (sp == 1 ? mid : lo);
        memcpy(w2 + (size_t)sp * S_W2_SPLIT + (n / 8) * S_W2_SBO + (k / 8) * LBO + (n % 8) * 16 + (k % 8) * 2, &v, 2);
      }
}

// D[tmem] (+)= A[tmem] . B[smem desc]: the A operand read from tensor memory
__device__ __forceinline__ void mma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t db, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
               :: "r"(tmem_d), "r"(tmem_a), "l"(db), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void tmem_st8u(uint32_t taddr, const uint32_t* u) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               :: "r"(taddr), "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]) : "memory");
}

constexpr int S2_PROD_WARPS = 8, S2_EPI_WARPS = 16;          // 16 epilogue warps: 4 TMEM lane quarters x 4 column quarters of 16 hidden units
constexpr int S2_W_MMA = S2_PROD_WARPS + S2_EPI_WARPS, S2_W_LOAD = S2_W_MMA + 1;
constexpr int S2_THREADS = (S2_W_LOAD + 1) * 32;               // 832: 7 warps on the fullest scheduler -> 72 registers per thread

// DBG (tools/scores_probe.cu only): dbg[0..15] = cycles CTA (0, 0) spent per role and phase, summed over its tiles:
//   producer thread 0:  [0] bar.sync (q rows)  [1] wait A stage free  [2] convert + store
//   MMA leader:         [4] wait A full  [5] wait accumulators free  [6] issue layer 1  [7] wait A2 full  [8] issue layer 2
//   epilogue thread 0:  [10] wait layer-1 accumulators  [11] z1 + pack  [12] wait A2 free + store  [13] tail
// How many of `ctas` CTAs walk sequence 0 (the rest walk sequence 1).  A sequence whose cached rows are SHARED by all feature
// rows (Slate's constant second sequence) streams nothing from HBM and its tiles finish sooner (tools/scores_probe.cu): it
// gets the smaller share, `shared_pct` per cent of an even split's.
__host__ __device__ inline int scores_grid_split(int ctas, int ntiles, int shared0, int shared1, int shared_pct) {
  if (ctas < 2) return ctas;
  int n0 = ctas / 2;
  if (shared0 != shared1) {
    const int small = max(1, (ctas / 2) * shared_pct / 100);
    n0 = shared1 ? ctas - small : small;
  }
  (void)ntiles;
  return n0;
}

template <bool DBG>
__global__ void __launch_bounds__(S2_THREADS, 1) k_scores_tc2(ScoreTcParams p, int n0, long long* dbg = nullptr) {
  // 1-D grid: CTAs [0, n0) walk the tiles of sequence 0, CTAs [n0, gridDim.x) those of sequence 1 (scores_grid_split)
  const int sq = (int)blockIdx.x >= n0 ? 1 : 0;
  const int bx = (int)blockIdx.x - (sq ? n0 : 0), nbx = sq ? (int)gridDim.x - n0 : n0;
  const bool probe = DBG && dbg != nullptr && bx == 0;
  if (DBG && dbg) dbg += 16 * sq;
  long long acc[5] = {0, 0, 0, 0, 0};
  auto clk = [&]() -> long long { return DBG ? clock64() : 0; };
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sA = smem;                           // 2 stages x (hi, lo)
  uint8_t* sB = smem + 2 * S_A_STAGE;           // Wp hi/mid/lo, then W2 hi/mid/lo
  __shared__ uint64_t bar_afull[2], bar_aempty[2], bar_tfull[2], bar_tempty[2], bar_a2full[2], bar_t2full[2], bar_w;
  __shared__ uint32_t tmem_base_s;
  __shared__ float b2_s[AH2_N], kv_s[AH2_N];
  __shared__ __align__(16) float qa_s[2][2 * S_N];      // q (Wq+Wd) + b1 of the tile's two feature rows, double buffered
  __shared__ __align__(16) float q_s[2][2 * S_K];       // the two query rows themselves (producers), double buffered
  const ScoreTcSeq& S = p.s[sq];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ntiles = (p.R + 1) / 2;

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bar_afull[i], S2_PROD_WARPS * 32); mbar_init(&bar_aempty[i], 1);
      mbar_init(&bar_tfull[i], 1); mbar_init(&bar_tempty[i], S2_EPI_WARPS * 32);
      mbar_init(&bar_a2full[i], S2_EPI_WARPS * 32); mbar_init(&bar_t2full[i], 1);
    }
    mbar_init(&bar_w, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == S2_W_MMA) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (tid < AH2_N) { b2_s[tid] = __ldg(S.b2 + tid); kv_s[tid] = __ldg(S.kv + tid); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = tmem_base_s;

  if (warp == S2_W_LOAD) {
    if (lane == 0) {                                   // Wp + W2 images: once per CTA
      mbar_expect_tx(&bar_w, S_IMG_BYTES);
      bulk_g2s(sB, S.WpImg, S_IMG_BYTES, &bar_w);
    }
  } else if (warp == S2_W_MMA) {
    // ===== MMA issuer: the whole warp walks the tiles in uniform control flow, one elected lane issues (the
    // `if (lane == 0)` form wraps every tcgen05.mma in an ELECT / BRA.U.ANY convergence loop: r4_augru_pair2.cuh) =====
    const uint32_t leader = elect_one();
    constexpr uint32_t idesc = make_idesc(TM, S_N), idesc2 = make_idesc(TM, AH2_N);
    mbar_wait(&bar_w, 0);
    const uint32_t b0 = smem_u32(sB), w0 = b0 + S_B_BYTES;
    auto layer2 = [&](int it2) {                       // second layer of tile number it2 of this CTA
      const int s2 = it2 & 1;
      const long long c0 = clk();
      mbar_wait(&bar_a2full[s2], (it2 >> 1) & 1);
      tc_fence_after();
      const long long c1 = clk();
      const uint32_t ah = tbase + S2_TC_A2 + s2 * S_N, al = ah + S_N / 2;
      const uint32_t d2 = tbase + S2_TC_D2 + s2 * AH2_N;
      if (leader) {
#pragma unroll
        for (int j = 0; j < S_N / 16; ++j) {
          const uint32_t ko = j * 2 * LBO;
          const uint64_t wh = make_desc(w0 + ko, LBO, S_W2_SBO), wm = make_desc(w0 + S_W2_SPLIT + ko, LBO, S_W2_SBO);
          const uint64_t wl = make_desc(w0 + 2 * S_W2_SPLIT + ko, LBO, S_W2_SBO);
          mma_bf16_ts(d2, al + j * 8, wm, idesc2, j ? 1u : 0u);
          mma_bf16_ts(d2, ah + j * 8, wl, idesc2, 1u);
          mma_bf16_ts(d2, al + j * 8, wh, idesc2, 1u);
          mma_bf16_ts(d2, ah + j * 8, wm, idesc2, 1u);
          mma_bf16_ts(d2, ah + j * 8, wh, idesc2, 1u);
        }
        umma_commit(&bar_t2full[s2]);
      }
      __syncwarp();
      if (DBG) { acc[3] += c1 - c0; acc[4] += clk() - c1; }
    };
    int it = 0;
    for (int tile = bx; tile < ntiles; tile += nbx, ++it) {
      const int s = it & 1;
      const uint32_t ph = (it >> 1) & 1;
      const long long c0 = clk();
      mbar_wait(&bar_afull[s], ph);
      const long long c1 = clk();
      mbar_wait(&bar_tempty[s], ph ^ 1);
      tc_fence_after();
      const long long c2 = clk();
      if (leader) {
        const uint32_t a0 = smem_u32(sA + s * S_A_STAGE);
        const uint32_t d = tbase + s * S_N;
#pragma unroll
        for (int j = 0; j < S_K / 16; ++j) {
          const uint32_t ko = j * 2 * LBO, ka = j * 2 * S_A_LBO;
          uint64_t ah = make_desc(a0 + ka, S_A_LBO, S_A_SBO), al = make_desc(a0 + S_A_SPLIT + ka, S_A_LBO, S_A_SBO);
          uint64_t bh = make_desc(b0 + ko, LBO, S_SBO), bm = make_desc(b0 + S_B_SPLIT + ko, LBO, S_SBO);
          uint64_t bl = make_desc(b0 + 2 * S_B_SPLIT + ko, LBO, S_SBO);
          mma_bf16(d, al, bm, idesc, j ? 1u : 0u);
          mma_bf16(d, ah, bl, idesc, 1u);
          mma_bf16(d, al, bh, idesc, 1u);
          mma_bf16(d, ah, bm, idesc, 1u);
          mma_bf16(d, ah, bh, idesc, 1u);
        }
        umma_commit(&bar_aempty[s]);
        umma_commit(&bar_tfull[s]);
      }
      __syncwarp();
      if (DBG) { acc[0] += c1 - c0; acc[1] += c2 - c1; acc[2] += clk() - c2; }
      if (it > 0) layer2(it - 1);
    }
    if (it > 0) layer2(it - 1);
    if (probe && leader) for (int i = 0; i < 5; ++i) dbg[4 + i] = acc[i];
  } else if (warp < S2_PROD_WARPS) {
    // ===== producers: A = q * H as bf16 hi/lo.  Load g = 0..15 of a thread: K block kb = g % 4, row group g / 4; a warp reads
    // 4 rows x 128 contiguous bytes per 128-bit load (lane = row lane / 8, 16-byte piece lane % 8): whole lines, 4 L1
    // wavefronts per warp load (a (row, 32-byte chunk) mapping reads half of every sector per load: 8 wavefronts).
    // A thread therefore owns HALF a core-matrix row (4 of its 8 K values) and stores it with one 64-bit store per split; with
    // the 160-byte K stride the 32 half rows of a warp store (4 rows x 4 chunks x 2 halves) cover every bank exactly twice.
    // Eight loads are in flight per thread: load g + 8 is issued into the register load g has just been consumed from.
    // (Pulling the next tile's lines into L2 a tile period early measured 90.1 against 90.3 us per pass: the producers of
    // an HBM-fed sequence are capped by what one SM's L1 keeps in flight, 11.5 B/clk, not by DRAM latency.)
    const int prow = warp * 4 + (lane >> 3), piece = lane & 7;
    // the 16 loads of a tile are constant offsets from two row bases (feature rows 2 tile, 2 tile + 1): g / 8 picks the
    // feature row, (g / 4) % 2 the upper 32 keys, g % 4 the K block
    auto hbase = [&](int tile, int fr) {
      const int r = min(tile * 2 + fr, p.R - 1);
      const size_t ci = S.shared ? 0 : (size_t)((p.row0 + r) / p.div);
      return S.H + (ci * S_KEYS + prow) * S_K + piece * 4;
    };
    auto hoff = [](int g) { return ((g >> 2) & 1) * 32 * S_K + (g & 3) * 32; };
    auto qptr = [&](int tile) {
      const int r = min(tile * 2 + (tid >> 5), p.R - 1);
      return reinterpret_cast<const float4*>(p.q + (size_t)r * S_K) + (tid & 31);
    };
    float4 hv[8];
    float4 qreg = make_float4(0.f, 0.f, 0.f, 0.f);
    {
      const float* h0 = hbase(bx, 0);
#pragma unroll
      for (int g = 0; g < 8; ++g) hv[g] = __ldg(reinterpret_cast<const float4*>(h0 + hoff(g)));
      if (tid < 64) qreg = __ldg(qptr(bx));
    }
    int it = 0;
    for (int tile = bx; tile < ntiles; tile += nbx, ++it) {
      const int s = it & 1;
      const uint32_t ph = (it >> 1) & 1;
      const int tn = tile + nbx;
      const bool more = tn < ntiles;
      if (tid < 64) {                              // the tile's two query rows: 2 x 128 floats, loaded one tile ahead
        reinterpret_cast<float4*>(q_s[s])[tid] = qreg;
        if (more) qreg = __ldg(qptr(tn));
      }
      const long long c0 = clk();
      named_bar_sync(3, S2_PROD_WARPS * 32);       // q_s[s] is complete; it is rewritten two tiles later
      const long long c1 = clk();
      mbar_wait(&bar_aempty[s], ph ^ 1);          // MMA finished reading this A stage
      const long long c2 = clk();
      uint8_t* a = sA + s * S_A_STAGE;
      const float* h1 = hbase(tile, 1);            // second feature row of this tile (loads 8..15)
      const float* hn = hbase(more ? tn : tile, 0);   // first feature row of the next tile
#pragma unroll
      for (int g = 0; g < 16; ++g) {
        const int m = (g >> 2) * 32 + prow;
        const int k = (g & 3) * 32 + piece * 4;
        const float4 q0 = *reinterpret_cast<const float4*>(q_s[s] + (m >> 6) * S_K + k);
        const float4 h0 = hv[g & 7];
        if (g < 8) hv[g & 7] = __ldg(reinterpret_cast<const float4*>(h1 + hoff(g + 8)));
        else if (more) hv[g & 7] = __ldg(reinterpret_cast<const float4*>(hn + hoff(g - 8)));
        uint32_t hi01, lo01, hi23, lo23;
        split2(fmul2(make_float2(h0.x, h0.y), make_float2(q0.x, q0.y)), hi01, lo01);
        split2(fmul2(make_float2(h0.z, h0.w), make_float2(q0.z, q0.w)), hi23, lo23);
        const uint32_t off = (uint32_t)(m / 8) * S_A_SBO + (uint32_t)(k / 8) * S_A_LBO + (uint32_t)(m % 8) * 16 + (uint32_t)(k % 8) * 2;
        *reinterpret_cast<uint2*>(a + off) = make_uint2(hi01, hi23);
        *reinterpret_cast<uint2*>(a + S_A_SPLIT + off) = make_uint2(lo01, lo23);
      }
      proxy_fence();
      mbar_arrive(&bar_afull[s]);
      if (DBG) { acc[0] += c1 - c0; acc[1] += c2 - c1; acc[2] += clk() - c2; }
    }
    if (probe && tid == 0) for (int i = 0; i < 3; ++i) dbg[i] = acc[i];
  } else if (warp < S2_W_MMA) {
    // ===== epilogue: lane = key row of the tile; the four warps of a TMEM lane quarter take 16 hidden units of the first
    // attention layer each (jq = 0..3) and write their columns of the second GEMM's A operand; the 16-wide tail of tile i is
    // run, one tile behind, by column quarter i % 4. =====
    const int e = (tid - S2_PROD_WARPS * 32) & 127;  // row of the tile: 0..127
    const int jq = (tid - S2_PROD_WARPS * 32) >> 7;  // column quarter
    const int ew = e >> 5;                       // TMEM lane quarter (= warp % 4)
    const int rr = e >> 6, key = e & 63;
    const int j0 = jq * (S_N / 4);
    const uint32_t tl = tbase + ((uint32_t)(ew * 32) << 16);
    auto kptr = [&](int tile) {
      const int rc = min(tile * 2 + rr, p.R - 1);
      const size_t ci = S.shared ? 0 : (size_t)((p.row0 + rc) / p.div);
      return reinterpret_cast<const float4*>(S.Kp + kq_index(ci, S_N / 4, j0 / 4, S_KEYS, key));   // quad jq4 at [jq4 * 64]
    };
    auto tail = [&](int it2, int tile2) {            // second-layer tail of this CTA's tile number it2
      const int s2 = it2 & 1;
      mbar_wait(&bar_t2full[s2], (it2 >> 1) & 1);
      tc_fence_after();
      float o[AH2_N];
      tmem_ld16(tl + S2_TC_D2 + s2 * AH2_N, o);
      tmem_wait_ld();
      float sc = S.bk;
#pragma unroll
      for (int jj = 0; jj < AH2_N; ++jj) sc = fmaf(fast_sigmoid(o[jj] + b2_s[jj]), kv_s[jj], sc);
      const int r2 = tile2 * 2 + rr;
      if (r2 < p.R) S.scoresT[((size_t)(r2 >> 7) * S_KEYS + key) * 128 + (r2 & 127)] = sc;
    };
    float4 kk[S_N / 16];
    float qa_next = 0.f;
    {
      const float4* kp = kptr(bx);
#pragma unroll
      for (int j = 0; j < S_N / 16; ++j) kk[j] = __ldg(kp + j * S_KEYS);
      if (jq == 0) qa_next = __ldg(S.qa + (size_t)min(bx * 2 + rr, p.R - 1) * S_N + key);
    }
    int it = 0, prev_tile = 0;
    for (int tile = bx; tile < ntiles; tile += nbx, ++it) {
      const int s = it & 1;
      const uint32_t ph = (it >> 1) & 1;
      const int tn = tile + nbx;
      const bool more = tn < ntiles;
      if (jq == 0) {
        qa_s[s][e] = qa_next;
        if (more) qa_next = __ldg(S.qa + (size_t)min(tn * 2 + rr, p.R - 1) * S_N + key);
      }
      named_bar_sync(2, S2_EPI_WARPS * 32);        // epilogue warps only; buffer s is rewritten two tiles later
      const long long c0 = clk();
      mbar_wait(&bar_tfull[s], ph);
      tc_fence_after();
      const long long c1 = clk();
      float z[16];
      tmem_ld16(tl + s * S_N + j0, z);
      tmem_wait_ld();
      tc_fence_before();
      mbar_arrive(&bar_tempty[s]);               // first-layer accumulators are free again
      const float* qap = qa_s[s] + rr * S_N + j0;
      const float4* kpn = kptr(more ? tn : tile);
      uint32_t zh[8], zl[8];
#pragma unroll
      for (int j = 0; j < 16; j += 4) {
        const float4 kq = kk[j / 4];
        if (more) kk[j / 4] = __ldg(kpn + (j / 4) * S_KEYS);   // rolling refill: the next tile's cached key half
        const float4 qq = *reinterpret_cast<const float4*>(qap + j);
        const float a0 = fast_sigmoid(z[j] + qq.x + kq.x), a1 = fast_sigmoid(z[j + 1] + qq.y + kq.y);
        const float a2 = fast_sigmoid(z[j + 2] + qq.z + kq.z), a3 = fast_sigmoid(z[j + 3] + qq.w + kq.w);
        split2(make_float2(a0, a1), zh[j / 2], zl[j / 2]);             // .x = low half = even k
        split2(make_float2(a2, a3), zh[j / 2 + 1], zl[j / 2 + 1]);
      }
      // A2 buffer s was read by the second-layer MMAs of tile it - 2: wait for their commit (the warps that ran that tile's
      // tail already have)
      const long long c2 = clk();
      if (it >= 2) { mbar_wait(&bar_t2full[s], ((it - 2) >> 1) & 1); tc_fence_after(); }
      const uint32_t ta = tl + S2_TC_A2 + s * S_N + jq * 8;
      tmem_st8u(ta, zh);
      tmem_st8u(ta + S_N / 2, zl);
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(&bar_a2full[s]);
      const long long c3 = clk();
      if (it > 0 && jq == ((it - 1) & 3)) tail(it - 1, prev_tile);
      prev_tile = tile;
      if (DBG) { acc[0] += c1 - c0; acc[1] += c2 - c1; acc[2] += c3 - c2; acc[3] += clk() - c3; }
    }
    if (it > 0 && jq == ((it - 1) & 3)) tail(it - 1, prev_tile);
    if (probe && tid == S2_PROD_WARPS * 32) for (int i = 0; i < 4; ++i) dbg[10 + i] = acc[i];
  }
  tc_fence_before();
  __syncthreads();
  if (warp == S2_W_MMA) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tbase), "r"(512));
}

}  // namespace r4tc
