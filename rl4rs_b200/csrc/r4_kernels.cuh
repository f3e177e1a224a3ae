// r4_kernels.cuh -- sm_100a kernels of the RL4RS hot path (SURVEY.md section 2a): the integer / gather half
// (K1-K5, K10 tail, K11).  The GEMM-shaped half lives in r4_gemm_tc.cuh, r4_gru_tc.cuh, r4_scores_tc.cuh,
// r4_augru_pair2.cuh, r4_augru_pp.cuh (tcgen05) and the policy/learner in r4_ppo.cuh.
//
// Every kernel cites the reference operation it replaces.  Arithmetic is fp32 with precise
// expf/tanhf/expm1f (parity: 1e-4 relative against the f32 CPU oracle); reward and kNN scores are
// f64 like the reference (slate.py:188,302).  Layouts are described in DESIGN.md section 3.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace r4 {

constexpr int EMB = 128;        // emb_size
constexpr int MAXLEN = 64;      // maxlen
constexpr int NCAT = 21;        // category_feature_num
constexpr int NDENSE = 432;     // dense_feature_num
constexpr int VEC = 40;         // item vector width (item_info.csv)
constexpr int UD = 32;          // user dense floats  (user_protrait[10:])
constexpr int UC = 10;          // user categorical ids (user_protrait[:10])
constexpr int PAGE = 9;         // page_items
constexpr int HU = 128;         // hidden_units (dense tower)
constexpr int AH1 = 64;         // attention MLP hidden 1
constexpr int AH2 = 16;         // attention MLP hidden 2
constexpr int AUH = 256;        // AUGRU hidden (emb_size * 2, nets/utils.py:123)
constexpr int OBSD = 256;       // simulator_obs width (dien.py:35, dnn.py:35)
constexpr int OBSD_WD = 2 * EMB + HU + NCAT * EMB;   // 3072: widedeep's simulator_obs is the concat itself (widedeep.py:35-37)
constexpr int ALLF = 2 * AUH + HU + EMB + NCAT * EMB;   // 3456, dien.py:34
constexpr int XIN_LD = 3 * EMB;                          // GRU-1 input projection: [r|u|c] = 384
constexpr int XK_LD = 2 * AUH + AUH + AH1;               // AUGRU input proj [r|u (512) | c (256) | key (64)] = 832
constexpr int XK_C = 2 * AUH;                            // offset of candidate part
constexpr int XK_K = 3 * AUH;                            // offset of attention key part
constexpr int MAX_WORDS = 16;                            // action_size <= 512

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }
__device__ __forceinline__ float eluf_(float x) { return x > 0.f ? x : expm1f(x); }
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// location_mask rows (slate.py:60-64): layer 0 = ids 1..39, 1 = 40..147, 2 = 148.., 3 = {0}
__device__ __forceinline__ bool loc_allowed(int layer, int a) {
  switch (layer) {
    case 0: return a >= 1 && a < 40;
    case 1: return a >= 40 && a < 148;
    case 2: return a >= 148;
    default: return a == 0;
  }
}

// ------------------------------------------------------------------------------------------
// K1 reset: SlateState.__init__ (slate.py:16-19): prev_actions = 0, masks = 1
// ------------------------------------------------------------------------------------------
__global__ void k_init_state(int B, int T, int A, int words, int32_t* prev_actions, uint32_t* amask,
                             uint8_t* sflag, uint8_t* mask_out /*[B,A] or null*/, int layer0) {
  int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (b >= B) return;
  for (int t = lane; t < T; t += 32) prev_actions[(size_t)b * T + t] = 0;
  for (int w = lane; w < words; w += 32) {
    int lo = w * 32;
    uint32_t bits = (A - lo >= 32) ? 0xffffffffu : ((A - lo) <= 0 ? 0u : ((1u << (A - lo)) - 1u));
    amask[(size_t)b * words + w] = bits;
  }
  if (lane == 0) sflag[b] = 0;
  if (mask_out)
    for (int a = lane; a < A; a += 32) mask_out[(size_t)b * A + a] = loc_allowed(layer0, a) ? 1 : 0;
}

// ------------------------------------------------------------------------------------------
// K1 + K2  SlateState.act (slate.py:193-202) / SeqSlateState.act (seqslate.py:92-102,124-126)
// one warp per env row.  Conti mode resolves the action by masked kNN in f64 (slate.py:186-191):
// fill -2^31, first index wins ties.
// ------------------------------------------------------------------------------------------
struct ActParams {
  int B, T, P, A, words, seq, conti, emb_dim, cur_steps, act_f64;
};

__global__ void k_act(ActParams p, const void* __restrict__ action, const double* __restrict__ action_emb,
                      const uint8_t* __restrict__ special, int32_t* __restrict__ prev_actions,
                      uint32_t* __restrict__ amask, uint8_t* __restrict__ sflag,
                      int32_t* __restrict__ chosen_out, uint8_t* __restrict__ mask_out) {
  int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (b >= p.B) return;
  uint32_t* am = amask + (size_t)b * p.words;
  int32_t* pa = prev_actions + (size_t)b * p.T;
  int cur = p.cur_steps;
  int a_sel;
  if (p.conti) {
    int layer = p.seq ? (cur % p.P) / 3 : cur / 3;          // pre-act layer (Q4)
    bool sf = sflag[b] != 0;
    double best = -1e308;
    int besti = 0x7fffffff;
    const float* af = reinterpret_cast<const float*>(action) + (size_t)b * p.emb_dim;
    const double* ad = reinterpret_cast<const double*>(action) + (size_t)b * p.emb_dim;
    for (int a = lane; a < p.A; a += 32) {
      bool ok = ((am[a >> 5] >> (a & 31)) & 1u) && loc_allowed(layer, a) && !(sf && special[a]);
      double s;
      if (ok) {
        s = 0.0;
        const double* e = action_emb + (size_t)a * p.emb_dim;
        if (p.act_f64) { for (int k = 0; k < p.emb_dim; ++k) s += ad[k] * e[k]; }
        else { for (int k = 0; k < p.emb_dim; ++k) s += (double)af[k] * e[k]; }
      } else {
        s = -2147483648.0;
      }
      if (s > best) { best = s; besti = a; }
    }
    for (int o = 16; o > 0; o >>= 1) {
      double s2 = __shfl_xor_sync(0xffffffffu, best, o);
      int i2 = __shfl_xor_sync(0xffffffffu, besti, o);
      if (s2 > best || (s2 == best && i2 < besti)) { best = s2; besti = i2; }
    }
    a_sel = besti;
  } else {
    a_sel = reinterpret_cast<const int32_t*>(action)[b];
    a_sel = a_sel < 0 ? 0 : (a_sel >= p.A ? p.A - 1 : a_sel);   // memory safety; host validates
  }
  if (lane == 0) {
    pa[cur] = a_sel;                                           // slate.py:198
    am[a_sel >> 5] &= ~(1u << (a_sel & 31));                   // slate.py:199 (also for a == 0, Q5)
    if (chosen_out) chosen_out[b] = a_sel;
  }
  __syncwarp();
  // slate.py:200-202: special mask closes once the WHOLE history holds a special item (Q6, Q8)
  bool any_sp = false;
  for (int t = lane; t < p.T; t += 32) any_sp |= special[pa[t]] != 0;
  any_sp = __any_sync(0xffffffffu, any_sp);
  int nxt = cur + 1;
  bool page_reset = p.seq && (nxt % p.P == 0);                 // seqslate.py:124-126
  if (page_reset) {
    any_sp = false;
    for (int w = lane; w < p.words; w += 32) {
      int lo = w * 32;
      am[w] = (p.A - lo >= 32) ? 0xffffffffu : ((1u << (p.A - lo)) - 1u);
    }
    __syncwarp();
  }
  if (lane == 0) sflag[b] = any_sp ? 1 : 0;
  if (mask_out) {                                              // slate.py:93-97 / seqslate.py:15-17
    int layer = p.seq ? (nxt % p.P) / 3 : nxt / 3;
    for (int a = lane; a < p.A; a += 32) {
      bool ok = ((am[a >> 5] >> (a & 31)) & 1u) && loc_allowed(layer, a) && !(any_sp && special[a]);
      mask_out[(size_t)b * p.A + a] = ok ? 1 : 0;
    }
  }
}

// unmasked kNN (slate.py:180-184), one warp per query row
__global__ void k_knn_plain(int n, int A, int emb_dim, int act_f64, const void* __restrict__ action,
                            const double* __restrict__ action_emb, int32_t* __restrict__ out) {
  int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (b >= n) return;
  const float* af = reinterpret_cast<const float*>(action) + (size_t)b * emb_dim;
  const double* ad = reinterpret_cast<const double*>(action) + (size_t)b * emb_dim;
  double best = -1e308;
  int besti = 0x7fffffff;
  for (int a = lane; a < A; a += 32) {
    double s = 0.0;
    const double* e = action_emb + (size_t)a * emb_dim;
    if (act_f64) { for (int k = 0; k < emb_dim; ++k) s += ad[k] * e[k]; }
    else { for (int k = 0; k < emb_dim; ++k) s += (double)af[k] * e[k]; }
    if (s > best) { best = s; besti = a; }
  }
  for (int o = 16; o > 0; o >>= 1) {
    double s2 = __shfl_xor_sync(0xffffffffu, best, o);
    int i2 = __shfl_xor_sync(0xffffffffu, besti, o);
    if (s2 > best || (s2 == best && i2 < besti)) { best = s2; besti = i2; }
  }
  if (lane == 0) out[b] = besti;
}

// ------------------------------------------------------------------------------------------
// K3 feature assembly: the state rebuild of SlateState.act (slate.py:203-213) /
// SeqSlateState.act (seqslate.py:103-121) / get_complete_states (slate.py:117-131,
// seqslate.py:27-50) followed by FeatureUtil.feature_extraction's post-pad/truncate
// (datautil.py:52-65).  One warp per feature row; rows r0.. of the pass.
//   mode 0: initial state (slate.py:72-80)      rows = B
//   mode 1: state after act at step `step`      rows = B
//   mode 2: reward rows, env-row major          rows = B * rpe (rpe = T for Slate, P for SeqSlate)
// ------------------------------------------------------------------------------------------
struct AsmParams {
  int mode, B, T, P, seq, step, rpe, row0, nrows;
};

__global__ void k_assemble(AsmParams p, const int32_t* __restrict__ row_idx,
                           const int32_t* __restrict__ log_cat, const float* __restrict__ log_dense,
                           const float* __restrict__ item_vec, const int32_t* __restrict__ prev_actions,
                           int32_t* __restrict__ cat_out, float* __restrict__ dense_out) {
  int rl = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (rl >= p.nrows) return;
  int r = p.row0 + rl;
  int b = (p.mode == 2) ? r / p.rpe : r;
  int j = (p.mode == 2) ? r % p.rpe : 0;
  const int32_t* pa = prev_actions + (size_t)b * p.T;
  int64_t lr = row_idx[b];
  int W = 0, w0 = 0, sid = 0, cur_a = 0;
  if (p.mode != 0) {
    int st = (p.mode == 1) ? p.step : (p.seq ? p.step - p.P + j : j);   // step this row's state was built at
    if (p.seq) { w0 = st / p.P * p.P; W = p.P; sid = st / p.P + 1; }
    else { w0 = 0; W = p.T; sid = 1; }
    cur_a = pa[st];
  }
  int32_t* co = cat_out + (size_t)rl * NCAT;
  float* dn = dense_out + (size_t)rl * NDENSE;
  if (lane < NCAT) {
    int c = lane, v = 0;
    if (c < UC) v = log_cat[lr * UC + c];
    else if (p.mode != 0) {
      if (c == UC) v = sid;
      else if (c < UC + 1 + W) v = pa[w0 + c - UC - 1];
      else if (c == UC + 1 + W) v = cur_a;
    }
    co[c] = v;
  }
  for (int d = lane; d < NDENSE; d += 32) {
    float v = 0.f;
    if (d < UD) v = log_dense[lr * UD + d];
    else if (p.mode != 0) {
      int k = (d - UD) / VEC, e = (d - UD) % VEC;
      if (k < W) v = item_vec[(size_t)pa[w0 + k] * VEC + e];
      else if (k == W) v = item_vec[(size_t)cur_a * VEC + e];
    }
    dn[d] = v;
  }
}

// sequence ids: seq0 = user history (pre-padded in the log), seq1 = previous pages of the episode
// (seqslate.py:36-37,109-110 + pad_sequences at datautil.py:43-46) or zeros.
__global__ void k_seq_ids(int B, int T, int p0, const int32_t* __restrict__ row_idx,
                          const int32_t* __restrict__ log_seq, const int32_t* __restrict__ prev_actions,
                          int32_t* __restrict__ seq0 /*[B,64] or null*/, int32_t* __restrict__ seq1 /*[B,64] or null*/,
                          int32_t* __restrict__ seq_out /*[B,2,64] or null*/) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * MAXLEN) return;
  int b = i / MAXLEN, t = i % MAXLEN;
  int v0 = log_seq[(size_t)row_idx[b] * MAXLEN + t];
  int n = p0 < MAXLEN ? p0 : MAXLEN;                   // keep the last maxlen ids
  int v1 = 0;
  if (t >= MAXLEN - n) v1 = prev_actions[(size_t)b * T + (p0 - n) + (t - (MAXLEN - n))];
  if (seq0) seq0[i] = v0;
  if (seq1) seq1[i] = v1;
  if (seq_out) { seq_out[(size_t)b * 2 * MAXLEN + t] = v0; seq_out[(size_t)b * 2 * MAXLEN + MAXLEN + t] = v1; }
}

// ------------------------------------------------------------------------------------------
// K4 + K5 category features (nets/utils.py:16-25): E_c gather, tf.keras.layers.Attention()
// (softmax(Q K^T) V, no scale, no mask), GlobalAveragePooling1D, and the flattened embeddings.
// One warp per row; softmax rows are reduced with warp shuffles.  Writes the pooled attention straight into the
// head input: allf[r, 640:768] (row stride out_ld).  The Flatten() half of the category feature is NOT materialised:
// the head GEMM gathers those 21 x 128 values from the embedding table itself (r4_gemm_tc.cuh: A2 / gather2).
// mean_t(P emb) is evaluated as (mean_t P) emb -- same value up to fp32 rounding order.
// ------------------------------------------------------------------------------------------
constexpr int CAT_LD = 132;
constexpr int ALLF_LD = 2 * AUH + HU + EMB;    // 768: [sequence 512 | dense 128 | pooled category attention 128]
__global__ void __launch_bounds__(128) k_cat_attn(int R, const int32_t* __restrict__ cat,
                                                  const float* __restrict__ emb_cat, float* __restrict__ allf) {
  extern __shared__ __align__(16) float smem[];
  int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int r = blockIdx.x * 4 + w;
  float* e = smem + w * (NCAT * CAT_LD + NCAT * 24);     // [21][132]
  float* Ssm = e + NCAT * CAT_LD;                         // [21][24]
  if (r >= R) return;
  const int32_t* crow = cat + (size_t)r * NCAT;
  float* out = allf + (size_t)r * ALLF_LD;
  {                                  // ids with one coalesced load, then all 21 row gathers in flight together
    const int myid = lane < NCAT ? crow[lane] : 0;
    float4 v[NCAT];
#pragma unroll
    for (int j = 0; j < NCAT; ++j) v[j] = ldg4(emb_cat + (size_t)__shfl_sync(0xffffffffu, myid, j) * EMB + lane * 4);
#pragma unroll
    for (int j = 0; j < NCAT; ++j) *reinterpret_cast<float4*>(&e[j * CAT_LD + lane * 4]) = v[j];
  }
  __syncwarp();
  // S[t][j] = <e_t, e_j>, symmetric.  The 21 rows form 7 groups of 3; lane b < 28 owns the 3 x 3 block (gi <= gj) of the group
  // pair b: per 4 columns it reads 6 row quads (instead of 2 per PAIR in the first version: 462 128-bit shared loads per lane
  // against 192 here -- the kernel sat on the shared-memory pipe) and feeds 9 accumulators.  Every dot product is still the
  // same k-ascending fmaf chain, so the scores are bit-identical to the pair-per-lane form.
  if (lane < 28) {
    int gi = 0, rem = lane;
    while (rem >= 7 - gi) { rem -= 7 - gi; ++gi; }
    const int gj = gi + rem;
    const float* a = e + 3 * gi * CAT_LD;
    const float* b = e + 3 * gj * CAT_LD;
    float acc[3][3];
#pragma unroll
    for (int x = 0; x < 3; ++x)
#pragma unroll
      for (int y = 0; y < 3; ++y) acc[x][y] = 0.f;
#pragma unroll 4
    for (int k = 0; k < EMB; k += 4) {
      float4 av[3], bv[3];
#pragma unroll
      for (int x = 0; x < 3; ++x) {
        av[x] = *reinterpret_cast<const float4*>(a + x * CAT_LD + k);
        bv[x] = *reinterpret_cast<const float4*>(b + x * CAT_LD + k);
      }
#pragma unroll
      for (int x = 0; x < 3; ++x)
#pragma unroll
        for (int y = 0; y < 3; ++y) {
          float s = acc[x][y];
          s = fmaf(av[x].x, bv[y].x, s); s = fmaf(av[x].y, bv[y].y, s); s = fmaf(av[x].z, bv[y].z, s); s = fmaf(av[x].w, bv[y].w, s);
          acc[x][y] = s;
        }
    }
#pragma unroll
    for (int x = 0; x < 3; ++x)
#pragma unroll
      for (int y = 0; y < 3; ++y) {
        Ssm[(3 * gi + x) * 24 + 3 * gj + y] = acc[x][y];
        Ssm[(3 * gj + y) * 24 + 3 * gi + x] = acc[x][y];
      }
  }
  __syncwarp();
  float wcol = 0.f;      // lane j accumulates sum_t P[t][j]
  for (int t = 0; t < NCAT; ++t) {
    float v = lane < NCAT ? Ssm[t * 24 + lane] : -INFINITY;
    float m = v;
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float ex = lane < NCAT ? expf(v - m) : 0.f;
    float sum = ex;
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    wcol += ex / sum;
  }
  wcol = wcol / (float)NCAT;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int j = 0; j < NCAT; ++j) {
    float wj = __shfl_sync(0xffffffffu, wcol, j);
    float4 v = *reinterpret_cast<const float4*>(&e[j * CAT_LD + lane * 4]);
    acc.x = fmaf(wj, v.x, acc.x); acc.y = fmaf(wj, v.y, acc.y);
    acc.z = fmaf(wj, v.z, acc.z); acc.w = fmaf(wj, v.w, acc.w);
  }
  *reinterpret_cast<float4*>(out + 2 * AUH + HU + lane * 4) = acc;
}

// ------------------------------------------------------------------------------------------
// dnn simulator (nets/dnn.py:31, nets/utils.py:7-14): category_feature = GlobalAveragePooling1D(Embedding(cat)).
// THE gather kernel of the path: per feature row 21 x 512 B embedding rows in, 512 B out (SURVEY.md 8d: G_dnn).
// One warp per row, persistent grid.  The 21 rows of a feature row are staged into shared memory by the bulk-copy
// engine (cp.async.bulk, 1-D TMA): lanes 0..20 each issue ONE 512-byte copy for their id, all completing on the warp's
// mbarrier, two rows in flight per warp (double buffer) -- the loads of row i+1 are in the memory system while row i is
// reduced, with no registers tied up.  The reduction reads shared memory with 128-bit loads (lane = 4 columns) and
// writes the pooled row with one coalesced 512-byte store.  Sum order j = 0..20 then * (1/21) (fp32; the reference's
// reduce_mean is order-free up to rounding).
// ------------------------------------------------------------------------------------------
constexpr int POOL_WARPS = 4;
constexpr int POOL_SMEM = POOL_WARPS * 2 * NCAT * EMB * 4;          // 86 016 B: 2 CTAs per SM
__global__ void __launch_bounds__(POOL_WARPS * 32) k_cat_pool(int R, const int32_t* __restrict__ cat,
                                                              const float* __restrict__ emb_cat, float* __restrict__ out,
                                                              int out_ld) {
  extern __shared__ __align__(128) float pool_s[];
  __shared__ uint64_t bar[POOL_WARPS][2];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* buf = pool_s + (size_t)w * 2 * NCAT * EMB;
  const int gw = blockIdx.x * POOL_WARPS + w, nw = gridDim.x * POOL_WARPS;
  if (lane == 0) {
    for (int i = 0; i < 2; ++i)
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"((uint32_t)__cvta_generic_to_shared(&bar[w][i])), "r"(1) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  auto issue = [&](int r, int b) {
    const uint32_t mb = (uint32_t)__cvta_generic_to_shared(&bar[w][b]);
    if (lane == 0) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(mb), "r"(NCAT * EMB * 4) : "memory");
    __syncwarp();
    if (lane < NCAT) {
      const float* src = emb_cat + (size_t)__ldg(cat + (size_t)r * NCAT + lane) * EMB;
      const uint32_t dst = (uint32_t)__cvta_generic_to_shared(buf + ((size_t)b * NCAT + lane) * EMB);
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   :: "r"(dst), "l"(src), "r"(EMB * 4), "r"(mb) : "memory");
    }
  };
  int it = 0;
  if (gw < R) issue(gw, 0);
  for (int r = gw; r < R; r += nw, ++it) {
    const int b = it & 1;
    if (r + nw < R) issue(r + nw, b ^ 1);                       // buffer b^1 was consumed one iteration ago (program order)
    const uint32_t mb = (uint32_t)__cvta_generic_to_shared(&bar[w][b]);
    const uint32_t par = (uint32_t)((it >> 1) & 1);
    asm volatile("{\n\t.reg .pred p;\n\tPOOL_WAIT:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra POOL_DONE;\n\tbra POOL_WAIT;\n\tPOOL_DONE:\n\t}\n"
                 :: "r"(mb), "r"(par) : "memory");
    const float* e = buf + (size_t)b * NCAT * EMB + lane * 4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int j = 0; j < NCAT; ++j) {
      const float4 v = *reinterpret_cast<const float4*>(e + j * EMB);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    const float n = (float)NCAT;                                 // sum / count, like Eigen's MeanReducer / numpy.mean
    *reinterpret_cast<float4*>(out + (size_t)r * out_ld + lane * 4) = make_float4(acc.x / n, acc.y / n, acc.z / n, acc.w / n);
    __syncwarp();                                                // every lane has read buffer b before it is refilled
  }
}

// ------------------------------------------------------------------------------------------
// widedeep simulator (nets/widedeep.py:31-38): the two gather halves of its 3072-wide 'simulator_obs' concat.
//   k_seq_pool     sequence_input_concat (nets/utils.py:56-77): per sequence GlobalAveragePooling1D over the 64
//                  embedded positions (ONE shared table; pad id 0 is embedded and averaged like any id) -> [R, 2 x 128]
//   k_cat_flatten  id_input_processing_concat (nets/utils.py:38-45): Flatten(Embedding(cat)) -> obs[r, 384:3072]
// One warp per feature row, 128-bit loads, coalesced 512-byte stores.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_seq_pool(int R, const int32_t* __restrict__ seq /*[R,2,64]*/,
                                                  const float* __restrict__ emb_seq, float* __restrict__ out /*[R,256]*/) {
  const int r = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (r >= R) return;
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    const int32_t* ids = seq + ((size_t)r * 2 + s) * MAXLEN;
    const int id0 = __ldg(ids + lane), id1 = __ldg(ids + 32 + lane);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 8
    for (int t = 0; t < MAXLEN; ++t) {
      const int id = __shfl_sync(0xffffffffu, t < 32 ? id0 : id1, t & 31);
      const float4 v = ldg4(emb_seq + (size_t)id * EMB + lane * 4);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    const float n = (float)MAXLEN;
    *reinterpret_cast<float4*>(out + (size_t)r * 2 * EMB + s * EMB + lane * 4) = make_float4(acc.x / n, acc.y / n, acc.z / n, acc.w / n);
  }
}
// lstm simulator (nets/utils.py:78-97): the cached LAST states of the two sequence GRUs -> columns [0, 256) of the
// feature slab of a pass (pass row i -> cache row (row0 + i) / div, or row 0 of a shared one-row cache).
__global__ void k_seq_last_rows(int R, int row0, int div, const float* __restrict__ h0, int shared0,
                                const float* __restrict__ h1, int shared1, float* __restrict__ out, int ld) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;      // one thread = one float4 of one row: 64 per row
  if (i >= R * 64) return;
  const int r = i >> 6, c = (i & 63) * 4, s = c >= EMB;
  const int ci = (s ? shared1 : shared0) ? 0 : (row0 + r) / div;
  *reinterpret_cast<float4*>(out + (size_t)r * ld + c) = ldg4((s ? h1 : h0) + (size_t)ci * EMB + (c & (EMB - 1)));
}
// sequence ids of the rows of one simulator pass (pass row i -> env row (row0 + i) / div): seq0 = user history, seq1 = the
// items of the previous pages (seqslate.py:36-37,109-110) or zeros, as k_seq_ids
__global__ void k_seq_rows(int R, int row0, int div, int T, int p0, const int32_t* __restrict__ row_idx,
                           const int32_t* __restrict__ log_seq, const int32_t* __restrict__ prev_actions,
                           int32_t* __restrict__ out /*[R,2,64]*/) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= R * MAXLEN) return;
  const int rr = i / MAXLEN, t = i % MAXLEN;
  const int b = (row0 + rr) / div;
  const int n = p0 < MAXLEN ? p0 : MAXLEN;
  int v1 = 0;
  if (t >= MAXLEN - n) v1 = prev_actions[(size_t)b * T + (p0 - n) + (t - (MAXLEN - n))];
  out[(size_t)rr * 2 * MAXLEN + t] = log_seq[(size_t)row_idx[b] * MAXLEN + t];
  out[(size_t)rr * 2 * MAXLEN + MAXLEN + t] = v1;
}
__global__ void __launch_bounds__(128) k_cat_flatten(int R, const int32_t* __restrict__ cat, const float* __restrict__ emb_cat,
                                                     float* __restrict__ out, int out_ld) {
  const int r = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (r >= R) return;
  const int id = lane < NCAT ? __ldg(cat + (size_t)r * NCAT + lane) : 0;
#pragma unroll 7
  for (int j = 0; j < NCAT; ++j) {
    const int idj = __shfl_sync(0xffffffffu, id, j);
    *reinterpret_cast<float4*>(out + (size_t)r * out_ld + j * EMB + lane * 4) = ldg4(emb_cat + (size_t)idj * EMB + lane * 4);
  }
}

// ------------------------------------------------------------------------------------------
// K10 tail: probs = softmax(obs Wr + br) (dien.py:36); click prob = probs[:,1] (slate.py:298).
// One warp per row, warp-shuffle reduction of the two OBSD-long dots (OBSD = 256; 3072 for widedeep).
// ------------------------------------------------------------------------------------------
__global__ void k_reward_head(int R, const float* __restrict__ obs, const float* __restrict__ Wr,
                              const float* __restrict__ br, float* __restrict__ p1 /*[R] or null*/,
                              float* __restrict__ probs /*[R,2] or null*/, int OBSD = 256) {
  int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (r >= R) return;
  float z0 = 0.f, z1 = 0.f;
  for (int k = lane; k < OBSD; k += 32) {
    float o = obs[(size_t)r * OBSD + k];
    z0 = fmaf(o, __ldg(Wr + k * 2), z0);
    z1 = fmaf(o, __ldg(Wr + k * 2 + 1), z1);
  }
  for (int o = 16; o > 0; o >>= 1) {
    z0 += __shfl_xor_sync(0xffffffffu, z0, o);
    z1 += __shfl_xor_sync(0xffffffffu, z1, o);
  }
  if (lane == 0) {
    z0 += br[0]; z1 += br[1];
    float m = fmaxf(z0, z1);
    float e0 = expf(z0 - m), e1 = expf(z1 - m);
    float s = e0 + e1;
    if (p1) p1[r] = e1 / s;
    if (probs) { probs[(size_t)r * 2] = e0 / s; probs[(size_t)r * 2 + 1] = e1 / s; }
  }
}

// ------------------------------------------------------------------------------------------
// K11 violation (slate.py:133-147 / seqslate.py:52-69) and reward (slate.py:293-308 /
// seqslate.py:147-157).  One thread per env row.
// ------------------------------------------------------------------------------------------
__device__ inline int violation_row(const int32_t* pa, int cur, int P, int seq, const uint8_t* special) {
  int ok = 1;
  for (int s = 0; s < cur; ++s) {
    int layer = seq ? (s % P) / 3 : s / 3;
    ok &= loc_allowed(layer, pa[s]) ? 1 : 0;
  }
  int n1 = cur - 1 > 1 ? cur - 1 : 1;                       // range(max(cur-1, 1))  (Q7)
  for (int s = 0; s < n1; ++s) ok &= (pa[s] != pa[s + 1]) ? 1 : 0;
  int n2 = cur - 2 > 1 ? cur - 2 : 1;
  for (int s = 0; s < n2; ++s) ok &= (pa[s] != pa[s + 2]) ? 1 : 0;
  return ok;
}

__device__ inline int distinct_specials_gt1(const int32_t* w, int n, const uint8_t* special) {
  int first = -1;
  for (int k = 0; k < n; ++k) {
    int a = w[k];
    if (special[a]) {
      if (first < 0) first = a;
      else if (a != first) return 1;
    }
  }
  return 0;
}

// T_alloc = row stride of prev_actions; the dup checks read pa[s+1], pa[s+2] with s+2 <= max(cur-1,2)
// which stays inside the row for cur <= T and T >= 3.
__global__ void k_violation(int B, int T, int P, int seq, int cur, const int32_t* __restrict__ prev_actions,
                            const uint8_t* __restrict__ special, int32_t* __restrict__ out) {
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int32_t* pa = prev_actions + (size_t)b * T;
  int ok = violation_row(pa, cur, P, seq, special);
  if (seq) {
    int cp = cur % P;                                        // Q9: pages 0..cur%P only
    for (int j = 0; j <= cp; ++j) {
      int lo = P * j, hi = P * (j + 1);
      if (lo >= T) break;
      if (hi > T) hi = T;
      if (distinct_specials_gt1(pa + lo, hi - lo, special)) ok = 0;
    }
  } else {
    if (distinct_specials_gt1(pa, T, special)) ok = 0;
  }
  out[b] = ok;
}

__global__ void k_reward(int B, int T, int P, int seq, int cur /*after act*/, int zero_on_violation,
                         const int32_t* __restrict__ prev_actions, const uint8_t* __restrict__ special,
                         const double* __restrict__ price, const float* __restrict__ p1 /*[B*rpe]*/,
                         int rpe, double* __restrict__ reward, float* __restrict__ click_p) {
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int32_t* pa = prev_actions + (size_t)b * T;
  int w0 = seq ? cur - P : 0;
  double s = 0.0;
  for (int j = 0; j < rpe; ++j) {
    float pj = p1[(size_t)b * rpe + j];
    s += price[pa[w0 + j]] * (double)pj;
    if (click_p) click_p[(size_t)b * rpe + j] = pj;
  }
  if (zero_on_violation) {
    int ok = violation_row(pa, cur, P, seq, special);
    if (seq) {
      int cp = cur % P;
      for (int j = 0; j <= cp; ++j) {
        int lo = P * j, hi = P * (j + 1);
        if (lo >= T) break;
        if (hi > T) hi = T;
        if (distinct_specials_gt1(pa + lo, hi - lo, special)) ok = 0;
      }
    } else if (distinct_specials_gt1(pa, T, special)) ok = 0;
    if (!ok) s = 0.0;
  }
  reward[b] = s;
}

__global__ void k_fill_f64(int n, double v, double* out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = v;
}
__global__ void k_fill_u8(int n, uint8_t v, uint8_t* out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = v;
}

// out[b, :] = src[b * rpe + j, :] (128-bit columns): the observation of a paying step is row j = rpe - 1 of that step's
// reward pass (see reward_pass in r4_capi.cu)
__global__ void k_take_rows(int nb, int rpe, int j, int ld4, const float4* __restrict__ src, float4* __restrict__ out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)nb * ld4) return;
  const size_t b = i / ld4, c = i % ld4;
  out[i] = src[(b * rpe + j) * ld4 + c];
}

// d3rl 'masked_actions' (slate.py:98-104 / seqslate.py:18-23)
__global__ void k_masked_actions(int B, int T, int w0, int W, const int32_t* __restrict__ prev_actions,
                                 int32_t* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * W) return;
  int b = i / W, k = i % W;
  out[i] = prev_actions[(size_t)b * T + w0 + k];
}

// ------------------------------------------------------------------------------------------
// logged policy: SlateState.offline_action / offline_reward (slate.py:149-174, seqslate.py:71-86)
// ------------------------------------------------------------------------------------------
__global__ void k_offline_action(int B, int S, int cur, int T, int emb_dim, const int32_t* __restrict__ row_idx,
                                 const int32_t* __restrict__ log_items, const double* __restrict__ action_emb,
                                 int32_t* __restrict__ items, double* __restrict__ emb) {
  int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (b >= B) return;
  int a = (cur < T && cur < S) ? log_items[(size_t)row_idx[b] * S + cur] : 0;
  if (items && lane == 0) items[b] = a;
  if (emb)
    for (int k = lane; k < emb_dim; k += 32) emb[(size_t)b * emb_dim + k] = action_emb[(size_t)a * emb_dim + k];
}

__global__ void k_offline_reward(int B, int S, int lo, int hi, const int32_t* __restrict__ row_idx,
                                 const int32_t* __restrict__ log_items, const uint8_t* __restrict__ fb,
                                 const double* __restrict__ price, double* __restrict__ out) {
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  size_t base = (size_t)row_idx[b] * S;
  double s = 0.0;
  for (int k = lo; k < hi; ++k) s += price[log_items[base + k]] * (double)fb[base + k];
  out[b] = s;
}

}  // namespace r4
