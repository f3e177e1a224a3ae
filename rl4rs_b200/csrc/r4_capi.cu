// r4_capi.cu -- host side of librl4rs_b200.so: the C-ABI of include/rl4rs_b200.h over the
// kernels of r4_kernels.cuh.  No torch, no Python: plain CUDA runtime.  See DESIGN.md.
#include "../../include/rl4rs_b200.h"
#include "r4_kernels.cuh"
#include "r4_augru_pp.cuh"
#include "r4_gemm_tc.cuh"
#include "r4_scores_tc.cuh"
#include "r4_gru_tc.cuh"
#include "r4_ppo.cuh"
#include "r4_comm.cuh"

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <map>
#include <string>
#include <vector>

using namespace r4;

namespace {

std::string g_create_error;

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
};

struct SeqCache {   // one cached (sequence, weight-set): GRU-1 outputs + AUGRU/attention input halves
  DevBuf H;         // f32 [n, 64, 128]            GRU-1 outputs
  DevBuf Kp;        // f32 [n, 64, 64]             attention key half k_t (Wk - Wd)
  DevBuf XT;        // f32 [ceil(n/128), 64, 768, 128]: AUGRU input halves [r|u|c] (+bias), lane-major tiles
  int n = 0;
};

struct PerSeq {
  float *gru_wx = nullptr, *gru_bx = nullptr, *gru_wgh = nullptr, *gru_wch = nullptr;
  float *au_wx = nullptr, *au_bx = nullptr, *au_wgh = nullptr, *au_wch = nullptr;
  float *wqd = nullptr, *wp = nullptr, *ab1 = nullptr, *aw2 = nullptr, *ab2 = nullptr, *akv = nullptr;
  uint8_t *gru_wx_img = nullptr, *au_wx_img = nullptr, *wp_img = nullptr, *gru_img = nullptr;   // pre-tiled bf16 hi/lo images of the input projections
  uint8_t* au_pair_img = nullptr;   // the same weights tiled per CTA rank for the 2-CTA kernel (r4_augru_pair2.cuh)
  CUtensorMap au_pair_tmap;    // au_pair_img as a 2-D tensor of 1 KB rows (r4_augru_pp.cuh: tensor-map TMA ring)
  bool au_pair_tmap_ok = false;
  float abk = 0.f;
};

}  // namespace

struct r4_env {
  r4_config cfg;
  int device = 0;
  std::string err;
  int64_t launches = 0;
  int A = 0, words = 0, T = 0, P = 0, B = 0, seq = 0, emb_dim = 0, hash = 0;
  int max_rows = 0;
  // item tables
  float* item_vec = nullptr;
  double* price = nullptr;
  uint8_t* special = nullptr;
  double* action_emb = nullptr;
  bool items_ready = false;
  // weights
  std::map<std::string, std::vector<float>> hw;
  float *emb_cat = nullptr, *emb_seq = nullptr, *w1 = nullptr, *b1 = nullptr, *w2 = nullptr, *b2 = nullptr;
  float *wo = nullptr, *bo = nullptr, *wr = nullptr, *br = nullptr;
  uint8_t *w1_img = nullptr, *w2_img = nullptr, *wo_img = nullptr;   // tensor-core images (r4_gemm_tc.cuh)
  int sim = R4_SIM_DIEN;                                             // config['algo']: which simulator graph
  float* fcb = nullptr; uint8_t *fc_img = nullptr;                   // dnn: the unnamed Dense(256, ELU) of nets/dnn.py:34; widedeep: nets/widedeep.py:34
  int obs_dim = OBSD;                                                // 256, or 3072 for widedeep
  DevBuf ws_seq;                                                     // widedeep: sequence ids of a pass, i32 [R,2,64]
  // lstm (nets/lstm.py): the category GRU (Keras GRU over the 21 category embeddings, utils.py:34); the two sequence GRUs
  // (utils.py:92) reuse ps[i].gru_wx_img / gru_bx / gru_img, their LAST states are cached per sequence in SeqCache.H [n,128]
  uint8_t *cg_wx_img = nullptr, *cg_img = nullptr; float* cg_bx = nullptr;
  DevBuf ws_cgx;                                                     // lstm: category-GRU input halves of a pass, lane-major tiles
  PerSeq ps[2];
  bool weights_ready = false;
  std::vector<void*> owned;
  // log (borrowed device pointers)
  const int32_t* log_cat = nullptr;
  const float* log_dense = nullptr;
  const int32_t* log_seq = nullptr;
  const int32_t* log_items = nullptr;
  const uint8_t* log_fb = nullptr;
  int64_t log_n = 0;
  int log_slots = 0;
  // episode state
  int32_t* row_idx = nullptr;
  int32_t* prev_actions = nullptr;
  uint32_t* amask = nullptr;
  uint8_t* sflag = nullptr;
  int cur_steps = 0;
  bool has_reset = false;
  // caches
  SeqCache c0, c1const, c1page;
  bool c1_is_page = false;
  // workspaces
  DevBuf ws_cat, ws_dense, ws_scores, ws_allf, ws_tmp, ws_obs, ws_p1, ws_xin, ws_ids0, ws_ids1, ws_q, ws_part;
  // side stream: category attention + dense tower run concurrently with scores + AUGRU (they only
  // meet at the head GEMM), which fills the SMs the 128-row AUGRU tiles leave idle at small batch
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  // optional per-kernel CUDA-event timing (r4_profile): 0 off, 1 dominant kernel only, 2 every kernel
  int prof_mode = 0;
  struct ProfSlot { double ms = 0; int64_t n = 0; double work = 0; };
  struct PendingEv { cudaEvent_t a, b; int slot; };
  ProfSlot slots[16];
  std::vector<PendingEv> pending;
  std::vector<cudaEvent_t> evpool;
};

namespace {

int fail(r4_env* e, int code, const std::string& msg) {
  if (e) e->err = msg; else g_create_error = msg;
  return code;
}

enum { SL_ACT = 0, SL_ASSEMBLE, SL_SEQIDS, SL_GEMM_XIN, SL_GRU1, SL_GEMM_XK, SL_SCORES, SL_AUGRU, SL_CAT,
       SL_GEMM_DENSE, SL_GEMM_HEAD, SL_RHEAD, SL_REWARD, SL_XT, SL_MISC, SL_COUNT };
const char* const SLOT_NAMES[SL_COUNT] = {"k_act", "k_assemble", "k_seq_ids", "k_gemm_tc[gru1 input proj + E_s gather]",
    "k_gru_tc[GRU-1 tcgen05]", "k_gemm_tc[augru/att input proj]", "k_scores_tc", "k_augru[AUGRU tcgen05: pair2 / pp]", "k_cat_attn | k_cat_pool",
    "k_gemm_tc[dense tower]", "k_gemm_tc[head 3456x256]", "k_reward_head", "k_reward", "k_transpose_x", "k_query"};

// Brackets one launch with CUDA events on the launching stream when profiling is on.
struct ProfScope {
  r4_env* e; int slot; cudaStream_t st; cudaEvent_t a = nullptr, b = nullptr; bool on; double work;
  static cudaEvent_t get(r4_env* e) {
    if (!e->evpool.empty()) { cudaEvent_t x = e->evpool.back(); e->evpool.pop_back(); return x; }
    cudaEvent_t x; cudaEventCreate(&x); return x;
  }
  ProfScope(r4_env* e_, int slot_, cudaStream_t st_, double work_) : e(e_), slot(slot_), st(st_), work(work_) {
    // mode 1 = the dominant kernel only: the AUGRU recurrence (dien) / the embedding gather (dnn)
    on = e->prof_mode == 2 || (e->prof_mode == 1 && slot == (e->sim == R4_SIM_DNN ? SL_CAT : SL_AUGRU));
    if (on) { a = get(e); b = get(e); cudaEventRecord(a, st); }
  }
  ~ProfScope() {
    if (on) { cudaEventRecord(b, st); e->pending.push_back({a, b, slot}); e->slots[slot].work += work; }
  }
};

#define R4_CUDA(e, call)                                                                   \
  do {                                                                                     \
    cudaError_t _st = (call);                                                              \
    if (_st != cudaSuccess)                                                                \
      return fail((e), R4_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_st)); \
  } while (0)

#define R4_LAUNCH_CHECK(e, name)                                                          \
  do {                                                                                     \
    (e)->launches++;                                                                       \
    cudaError_t _st = cudaGetLastError();                                                  \
    if (_st != cudaSuccess)                                                                \
      return fail((e), R4_ERR_CUDA, std::string(name) + ": " + cudaGetErrorString(_st));  \
  } while (0)

int reserve(r4_env* e, DevBuf& b, size_t bytes) {
  if (b.bytes >= bytes && b.p) return R4_OK;
  if (b.p) { R4_CUDA(e, cudaFree(b.p)); b.p = nullptr; b.bytes = 0; }
  cudaError_t st = cudaMalloc(&b.p, bytes);
  if (st != cudaSuccess) return fail(e, R4_ERR_NOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(st));
  b.bytes = bytes;
  return R4_OK;
}

template <typename T>
int upload(r4_env* e, const std::vector<T>& h, T** dptr) {
  void* p = nullptr;
  cudaError_t st = cudaMalloc(&p, std::max<size_t>(h.size(), 1) * sizeof(T));
  if (st != cudaSuccess) return fail(e, R4_ERR_NOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(st));
  R4_CUDA(e, cudaMemcpy(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
  e->owned.push_back(p);
  *dptr = reinterpret_cast<T*>(p);
  return R4_OK;
}

inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// n-tile width of the observation-head GEMM (K = 3456, N = 256): 128 doubles its CTA count (64 at batch 4096).
// n-tile width of the observation head's weight image.  256: every 128-row tile converts its A rows (fp32 -> bf16 hi/mid/lo,
// the producers' work and the kernel's limiter) ONCE, and split-K (4 parts at 4096 rows: 32 tiles x 4 = 128 CTAs) fills the
// SMs; 128 (R4_HEAD_BNT=128, the earlier default) converted every A row twice for 64 tiles x 2 K parts.
static int head_bnt() {
  static const int v = [] { const char* e = getenv("R4_HEAD_BNT"); int x = e ? atoi(e) : 256; return (x == 128 || x == 256) ? x : 256; }();
  return v;
}
#define HEAD_BNT head_bnt()

int gemm(r4_env* e, int slot, int act, int M, int N, int K, const float* A, int lda, const int32_t* gather,
         const uint8_t* Wimg, const float* bias, float* C, int ldc, cudaStream_t st, int tm_ns = 0, int cr_base = 0,
         int ldT = 0, float* outT = nullptr, float* outK = nullptr, int bnt = r4tc::G_BNMAX,
         const float* A2 = nullptr, const int32_t* gather2 = nullptr, int k2_start = 0, int g2_n = 0, int tm_steps = MAXLEN,
         int ksplit_max = 1) {
  if (M <= 0) return R4_OK;
  if ((N & 15) || (K & 7) || (lda & 3) || (ldc & 3)) return fail(e, R4_ERR_ARG, "gemm: unaligned shape");
  ProfScope ps(e, slot, st, 2.0 * M * N * K);
  r4tc::GemmTcParams p{A, lda, gather, Wimg, bias, C, ldc, M, N, K, act, tm_ns, cr_base, ldT, outT, outK};
  p.bnt = bnt;
  p.A2 = A2; p.gather2 = gather2; p.k2_start = k2_start; p.g2_n = g2_n;
  p.tm_steps = tm_steps;
  static const int sms = [] { int d = 0, n = 148; cudaGetDevice(&d); cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, d); return n; }();
  int tiles = ((M + r4tc::G_BM - 1) / r4tc::G_BM) * ((N + bnt - 1) / bnt);
  // split-K when the output tiles leave SMs idle and K is long (each part keeps >= 16 K blocks): the head at 4096 rows
  static const bool no_splitk = getenv("R4_NO_SPLITK") != nullptr;
  const int ksplit = no_splitk ? 1 : std::max(1, std::min(std::min(ksplit_max, sms / std::max(tiles, 1)), K / (16 * r4tc::G_BK)));
  if (ksplit > 1) {
    if (tm_ns > 0 || !C || (N & 3)) return fail(e, R4_ERR_ARG, "gemm: split-K needs a plain row-major output");
    int rc;
    if ((rc = reserve(e, e->ws_part, (size_t)ksplit * M * N * 4))) return rc;
    p.ksplit = ksplit; p.part = reinterpret_cast<float*>(e->ws_part.p);
    tiles *= ksplit;
  }
  r4tc::k_gemm_tc<<<std::min(tiles, sms), r4tc::G_THREADS, r4tc::G_SMEM_BYTES, st>>>(p);
  R4_LAUNCH_CHECK(e, "k_gemm_tc");
  if (ksplit > 1) {
    const size_t n4 = (size_t)M * (N / 4);
    r4tc::k_splitk_finish<<<(unsigned)((n4 + 255) / 256), 256, 0, st>>>(M, N, ksplit, p.part, bias, act, C, ldc);
    R4_LAUNCH_CHECK(e, "k_splitk_finish");
  }
  return R4_OK;
}

int upload_image(r4_env* e, const float* W, int K, int N, uint8_t** out, int bnt = r4tc::G_BNMAX) {
  std::vector<uint8_t> img(r4tc::gemm_image_bytes(K, N, bnt));
  r4tc::build_gemm_image(W, K, N, img.data(), bnt);
  return upload(e, img, out);
}

constexpr int SMEM_CAT = 4 * (NCAT * CAT_LD + NCAT * 24) * 4;

// GRU-1 + input projections of one sequence set (nets/utils.py:113,120 and the x-halves of :121-124).
// ids: i32 [n,64] device.  Chunked (multiples of 128 sequences) so the input-projection scratch stays bounded.
int build_cache(r4_env* e, int si, const int32_t* ids, int n, SeqCache& c, cudaStream_t st) {
  int rc;
  const int TM = r4tc::TM;
  if (e->sim == R4_SIM_LSTM) {
    // nets/utils.py:90-92: Keras GRU over Embedding(seq_i), only the LAST state is used -> c.H is [n, 128]
    if ((rc = reserve(e, c.H, (size_t)n * EMB * 4))) return rc;
    c.n = n;
    const PerSeq& w = e->ps[si];
    const int chunk = 8192;
    const int nsmax = std::min(n, chunk);
    if ((rc = reserve(e, e->ws_xin, (size_t)((nsmax + TM - 1) / TM) * MAXLEN * r4tc::G1_XT_COLS * TM * 4))) return rc;
    float* xinT = reinterpret_cast<float*>(e->ws_xin.p);
    for (int s0 = 0; s0 < n; s0 += chunk) {
      const int ns = std::min(chunk, n - s0);
      if ((rc = gemm(e, SL_GEMM_XIN, 0, ns * MAXLEN, XIN_LD, EMB, e->emb_seq, EMB, ids + (size_t)s0 * MAXLEN, w.gru_wx_img,
                     w.gru_bx, nullptr, XIN_LD, st, ns, 0, XIN_LD, xinT, nullptr))) return rc;
      { ProfScope ps(e, SL_GRU1, st, (double)ns * MAXLEN * 2.0 * (EMB * 2 * EMB + EMB * EMB));
        r4tc::GruTcParams gp{xinT, w.gru_img, nullptr, ns};
        gp.hard = 1; gp.Hlast = reinterpret_cast<float*>(c.H.p) + (size_t)s0 * EMB; gp.ld_last = EMB;
        r4tc::k_gru_tc<<<(ns + TM - 1) / TM, r4tc::NTHREADS, r4tc::G1_SMEM_BYTES, st>>>(gp); }
      R4_LAUNCH_CHECK(e, "k_gru_tc");
    }
    return R4_OK;
  }
  if ((rc = reserve(e, c.H, (size_t)n * MAXLEN * EMB * 4))) return rc;
  if ((rc = reserve(e, c.Kp, (size_t)n * MAXLEN * AH1 * 4))) return rc;
  if ((rc = reserve(e, c.XT, (size_t)((n + TM - 1) / TM) * MAXLEN * r4tc::XT_COLS * TM * 4))) return rc;
  c.n = n;
  const PerSeq& w = e->ps[si];
  const int chunk = 8192;
  const int nsmax = std::min(n, chunk);
  if ((rc = reserve(e, e->ws_xin, (size_t)((nsmax + TM - 1) / TM) * MAXLEN * r4tc::G1_XT_COLS * TM * 4))) return rc;
  float* xinT = reinterpret_cast<float*>(e->ws_xin.p);
  for (int s0 = 0; s0 < n; s0 += chunk) {
    int ns = std::min(chunk, n - s0);
    float* Hc = reinterpret_cast<float*>(c.H.p) + (size_t)s0 * MAXLEN * EMB;
    // x_t [Wgx | Wcx] + [bg | bc]: Embedding gather fused into the A operand, output in lane-major tiles
    if ((rc = gemm(e, SL_GEMM_XIN, 0, ns * MAXLEN, XIN_LD, EMB, e->emb_seq, EMB, ids + (size_t)s0 * MAXLEN, w.gru_wx_img,
                   w.gru_bx, nullptr, XIN_LD, st, ns, 0, XIN_LD, xinT, nullptr))) return rc;
    { ProfScope ps(e, SL_GRU1, st, (double)ns * MAXLEN * 2.0 * (EMB * 2 * EMB + EMB * EMB));
      r4tc::GruTcParams gp{xinT, w.gru_img, Hc, ns};
      r4tc::k_gru_tc<<<(ns + TM - 1) / TM, r4tc::NTHREADS, r4tc::G1_SMEM_BYTES, st>>>(gp); }
    R4_LAUNCH_CHECK(e, "k_gru_tc");
    // H_t [Wgx | Wcx | Wk-Wd] + [bg | bc | 0]: AUGRU halves -> XT tiles, key half -> Kp
    if ((rc = gemm(e, SL_GEMM_XK, 0, ns * MAXLEN, XK_LD, EMB, Hc, EMB, nullptr, w.au_wx_img, w.au_bx, nullptr, XK_LD, st,
                   ns, s0, r4tc::XT_COLS, reinterpret_cast<float*>(c.XT.p), reinterpret_cast<float*>(c.Kp.p)))) return rc;
  }
  return R4_OK;
}

// Kernel-choice options (r4_set_option; the environment gives the initial values).
struct AugruOpts {
  int force = 0;          // 0 rule, 2 pair kernel (one recurrence per pair), 3 ping-pong pair kernel (1 was the deleted one-CTA kernel)
  // cost of one wave, measured (tools/augru_probe.cu, round 2, ms x 25): k_augru_pair2 0.51 ms per 74 tile-sequences,
  // k_augru_pp 0.96 ms per 74 TILES (= 148 tile-sequences)
  int cost_pair = 13, cost_pp = 24;
  int scores_shared_pct = 85;    // k_scores_tc2: CTA share of a shared (L2-resident) sequence, per cent of an even split (tools/scores_probe.cu,
                                 // us per 4096-row pass: 100 % 98.5, 85 % 86.8, 75 % 90.1, 65 % 100.6, 55 % 120.8)
  int pay_obs_reuse = 1;  // a paying step takes its observation from its reward pass (r4_step); 0 = separate observation pass
  AugruOpts() {
    if (getenv("R4_NO_PAY_OBS_REUSE")) pay_obs_reuse = 0;
    if (getenv("R4_AUGRU_PAIR")) force = 2; else if (getenv("R4_AUGRU_PP")) force = 3;
    if (const char* e = getenv("R4_AUGRU_RULE")) {
      int a = 0, b = 0;
      if (sscanf(e, "%d,%d", &a, &b) == 2 && a > 0 && b > 0) { cost_pair = a; cost_pp = b; }
    }
  }
};
AugruOpts& augru_opts() { static AugruOpts o; return o; }

// Which AUGRU kernel runs `ctas` = 2 x row tiles (tile-sequences) of work: 2 = k_augru_pair2 (a CTA pair per tile-sequence),
// 3 = k_augru_pp (a CTA pair per TILE, both sequences in flight).  The pair kernel finishes a tile sooner, the ping-pong
// kernel keeps the tensor pipe busier but needs twice the tiles to fill the chip: compare wave counts x measured wave times.
static int augru_rule(int ctas, int sms) {
  const AugruOpts& o = augru_opts();
  const int pairs = sms / 2;
  const long c2 = (long)o.cost_pair * ((ctas + pairs - 1) / pairs);
  const long c3 = (long)o.cost_pp * (((ctas + 1) / 2 + pairs - 1) / pairs);
  return c3 <= c2 ? 3 : 2;
}
static int augru_choice(int ctas) {
  static const int sms = [] { int d = 0, n = 148; cudaGetDevice(&d); cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, d); return n; }();
  const int force = augru_opts().force;
  return force ? force : augru_rule(ctas, sms);
}

// One simulator pass over `R` feature rows (cat/dense already assembled, chunk-local pointers).
int forward_rows(r4_env* e, int R, int row0, int div, const int32_t* cat, const float* dense,
                 const SeqCache& c0, int shared0, const SeqCache& c1, int shared1, float* obs_out,
                 float* p1_out, float* probs_out, cudaStream_t st) {
  int rc;
  if (e->sim == R4_SIM_LSTM) {
    // nets/lstm.py:29-36: all = [GRU(seq0) | GRU(seq1) | dense tower | GRU(E_c[cat]) | Flatten(E_c[cat])] -> Dense(256, ELU) =
    // simulator_obs -> softmax head.  The sequence GRUs' last states come from the caches; the category GRU (21 steps)
    // runs per pass: E_c gather fused into its input projection, then the tcgen05 recurrence writes its last state
    // straight into the feature slab; the Flatten() part is gathered by the head GEMM's A staging (as in the dien head).
    const int TM = r4tc::TM, LD = 4 * EMB;                  // materialised part of the feature vector: 512 columns
    const int rtiles = (R + TM - 1) / TM;
    if ((rc = reserve(e, e->ws_allf, (size_t)R * LD * 4))) return rc;
    if ((rc = reserve(e, e->ws_tmp, (size_t)R * HU * 4))) return rc;
    if ((rc = reserve(e, e->ws_cgx, (size_t)rtiles * NCAT * r4tc::G1_XT_COLS * TM * 4))) return rc;
    float* allf = reinterpret_cast<float*>(e->ws_allf.p);
    float* tmp = reinterpret_cast<float*>(e->ws_tmp.p);
    float* cgx = reinterpret_cast<float*>(e->ws_cgx.p);
    { ProfScope ps(e, SL_MISC, st, (double)R);
      k_seq_last_rows<<<(R * 64 + 255) / 256, 256, 0, st>>>(R, row0, div, reinterpret_cast<const float*>(c0.H.p), shared0,
                                                          reinterpret_cast<const float*>(c1.H.p), shared1, allf, LD); }
    R4_LAUNCH_CHECK(e, "k_seq_last_rows");
    if ((rc = gemm(e, SL_GEMM_XK, 0, R * NCAT, XIN_LD, EMB, e->emb_cat, EMB, cat, e->cg_wx_img, e->cg_bx, nullptr, XIN_LD, st,
                   R, 0, XIN_LD, cgx, nullptr, r4tc::G_BNMAX, nullptr, nullptr, 0, 0, NCAT))) return rc;
    { ProfScope ps(e, SL_GRU1, st, (double)R * NCAT * 2.0 * (EMB * 2 * EMB + EMB * EMB));
      r4tc::GruTcParams gp{cgx, e->cg_img, nullptr, R};
      gp.steps = NCAT; gp.hard = 1; gp.Hlast = allf + 3 * EMB; gp.ld_last = LD;
      r4tc::k_gru_tc<<<rtiles, r4tc::NTHREADS, r4tc::G1_SMEM_BYTES, st>>>(gp); }
    R4_LAUNCH_CHECK(e, "k_gru_tc");
    if ((rc = gemm(e, SL_GEMM_DENSE, 1, R, HU, NDENSE, dense, NDENSE, nullptr, e->w1_img, e->b1, tmp, HU, st))) return rc;
    if ((rc = gemm(e, SL_GEMM_DENSE, 1, R, HU, HU, tmp, HU, nullptr, e->w2_img, e->b2, allf + 2 * EMB, LD, st))) return rc;
    float* obs = obs_out;
    if (!obs) {
      if ((rc = reserve(e, e->ws_obs, (size_t)R * OBSD * 4))) return rc;
      obs = reinterpret_cast<float*>(e->ws_obs.p);
    }
    if ((rc = gemm(e, SL_GEMM_HEAD, 1, R, OBSD, LD + NCAT * EMB, allf, LD, nullptr, e->wo_img, e->bo, obs, OBSD, st, 0, 0, 0, nullptr,
                   nullptr, HEAD_BNT, e->emb_cat, cat, LD, NCAT, MAXLEN, 4))) return rc;
    if (p1_out || probs_out) {
      { ProfScope ps(e, SL_RHEAD, st, (double)R * 2.0 * OBSD * 2);
        k_reward_head<<<(R + 3) / 4, 128, 0, st>>>(R, obs, e->wr, e->br, p1_out, probs_out); }
      R4_LAUNCH_CHECK(e, "k_reward_head");
    }
    return R4_OK;
  }
  if (e->sim == R4_SIM_WIDEDEEP) {
    // nets/widedeep.py:31-38: simulator_obs = [Dense256(ELU)(seq mean-pools) | dense tower | Flatten(E_c[cat])]; softmax head on it.
    // The sequence ids of the pass rows are in e->ws_seq (obs / reward passes: k_seq_ids_rows; r4_dien_forward: the caller's).
    if ((rc = reserve(e, e->ws_allf, (size_t)R * 2 * EMB * 4))) return rc;
    if ((rc = reserve(e, e->ws_tmp, (size_t)R * HU * 4))) return rc;
    float* pooled = reinterpret_cast<float*>(e->ws_allf.p);
    float* tmp = reinterpret_cast<float*>(e->ws_tmp.p);
    float* obs = obs_out;
    if (!obs) {
      if ((rc = reserve(e, e->ws_obs, (size_t)R * OBSD_WD * 4))) return rc;
      obs = reinterpret_cast<float*>(e->ws_obs.p);
    }
    { ProfScope ps(e, SL_CAT, st, (double)R * (2 * MAXLEN * EMB * 4 + NCAT * EMB * 4));
      k_seq_pool<<<(R + 3) / 4, 128, 0, st>>>(R, reinterpret_cast<const int32_t*>(e->ws_seq.p), e->emb_seq, pooled);
      k_cat_flatten<<<(R + 3) / 4, 128, 0, st>>>(R, cat, e->emb_cat, obs + 2 * EMB + HU, OBSD_WD); }
    R4_LAUNCH_CHECK(e, "k_seq_pool / k_cat_flatten");
    e->launches++;
    if ((rc = gemm(e, SL_GEMM_HEAD, 1, R, 2 * EMB, 2 * EMB, pooled, 2 * EMB, nullptr, e->fc_img, e->fcb, obs, OBSD_WD, st))) return rc;
    if ((rc = gemm(e, SL_GEMM_DENSE, 1, R, HU, NDENSE, dense, NDENSE, nullptr, e->w1_img, e->b1, tmp, HU, st))) return rc;
    if ((rc = gemm(e, SL_GEMM_DENSE, 1, R, HU, HU, tmp, HU, nullptr, e->w2_img, e->b2, obs + 2 * EMB, OBSD_WD, st))) return rc;
    if (p1_out || probs_out) {
      { ProfScope ps(e, SL_RHEAD, st, (double)R * 2.0 * OBSD_WD * 2);
        k_reward_head<<<(R + 3) / 4, 128, 0, st>>>(R, obs, e->wr, e->br, p1_out, probs_out, OBSD_WD); }
      R4_LAUNCH_CHECK(e, "k_reward_head");
    }
    return R4_OK;
  }
  if (e->sim == R4_SIM_DNN) {
    // nets/dnn.py:31-37: all = [mean_t E_c[cat] | dense tower]; Dense(256, ELU); simulator_obs Dense(256, ELU); softmax head
    if ((rc = reserve(e, e->ws_allf, (size_t)R * 2 * HU * 4))) return rc;
    if ((rc = reserve(e, e->ws_tmp, (size_t)R * OBSD * 4))) return rc;
    float* allf = reinterpret_cast<float*>(e->ws_allf.p);
    float* tmp = reinterpret_cast<float*>(e->ws_tmp.p);
    static const int sms = [] { int d = 0, n = 148; cudaGetDevice(&d); cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, d); return n; }();
    { ProfScope ps(e, SL_CAT, st, (double)R * (NCAT * 4 + NCAT * EMB * 4));       // work = algorithmic gather bytes
      const int blocks = std::max(1, std::min((R + POOL_WARPS - 1) / POOL_WARPS, 2 * sms));
      k_cat_pool<<<blocks, POOL_WARPS * 32, POOL_SMEM, st>>>(R, cat, e->emb_cat, allf, 2 * HU); }
    R4_LAUNCH_CHECK(e, "k_cat_pool");
    if ((rc = gemm(e, SL_GEMM_DENSE, 1, R, HU, NDENSE, dense, NDENSE, nullptr, e->w1_img, e->b1, tmp, HU, st))) return rc;
    if ((rc = gemm(e, SL_GEMM_DENSE, 1, R, HU, HU, tmp, HU, nullptr, e->w2_img, e->b2, allf + HU, 2 * HU, st))) return rc;
    if ((rc = gemm(e, SL_GEMM_DENSE, 1, R, OBSD, 2 * HU, allf, 2 * HU, nullptr, e->fc_img, e->fcb, tmp, OBSD, st))) return rc;
    float* obs = obs_out;
    if (!obs) {
      if ((rc = reserve(e, e->ws_obs, (size_t)R * OBSD * 4))) return rc;
      obs = reinterpret_cast<float*>(e->ws_obs.p);
    }
    if ((rc = gemm(e, SL_GEMM_HEAD, 1, R, OBSD, OBSD, tmp, OBSD, nullptr, e->wo_img, e->bo, obs, OBSD, st))) return rc;
    if (p1_out || probs_out) {
      { ProfScope ps(e, SL_RHEAD, st, (double)R * 2.0 * OBSD * 2);
        k_reward_head<<<(R + 3) / 4, 128, 0, st>>>(R, obs, e->wr, e->br, p1_out, probs_out); }
      R4_LAUNCH_CHECK(e, "k_reward_head");
    }
    return R4_OK;
  }
  const int rtiles = (R + r4tc::TM - 1) / r4tc::TM;
  const size_t sc_per_seq = (size_t)rtiles * r4tc::TM * MAXLEN;
  if ((rc = reserve(e, e->ws_scores, 2 * sc_per_seq * 4))) return rc;
  if ((rc = reserve(e, e->ws_allf, (size_t)R * ALLF_LD * 4))) return rc;
  if ((rc = reserve(e, e->ws_tmp, (size_t)R * HU * 4))) return rc;
  if ((rc = reserve(e, e->ws_q, (size_t)R * (r4tc::S_K + 2 * r4tc::S_N) * 4))) return rc;
  float* qbuf = reinterpret_cast<float*>(e->ws_q.p);
  float* qa0 = qbuf + (size_t)R * r4tc::S_K;
  float* qa1 = qa0 + (size_t)R * r4tc::S_N;
  float* scores = reinterpret_cast<float*>(e->ws_scores.p);
  float* allf = reinterpret_cast<float*>(e->ws_allf.p);
  float* tmp = reinterpret_cast<float*>(e->ws_tmp.p);
  const SeqCache* cs[2] = {&c0, &c1};
  int sh[2] = {shared0, shared1};
  r4tc::ScoreTcParams sp{};
  r4tc::AugruTcParams rp{};
  for (int i = 0; i < 2; ++i) {
    const PerSeq& w = e->ps[i];
    r4tc::ScoreTcSeq& s = sp.s[i];
    s.H = reinterpret_cast<const float*>(cs[i]->H.p);
    s.Kp = reinterpret_cast<const float*>(cs[i]->Kp.p);
    s.qa = i ? qa1 : qa0; s.WpImg = w.wp_img; s.Wqd = w.wqd; s.b1 = w.ab1; s.W2 = w.aw2; s.b2 = w.ab2; s.kv = w.akv; s.bk = w.abk;
    s.scoresT = scores + (size_t)i * sc_per_seq;
    s.shared = sh[i];
    r4tc::AugruTcSeq& q = rp.s[i];
    q.XT = reinterpret_cast<const float*>(cs[i]->XT.p); q.Wimg = w.au_pair_img; q.scoresT = s.scoresT;
    q.out = allf + i * AUH; q.shared = sh[i];
  }
  sp.R = R; sp.row0 = row0; sp.div = div; sp.q = qbuf;
  rp.R = R; rp.row0 = row0; rp.div = div; rp.out_ld = ALLF_LD;
  // The side stream (lowest priority) does the AUGRU-independent half of the feature vector: category attention +
  // dense tower.  It forks AFTER k_scores_tc and is fed after the AUGRU launch, so the AUGRU pairs (1 CTA per SM,
  // 128 SMs at 4096 rows) are resident first and the side kernels fill the remaining SMs instead of delaying them.
  // R4_NO_SIDE_STREAM / the per-kernel breakdown mode (r4_profile(2)) serialise everything on one stream: event pairs
  // around a kernel on the low-priority side stream would time its wait for free SMs, not the kernel.
  static const bool no_side_env = getenv("R4_NO_SIDE_STREAM") != nullptr;
  const bool no_side = no_side_env || e->prof_mode == 2;
  auto side_work = [&]() -> int {
    cudaStream_t ss = no_side ? st : e->side;
    if (!no_side) R4_CUDA(e, cudaStreamWaitEvent(e->side, e->ev_fork, 0));
    { ProfScope ps(e, SL_CAT, ss, (double)R * 2.0 * (NCAT * NCAT * EMB * 2));
      k_cat_attn<<<(R + 3) / 4, 128, SMEM_CAT, ss>>>(R, cat, e->emb_cat, allf); }
    R4_LAUNCH_CHECK(e, "k_cat_attn");
    int rc2;
    if ((rc2 = gemm(e, SL_GEMM_DENSE, 1, R, HU, NDENSE, dense, NDENSE, nullptr, e->w1_img, e->b1, tmp, HU, ss))) return rc2;
    if ((rc2 = gemm(e, SL_GEMM_DENSE, 1, R, HU, HU, tmp, HU, nullptr, e->w2_img, e->b2, allf + 2 * AUH, ALLF_LD, ss))) return rc2;
    if (!no_side) R4_CUDA(e, cudaEventRecord(e->ev_join, ss));
    return R4_OK;
  };
  if (no_side && (rc = side_work())) return rc;
  { ProfScope ps(e, SL_MISC, st, (double)R);
    r4tc::k_query<<<(R + 7) / 8, 128, 0, st>>>(R, cat, e->emb_seq, e->ps[0].wqd, e->ps[0].ab1, e->ps[1].wqd, e->ps[1].ab1,
                                                qbuf, qa0, qa1); }
  R4_LAUNCH_CHECK(e, "k_query");
  { ProfScope ps(e, SL_SCORES, st, (double)R * 2 * MAXLEN * 2.0 * (EMB * AH1 + AH1 * AH2 + AH2));
    const int nt = (R + 1) / 2;
    const int ctas = std::min(2 * nt, 148);
    r4tc::k_scores_tc2<false><<<ctas, r4tc::S2_THREADS, r4tc::S2_SMEM_BYTES, st>>>(
        sp, r4tc::scores_grid_split(ctas, nt, sh[0], sh[1], augru_opts().scores_shared_pct)); }
  R4_LAUNCH_CHECK(e, "k_scores_tc");
  if (!no_side) R4_CUDA(e, cudaEventRecord(e->ev_fork, st));
  { ProfScope ps(e, SL_AUGRU, st, (double)R * 2 * MAXLEN * 2.0 * (AUH * 2 * AUH + AUH * AUH));
    r4tc::AugruPairParams pp;
    pp.b = rp; pp.tmap[0] = e->ps[0].au_pair_tmap; pp.tmap[1] = e->ps[1].au_pair_tmap;
    if (augru_choice(2 * rtiles) == 3) {
      r4tc::k_augru_pp<<<dim3(rtiles * 2), r4tc::NTHREADS, r4tc::PP_SMEM_BYTES, st>>>(pp);
    } else {
      // one 2-CTA cluster per tile and sequence
      cudaLaunchConfig_t lc = {};
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeClusterDimension;
      at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
      lc.gridDim = dim3(rtiles * 2, 2); lc.blockDim = dim3(r4tc::NTHREADS);
      lc.dynamicSmemBytes = r4tc::P_SMEM_BYTES; lc.stream = st; lc.attrs = at; lc.numAttrs = 1;
      (void)cudaLaunchKernelEx(&lc, r4tc::k_augru_pair2, pp);
    } }
  R4_LAUNCH_CHECK(e, augru_choice(2 * rtiles) == 3 ? "k_augru_pp" : "k_augru_pair2");
  if (!no_side && (rc = side_work())) return rc;
  if (!no_side) R4_CUDA(e, cudaStreamWaitEvent(st, e->ev_join, 0));
  float* obs = obs_out;
  if (!obs) {
    if ((rc = reserve(e, e->ws_obs, (size_t)R * OBSD * 4))) return rc;
    obs = reinterpret_cast<float*>(e->ws_obs.p);
  }
  // head: K = 768 materialised columns + 21 x 128 gathered from the category embedding table by `cat`
  if ((rc = gemm(e, SL_GEMM_HEAD, 1, R, OBSD, ALLF, allf, ALLF_LD, nullptr, e->wo_img, e->bo, obs, OBSD, st, 0, 0, 0, nullptr, nullptr, HEAD_BNT,
                 e->emb_cat, cat, ALLF_LD, NCAT, MAXLEN, 4))) return rc;
  if (p1_out || probs_out) {
    { ProfScope ps(e, SL_RHEAD, st, (double)R * 2.0 * OBSD * 2);
    k_reward_head<<<(R + 3) / 4, 128, 0, st>>>(R, obs, e->wr, e->br, p1_out, probs_out); }
    R4_LAUNCH_CHECK(e, "k_reward_head");
  }
  return R4_OK;
}

int assemble(r4_env* e, int mode, int step, int rpe, int row0, int nrows, int32_t* cat, float* dense,
             cudaStream_t st) {
  AsmParams p{mode, e->B, e->T, e->P, e->seq, step, rpe, row0, nrows};
  { ProfScope ps(e, SL_ASSEMBLE, st, (double)nrows);
    k_assemble<<<(nrows + 3) / 4, 128, 0, st>>>(p, e->row_idx, e->log_cat, e->log_dense, e->item_vec,
                                               e->prev_actions, cat, dense); }
  R4_LAUNCH_CHECK(e, "k_assemble");
  return R4_OK;
}

const SeqCache& seq1_cache(const r4_env* e) { return e->c1_is_page ? e->c1page : e->c1const; }

// widedeep reads the raw sequence ids of its pass rows (no sequence cache): stage them in e->ws_seq
int stage_seq_rows(r4_env* e, int R, int row0, int div, int p0, cudaStream_t st) {
  if (e->sim != R4_SIM_WIDEDEEP) return R4_OK;
  int rc;
  if ((rc = reserve(e, e->ws_seq, (size_t)R * 2 * MAXLEN * 4))) return rc;
  k_seq_rows<<<(R * MAXLEN + 255) / 256, 256, 0, st>>>(R, row0, div, e->T, p0, e->row_idx, e->log_seq, e->prev_actions,
                                                      reinterpret_cast<int32_t*>(e->ws_seq.p));
  R4_LAUNCH_CHECK(e, "k_seq_rows");
  return R4_OK;
}

// obs pass for the current state (mode 0 after reset, mode 1 after act at `step`)
int obs_pass(r4_env* e, int mode, int step, const r4_out* out, cudaStream_t st) {
  int rc;
  const int B = e->B;
  bool raw = (e->cfg.flags & R4_FLAG_RAWSTATE) != 0;
  bool need_obs = out && out->obs && !raw;
  bool need_feat = out && (out->cat || out->dense);
  if (!need_obs && !need_feat) return R4_OK;
  int chunk = need_obs ? std::min(B, e->max_rows) : B;
  for (int r0 = 0; r0 < B; r0 += chunk) {
    int nr = std::min(chunk, B - r0);
    int32_t* cat = (out && out->cat) ? out->cat + (size_t)r0 * NCAT : nullptr;
    float* dense = (out && out->dense) ? out->dense + (size_t)r0 * NDENSE : nullptr;
    if (!cat) { if ((rc = reserve(e, e->ws_cat, (size_t)chunk * NCAT * 4))) return rc; cat = (int32_t*)e->ws_cat.p; }
    if (!dense) { if ((rc = reserve(e, e->ws_dense, (size_t)chunk * NDENSE * 4))) return rc; dense = (float*)e->ws_dense.p; }
    if ((rc = assemble(e, mode, step, 1, r0, nr, cat, dense, st))) return rc;
    if (need_obs) {
      const SeqCache& c1 = seq1_cache(e);
      if ((rc = stage_seq_rows(e, nr, r0, 1, (mode == 1 && e->seq) ? step / e->P * e->P : 0, st))) return rc;
      if ((rc = forward_rows(e, nr, r0, 1, cat, dense, e->c0, 0, c1, e->c1_is_page ? 0 : 1,
                             out->obs + (size_t)r0 * e->obs_dim, nullptr, nullptr, st))) return rc;
    }
  }
  return R4_OK;
}

// reward pass: rpe rows per env row (slate.py:286-302 / seqslate.py:138-153).
// obs_take != null: also the step's observation.  A step pays when it completes a slate / a page, and the state it leaves
// behind (slate.py:203-213, seqslate.py:104-122: the complete page + the last action) is, field for field, the LAST of the
// page's complete states (slate.py:117-131, seqslate.py:27-50 with j = cur_steps - 1): the same feature row goes through the
// same network twice in the reference (obs_layer at base.py:160, reward_layer at slate.py:296).  Here row rpe - 1 of every
// env row's reward rows keeps its simulator_obs output and the separate observation pass is not launched.
int reward_pass(r4_env* e, int cur_after, const r4_out* out, cudaStream_t st, float* obs_take = nullptr) {
  int rc;
  const int B = e->B;
  const int rpe = e->seq ? e->P : e->T;
  if ((rc = reserve(e, e->ws_p1, (size_t)B * rpe * 4))) return rc;
  float* p1 = reinterpret_cast<float*>(e->ws_p1.p);
  int envs_per_chunk = std::max(1, e->max_rows / rpe);
  for (int b0 = 0; b0 < B; b0 += envs_per_chunk) {
    int nb = std::min(envs_per_chunk, B - b0);
    int nr = nb * rpe;
    if ((rc = reserve(e, e->ws_cat, (size_t)std::max(nr, 1) * NCAT * 4))) return rc;
    if ((rc = reserve(e, e->ws_dense, (size_t)std::max(nr, 1) * NDENSE * 4))) return rc;
    int32_t* cat = (int32_t*)e->ws_cat.p;
    float* dense = (float*)e->ws_dense.p;
    if ((rc = assemble(e, 2, cur_after, rpe, b0 * rpe, nr, cat, dense, st))) return rc;
    if ((rc = stage_seq_rows(e, nr, b0 * rpe, rpe, e->seq ? cur_after - e->P : 0, st))) return rc;
    const SeqCache& c1 = seq1_cache(e);
    if ((rc = forward_rows(e, nr, b0 * rpe, rpe, cat, dense, e->c0, 0, c1, e->c1_is_page ? 0 : 1, nullptr,
                           p1 + (size_t)b0 * rpe, nullptr, st))) return rc;
    if (obs_take) {                     // forward_rows left simulator_obs of the chunk's rows in ws_obs [nr, obs_dim]
      const int ld4 = e->obs_dim / 4;
      k_take_rows<<<(int)(((size_t)nb * ld4 + 255) / 256), 256, 0, st>>>(nb, rpe, rpe - 1, ld4, reinterpret_cast<const float4*>(e->ws_obs.p),
                                                                         reinterpret_cast<float4*>(obs_take + (size_t)b0 * e->obs_dim));
      R4_LAUNCH_CHECK(e, "k_take_rows");
    }
  }
  int zero = 1;                                                   // slate.py:303 `if 1:`
  if (e->seq) zero = (e->cfg.flags & (R4_FLAG_RLLIB_MASK | R4_FLAG_D3RL_MASK)) ? 1 : 0;   // seqslate.py:154-157
  float* click = (out && out->click_p && (e->cfg.flags & R4_FLAG_INFO_FETCH)) ? out->click_p : nullptr;
  { ProfScope ps(e, SL_REWARD, st, (double)B);
    k_reward<<<(B + 127) / 128, 128, 0, st>>>(B, e->T, e->P, e->seq, cur_after, zero, e->prev_actions, e->special,
                                             e->price, p1, rpe, out->reward, click); }
  R4_LAUNCH_CHECK(e, "k_reward");
  return R4_OK;
}

int write_masked_actions(r4_env* e, const r4_out* out, cudaStream_t st) {
  if (!out || !out->masked_actions) return R4_OK;
  int w0 = 0, W = e->T;
  if (e->seq) {                                                   // seqslate.py:20-22
    int p0 = e->cur_steps / e->P * e->P;
    int pe = std::min(p0 + e->P - 1, e->T - 1);
    w0 = pe + 1 - e->P; W = e->P;
  }
  k_masked_actions<<<(e->B * W + 255) / 256, 256, 0, st>>>(e->B, e->T, w0, W, e->prev_actions, out->masked_actions);
  R4_LAUNCH_CHECK(e, "k_masked_actions");
  return R4_OK;
}

const float* hw_get(r4_env* e, const std::string& name, size_t n) {
  auto it = e->hw.find(name);
  if (it == e->hw.end() || it->second.size() != n) return nullptr;
  return it->second.data();
}

}  // namespace

extern "C" {

int r4_abi_version(void) { return 2; }
int r4_obs_dim(int simulator) { return simulator == R4_SIM_WIDEDEEP ? OBSD_WD : OBSD; }

const char* r4_last_error(const r4_env* env) { return env ? env->err.c_str() : g_create_error.c_str(); }

int r4_create(const r4_config* cfg, int device, r4_env** out) {
  if (!cfg || !out) return fail(nullptr, R4_ERR_ARG, "r4_create: null argument");
  *out = nullptr;
  if (cfg->maxlen != MAXLEN || cfg->seq_num != 2 || cfg->dense_feature_num != NDENSE ||
      cfg->category_feature_num != NCAT || cfg->emb_size != EMB || cfg->hidden_units != HU ||
      cfg->page_items != PAGE)
    return fail(nullptr, R4_ERR_ARG,
                "r4_create: this build is specialised for maxlen=64 seq_num=2 dense_feature_num=432 "
                "category_feature_num=21 emb_size=128 hidden_units=128 page_items=9");
  if (cfg->batch_size < 1 || cfg->max_steps < 3 || cfg->action_size < 149 || cfg->action_size > 32 * MAX_WORDS)
    return fail(nullptr, R4_ERR_ARG, "r4_create: need batch_size>=1, max_steps>=3, 149<=action_size<=512");
  if (cfg->env_kind == R4_ENV_SLATE && cfg->max_steps > 11)
    return fail(nullptr, R4_ERR_ARG, "r4_create: SlateRecEnv needs max_steps<=11 (location_mask has 4 layers, slate.py:60-64,93)");
  if (cfg->env_kind == R4_ENV_SEQSLATE && cfg->max_steps % cfg->page_items != 0)
    return fail(nullptr, R4_ERR_ARG, "r4_create: SeqSlateRecEnv needs max_steps to be a multiple of page_items");
  if (cfg->category_hash_size < cfg->action_size)
    return fail(nullptr, R4_ERR_ARG, "r4_create: category_hash_size must cover the item ids");
  if (cfg->simulator < R4_SIM_DIEN || cfg->simulator > R4_SIM_LSTM)
    return fail(nullptr, R4_ERR_ARG, "r4_create: simulator must be R4_SIM_DIEN, R4_SIM_DNN, R4_SIM_WIDEDEEP or R4_SIM_LSTM (config['algo'] = 'dien' | 'dnn' | 'widedeep' | 'lstm')");
  cudaError_t st = cudaSetDevice(device);
  if (st != cudaSuccess) return fail(nullptr, R4_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(st));
  r4_env* e = new r4_env();
  e->cfg = *cfg;
  e->device = device;
  e->A = cfg->action_size; e->words = (e->A + 31) / 32; e->T = cfg->max_steps; e->P = cfg->page_items;
  e->B = cfg->batch_size; e->seq = cfg->env_kind == R4_ENV_SEQSLATE; e->hash = cfg->category_hash_size;
  e->max_rows = cfg->max_rows_per_pass > 0 ? cfg->max_rows_per_pass : 36864;
  e->sim = cfg->simulator;
  e->obs_dim = cfg->simulator == R4_SIM_WIDEDEEP ? OBSD_WD : OBSD;
  bool ok = cudaMalloc(&e->row_idx, (size_t)e->B * 4) == cudaSuccess &&
            cudaMalloc(&e->prev_actions, (size_t)e->B * e->T * 4) == cudaSuccess &&
            cudaMalloc(&e->amask, (size_t)e->B * e->words * 4) == cudaSuccess &&
            cudaMalloc(&e->sflag, (size_t)e->B) == cudaSuccess;
  if (!ok) { r4_destroy(e); return fail(nullptr, R4_ERR_NOMEM, "r4_create: cudaMalloc failed"); }
  cudaFuncSetAttribute(r4tc::k_gru_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, r4tc::G1_SMEM_BYTES);
  cudaFuncSetAttribute(r4tc::k_augru_pp, cudaFuncAttributeMaxDynamicSharedMemorySize, r4tc::PP_SMEM_BYTES);
  cudaFuncSetAttribute(r4tc::k_augru_pair2, cudaFuncAttributeMaxDynamicSharedMemorySize, r4tc::P_SMEM_BYTES);
  cudaFuncSetAttribute(r4tc::k_gemm_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, r4tc::G_SMEM_BYTES);
  cudaFuncSetAttribute(r4tc::k_scores_tc2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, r4tc::S2_SMEM_BYTES);
  cudaFuncSetAttribute(k_cat_attn, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_CAT);
  cudaFuncSetAttribute(k_cat_pool, cudaFuncAttributeMaxDynamicSharedMemorySize, POOL_SMEM);
  st = cudaGetLastError();
  if (st != cudaSuccess) { r4_destroy(e); return fail(nullptr, R4_ERR_CUDA, std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(st)); }
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  if (cudaStreamCreateWithPriority(&e->side, cudaStreamNonBlocking, prio_lo) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming) != cudaSuccess) {
    r4_destroy(e); return fail(nullptr, R4_ERR_CUDA, "r4_create: stream/event creation failed");
  }
  *out = e;
  return R4_OK;
}

void r4_destroy(r4_env* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  for (void* p : e->owned) cudaFree(p);
  void* own[] = {e->row_idx, e->prev_actions, e->amask, e->sflag, e->item_vec, e->price, e->special, e->action_emb};
  for (void* p : own) if (p) cudaFree(p);
  DevBuf* bufs[] = {&e->c0.H, &e->c0.Kp, &e->c1const.H, &e->c1const.Kp, &e->c1page.H, &e->c1page.Kp,
                    &e->c0.XT, &e->c1const.XT, &e->c1page.XT,
                    &e->ws_cat, &e->ws_dense, &e->ws_scores, &e->ws_allf, &e->ws_tmp, &e->ws_obs, &e->ws_p1,
                    &e->ws_xin, &e->ws_ids0, &e->ws_ids1, &e->ws_q, &e->ws_seq, &e->ws_cgx, &e->ws_part};
  for (DevBuf* b : bufs) if (b->p) cudaFree(b->p);
  if (e->side) cudaStreamDestroy(e->side);
  if (e->ev_fork) cudaEventDestroy(e->ev_fork);
  if (e->ev_join) cudaEventDestroy(e->ev_join);
  for (auto& pe : e->pending) { cudaEventDestroy(pe.a); cudaEventDestroy(pe.b); }
  for (cudaEvent_t ev : e->evpool) cudaEventDestroy(ev);
  delete e;
}

int r4_load_items(r4_env* e, const double* item_vec, int vec_dim, const double* price, const uint8_t* special,
                  const double* action_emb, int emb_dim, int n) {
  if (!e || !item_vec || !price || !special || !action_emb) return fail(e, R4_ERR_ARG, "r4_load_items: null argument");
  if (n != e->A) return fail(e, R4_ERR_ARG, "r4_load_items: n must equal action_size");
  if (vec_dim != VEC) return fail(e, R4_ERR_ARG, "r4_load_items: item vectors must have 40 dims");
  int want = (e->cfg.flags & R4_FLAG_ONEHOT) ? e->A : e->cfg.action_emb_size;
  if (emb_dim != want) return fail(e, R4_ERR_ARG, "r4_load_items: emb_dim does not match the config");
  R4_CUDA(e, cudaSetDevice(e->device));
  std::vector<float> v32((size_t)n * VEC);
  for (size_t i = 0; i < v32.size(); ++i) v32[i] = (float)item_vec[i];     // f64 text -> f32 (datautil.py:52-58)
  void* olds[] = {e->item_vec, e->price, e->special, e->action_emb};
  for (void* p : olds) if (p) cudaFree(p);
  e->item_vec = nullptr; e->price = nullptr; e->special = nullptr; e->action_emb = nullptr;
  R4_CUDA(e, cudaMalloc(&e->item_vec, v32.size() * 4));
  R4_CUDA(e, cudaMalloc(&e->price, (size_t)n * 8));
  R4_CUDA(e, cudaMalloc(&e->special, (size_t)n));
  R4_CUDA(e, cudaMalloc(&e->action_emb, (size_t)n * emb_dim * 8));
  R4_CUDA(e, cudaMemcpy(e->item_vec, v32.data(), v32.size() * 4, cudaMemcpyHostToDevice));
  R4_CUDA(e, cudaMemcpy(e->price, price, (size_t)n * 8, cudaMemcpyHostToDevice));
  R4_CUDA(e, cudaMemcpy(e->special, special, (size_t)n, cudaMemcpyHostToDevice));
  R4_CUDA(e, cudaMemcpy(e->action_emb, action_emb, (size_t)n * emb_dim * 8, cudaMemcpyHostToDevice));
  e->emb_dim = emb_dim;
  e->items_ready = true;
  return R4_OK;
}

int r4_load_weight(r4_env* e, const char* name, const float* data, const int64_t* shape, int rank) {
  if (!e || !name || !data || !shape || rank < 1) return fail(e, R4_ERR_ARG, "r4_load_weight: bad argument");
  size_t n = 1;
  for (int i = 0; i < rank; ++i) n *= (size_t)shape[i];
  R4_CUDA(e, cudaSetDevice(e->device));
  std::vector<float>& v = e->hw[name];
  v.resize(n);
  R4_CUDA(e, cudaMemcpy(v.data(), data, n * 4, cudaMemcpyDefault));
  e->weights_ready = false;
  return R4_OK;
}

int r4_finalize_weights(r4_env* e, void* stream) {
  if (!e) return R4_ERR_ARG;
  R4_CUDA(e, cudaSetDevice(e->device));
  const size_t Hh = (size_t)e->hash;
  struct Need { const char* n; size_t sz; };
  if (e->sim == R4_SIM_LSTM) {
    // W-table of nets/lstm.py:8-45 (rl4rs_b200/synth.py: lstm_weight_shapes): Keras GRU layers = kernel [128, 384],
    // recurrent kernel [128, 384], ONE bias [384], gate columns [z | r | h].  The recurrence kernel wants [r | u | c]
    // (u = Keras z), the x-side projection carries the whole bias.
    std::vector<Need> need = {{"emb_cat", Hh * EMB}, {"emb_seq", Hh * EMB}, {"dense_w1", (size_t)NDENSE * HU}, {"dense_b1", HU},
                              {"dense_w2", (size_t)HU * HU}, {"dense_b2", HU}, {"cgru_k", (size_t)EMB * 3 * EMB},
                              {"cgru_rk", (size_t)EMB * 3 * EMB}, {"cgru_b", 3 * EMB}, {"sgru0_k", (size_t)EMB * 3 * EMB},
                              {"sgru0_rk", (size_t)EMB * 3 * EMB}, {"sgru0_b", 3 * EMB}, {"sgru1_k", (size_t)EMB * 3 * EMB},
                              {"sgru1_rk", (size_t)EMB * 3 * EMB}, {"sgru1_b", 3 * EMB},
                              {"obs_w", (size_t)(4 * EMB + NCAT * EMB) * OBSD}, {"obs_b", OBSD}, {"rew_w", OBSD * 2}, {"rew_b", 2}};
    for (auto& nd : need)
      if (!hw_get(e, nd.n, nd.sz)) return fail(e, R4_ERR_ARG, std::string("r4_finalize_weights(lstm): missing or mis-shaped ") + nd.n);
    for (void* p : e->owned) cudaFree(p);
    e->owned.clear();
    int rc;
    if ((rc = upload(e, e->hw["emb_cat"], &e->emb_cat)) || (rc = upload(e, e->hw["emb_seq"], &e->emb_seq)) ||
        (rc = upload(e, e->hw["dense_b1"], &e->b1)) || (rc = upload(e, e->hw["dense_b2"], &e->b2)) ||
        (rc = upload(e, e->hw["obs_b"], &e->bo)) || (rc = upload(e, e->hw["rew_w"], &e->wr)) ||
        (rc = upload(e, e->hw["rew_b"], &e->br)) ||
        (rc = upload_image(e, e->hw["dense_w1"].data(), NDENSE, HU, &e->w1_img)) ||
        (rc = upload_image(e, e->hw["dense_w2"].data(), HU, HU, &e->w2_img)) ||
        (rc = upload_image(e, e->hw["obs_w"].data(), 4 * EMB + NCAT * EMB, OBSD, &e->wo_img, HEAD_BNT))) return rc;
    auto keras_gru = [&](const std::string& pre, uint8_t** wx_img, float** bx_dev, uint8_t** rec_img) -> int {
      const float* k = e->hw[pre + "_k"].data(); const float* rk = e->hw[pre + "_rk"].data(); const float* b = e->hw[pre + "_b"].data();
      std::vector<float> wx((size_t)EMB * XIN_LD), bx(XIN_LD), wgh((size_t)EMB * 2 * EMB), wch((size_t)EMB * EMB);
      const int src_of[3] = {EMB, 0, 2 * EMB};            // ours [r | u | c] <- Keras [z | r | h] column blocks
      for (int kk = 0; kk < EMB; ++kk)
        for (int g = 0; g < 3; ++g)
          for (int n = 0; n < EMB; ++n) {
            wx[(size_t)kk * XIN_LD + g * EMB + n] = k[(size_t)kk * 3 * EMB + src_of[g] + n];
            const float r = rk[(size_t)kk * 3 * EMB + src_of[g] + n];
            if (g < 2) wgh[(size_t)kk * 2 * EMB + g * EMB + n] = r; else wch[(size_t)kk * EMB + n] = r;
          }
      for (int g = 0; g < 3; ++g) for (int n = 0; n < EMB; ++n) bx[g * EMB + n] = b[src_of[g] + n];
      std::vector<uint8_t> gi(r4tc::G1_IMAGE_BYTES);
      r4tc::build_gru_image(wgh.data(), wch.data(), gi.data());
      int rc2;
      if ((rc2 = upload(e, gi, rec_img)) || (rc2 = upload(e, bx, bx_dev)) || (rc2 = upload_image(e, wx.data(), EMB, XIN_LD, wx_img))) return rc2;
      return R4_OK;
    };
    if ((rc = keras_gru("cgru", &e->cg_wx_img, &e->cg_bx, &e->cg_img)) ||
        (rc = keras_gru("sgru0", &e->ps[0].gru_wx_img, &e->ps[0].gru_bx, &e->ps[0].gru_img)) ||
        (rc = keras_gru("sgru1", &e->ps[1].gru_wx_img, &e->ps[1].gru_bx, &e->ps[1].gru_img))) return rc;
    e->hw.clear();
    e->weights_ready = true;
    // SlateRecEnv's second sequence is the constant [0] (slate.py:75 -> 64 x id 0): cache its last GRU state once
    cudaStream_t st = S(stream);
    if ((rc = reserve(e, e->ws_ids1, (size_t)std::max(e->B, 1) * MAXLEN * 4))) return rc;
    R4_CUDA(e, cudaMemsetAsync(e->ws_ids1.p, 0, (size_t)MAXLEN * 4, st));
    if ((rc = build_cache(e, 1, reinterpret_cast<const int32_t*>(e->ws_ids1.p), 1, e->c1const, st))) return rc;
    return R4_OK;
  }
  if (e->sim == R4_SIM_WIDEDEEP) {
    // W-table of nets/widedeep.py:8-45: emb_cat, dense tower, emb_seq (ONE table for both sequences), fc [256,256] (the
    // Dense on the pooled sequences, :34), simulator_reward [3072,2]; 'simulator_obs' is a Concatenate (no weights)
    std::vector<Need> need = {{"emb_cat", Hh * EMB}, {"emb_seq", Hh * EMB}, {"dense_w1", (size_t)NDENSE * HU}, {"dense_b1", HU},
                              {"dense_w2", (size_t)HU * HU}, {"dense_b2", HU}, {"fc_w", (size_t)2 * EMB * 2 * EMB}, {"fc_b", 2 * EMB},
                              {"rew_w", (size_t)OBSD_WD * 2}, {"rew_b", 2}};
    for (auto& nd : need)
      if (!hw_get(e, nd.n, nd.sz)) return fail(e, R4_ERR_ARG, std::string("r4_finalize_weights(widedeep): missing or mis-shaped ") + nd.n);
    for (void* p : e->owned) cudaFree(p);
    e->owned.clear();
    int rc;
    if ((rc = upload(e, e->hw["emb_cat"], &e->emb_cat)) || (rc = upload(e, e->hw["emb_seq"], &e->emb_seq)) ||
        (rc = upload(e, e->hw["dense_b1"], &e->b1)) || (rc = upload(e, e->hw["dense_b2"], &e->b2)) ||
        (rc = upload(e, e->hw["fc_b"], &e->fcb)) || (rc = upload(e, e->hw["rew_w"], &e->wr)) ||
        (rc = upload(e, e->hw["rew_b"], &e->br)) ||
        (rc = upload_image(e, e->hw["dense_w1"].data(), NDENSE, HU, &e->w1_img)) ||
        (rc = upload_image(e, e->hw["dense_w2"].data(), HU, HU, &e->w2_img)) ||
        (rc = upload_image(e, e->hw["fc_w"].data(), 2 * EMB, 2 * EMB, &e->fc_img))) return rc;
    e->hw.clear();
    e->weights_ready = true;
    return R4_OK;
  }
  if (e->sim == R4_SIM_DNN) {
    // W-table of nets/dnn.py:8-45: emb_cat [H,128], dense tower, fc [256,256] (the unnamed Dense of :34), simulator_obs
    // [256,256], simulator_reward [256,2].  The graph's second Embedding (sequence_input_concat) feeds nothing.
    std::vector<Need> need = {{"emb_cat", Hh * EMB}, {"dense_w1", (size_t)NDENSE * HU}, {"dense_b1", HU},
                              {"dense_w2", (size_t)HU * HU}, {"dense_b2", HU}, {"fc_w", (size_t)2 * HU * OBSD}, {"fc_b", OBSD},
                              {"obs_w", (size_t)OBSD * OBSD}, {"obs_b", OBSD}, {"rew_w", OBSD * 2}, {"rew_b", 2}};
    for (auto& nd : need)
      if (!hw_get(e, nd.n, nd.sz)) return fail(e, R4_ERR_ARG, std::string("r4_finalize_weights(dnn): missing or mis-shaped ") + nd.n);
    for (void* p : e->owned) cudaFree(p);
    e->owned.clear();
    int rc;
    if ((rc = upload(e, e->hw["emb_cat"], &e->emb_cat)) || (rc = upload(e, e->hw["dense_b1"], &e->b1)) ||
        (rc = upload(e, e->hw["dense_b2"], &e->b2)) || (rc = upload(e, e->hw["fc_b"], &e->fcb)) ||
        (rc = upload(e, e->hw["obs_b"], &e->bo)) || (rc = upload(e, e->hw["rew_w"], &e->wr)) ||
        (rc = upload(e, e->hw["rew_b"], &e->br)) ||
        (rc = upload_image(e, e->hw["dense_w1"].data(), NDENSE, HU, &e->w1_img)) ||
        (rc = upload_image(e, e->hw["dense_w2"].data(), HU, HU, &e->w2_img)) ||
        (rc = upload_image(e, e->hw["fc_w"].data(), 2 * HU, OBSD, &e->fc_img)) ||
        (rc = upload_image(e, e->hw["obs_w"].data(), OBSD, OBSD, &e->wo_img))) return rc;
    e->hw.clear();
    e->weights_ready = true;
    return R4_OK;
  }
  std::vector<Need> need = {{"emb_cat", Hh * EMB}, {"emb_seq", Hh * EMB}, {"dense_w1", (size_t)NDENSE * HU},
                            {"dense_b1", HU}, {"dense_w2", (size_t)HU * HU}, {"dense_b2", HU},
                            {"obs_w", (size_t)ALLF * OBSD}, {"obs_b", OBSD}, {"rew_w", OBSD * 2}, {"rew_b", 2}};
  for (auto& nd : need)
    if (!hw_get(e, nd.n, nd.sz)) return fail(e, R4_ERR_ARG, std::string("r4_finalize_weights: missing or mis-shaped ") + nd.n);
  for (void* p : e->owned) cudaFree(p);
  e->owned.clear();
  int rc;
#define UP(dst, nm) if ((rc = upload(e, e->hw[nm], &(dst)))) return rc;
  UP(e->emb_cat, "emb_cat"); UP(e->emb_seq, "emb_seq"); UP(e->w1, "dense_w1"); UP(e->b1, "dense_b1");
  UP(e->w2, "dense_w2"); UP(e->b2, "dense_b2"); UP(e->wo, "obs_w"); UP(e->bo, "obs_b");
  UP(e->wr, "rew_w"); UP(e->br, "rew_b");
#undef UP
  if ((rc = upload_image(e, e->hw["dense_w1"].data(), NDENSE, HU, &e->w1_img)) ||
      (rc = upload_image(e, e->hw["dense_w2"].data(), HU, HU, &e->w2_img)) ||
      (rc = upload_image(e, e->hw["obs_w"].data(), ALLF, OBSD, &e->wo_img, HEAD_BNT))) return rc;
  for (int i = 0; i < 2; ++i) {
    std::string si = std::to_string(i);
    const float* gwg = hw_get(e, "gru" + si + "_wg", (size_t)2 * EMB * 2 * EMB);
    const float* gbg = hw_get(e, "gru" + si + "_bg", 2 * EMB);
    const float* gwc = hw_get(e, "gru" + si + "_wc", (size_t)2 * EMB * EMB);
    const float* gbc = hw_get(e, "gru" + si + "_bc", EMB);
    const float* aw1 = hw_get(e, "att" + si + "_w1", (size_t)4 * EMB * AH1);
    const float* ab1 = hw_get(e, "att" + si + "_b1", AH1);
    const float* aw2 = hw_get(e, "att" + si + "_w2", (size_t)AH1 * AH2);
    const float* ab2 = hw_get(e, "att" + si + "_b2", AH2);
    const float* akv = hw_get(e, "att" + si + "_k", AH2);
    const float* abk = hw_get(e, "att" + si + "_b", 1);
    const float* uwg = hw_get(e, "augru" + si + "_wg", (size_t)(EMB + AUH) * 2 * AUH);
    const float* ubg = hw_get(e, "augru" + si + "_bg", 2 * AUH);
    const float* uwc = hw_get(e, "augru" + si + "_wc", (size_t)(EMB + AUH) * AUH);
    const float* ubc = hw_get(e, "augru" + si + "_bc", AUH);
    if (!gwg || !gbg || !gwc || !gbc || !aw1 || !ab1 || !aw2 || !ab2 || !akv || !abk || !uwg || !ubg || !uwc || !ubc)
      return fail(e, R4_ERR_ARG, "r4_finalize_weights: missing or mis-shaped per-sequence weight (seq " + si + ")");
    PerSeq& w = e->ps[i];
    // GRU-1 (TF1 GRUCell): gate kernel [x;h] x [r|u], candidate kernel [x;h] x c
    std::vector<float> wx((size_t)EMB * XIN_LD), bx(XIN_LD), wgh((size_t)EMB * 2 * EMB), wch((size_t)EMB * EMB);
    for (int k = 0; k < EMB; ++k) {
      for (int n = 0; n < 2 * EMB; ++n) wx[(size_t)k * XIN_LD + n] = gwg[(size_t)k * 2 * EMB + n];
      for (int n = 0; n < EMB; ++n) wx[(size_t)k * XIN_LD + 2 * EMB + n] = gwc[(size_t)k * EMB + n];
      for (int n = 0; n < 2 * EMB; ++n) wgh[(size_t)k * 2 * EMB + n] = gwg[(size_t)(EMB + k) * 2 * EMB + n];
      for (int n = 0; n < EMB; ++n) wch[(size_t)k * EMB + n] = gwc[(size_t)(EMB + k) * EMB + n];
    }
    for (int n = 0; n < 2 * EMB; ++n) bx[n] = gbg[n];
    for (int n = 0; n < EMB; ++n) bx[2 * EMB + n] = gbc[n];
    // AUGRU (VecAttGRUCell) input halves + attention key half
    std::vector<float> awx((size_t)EMB * XK_LD), abx(XK_LD, 0.f), awgh((size_t)AUH * 2 * AUH), awch((size_t)AUH * AUH);
    std::vector<float> wqd((size_t)EMB * AH1), wp((size_t)EMB * AH1);
    for (int k = 0; k < EMB; ++k) {
      for (int n = 0; n < 2 * AUH; ++n) awx[(size_t)k * XK_LD + n] = uwg[(size_t)k * 2 * AUH + n];
      for (int n = 0; n < AUH; ++n) awx[(size_t)k * XK_LD + XK_C + n] = uwc[(size_t)k * AUH + n];
      for (int n = 0; n < AH1; ++n) {
        float wq = aw1[(size_t)k * AH1 + n], wk = aw1[(size_t)(EMB + k) * AH1 + n];
        float wd = aw1[(size_t)(2 * EMB + k) * AH1 + n], wpp = aw1[(size_t)(3 * EMB + k) * AH1 + n];
        awx[(size_t)k * XK_LD + XK_K + n] = wk - wd;        // keys * (Wk - Wd)
        wqd[(size_t)k * AH1 + n] = wq + wd;                 // query * (Wq + Wd)
        wp[(size_t)k * AH1 + n] = wpp;                      // (query*keys) * Wp
      }
    }
    for (int n = 0; n < 2 * AUH; ++n) abx[n] = ubg[n];
    for (int n = 0; n < AUH; ++n) abx[XK_C + n] = ubc[n];
    for (int k = 0; k < AUH; ++k) {
      for (int n = 0; n < 2 * AUH; ++n) awgh[(size_t)k * 2 * AUH + n] = uwg[(size_t)(EMB + k) * 2 * AUH + n];
      for (int n = 0; n < AUH; ++n) awch[(size_t)k * AUH + n] = uwc[(size_t)(EMB + k) * AUH + n];
    }
    {
      std::vector<uint8_t> gi(r4tc::G1_IMAGE_BYTES);
      r4tc::build_gru_image(wgh.data(), wch.data(), gi.data());
      if ((rc = upload(e, gi, &w.gru_img))) return rc;
    }
    if ((rc = upload_image(e, wx.data(), EMB, XIN_LD, &w.gru_wx_img)) ||
        (rc = upload_image(e, awx.data(), EMB, XK_LD, &w.au_wx_img))) return rc;
    {
      std::vector<uint8_t> wpi(r4tc::S_IMG_BYTES);      // Wp image, then the W2 image of k_scores_tc2
      r4tc::build_scores_image2(wp.data(), aw2, wpi.data());
      if ((rc = upload(e, wpi, &w.wp_img))) return rc;
    }
    std::vector<uint8_t> img(r4tc::W_IMAGE_BYTES);
    r4tc::build_pair_image(awgh.data(), awch.data(), img.data());
    if ((rc = upload(e, img, &w.au_pair_img))) return rc;
    {
      int trc = r4tc::make_pair_tensor_map(w.au_pair_img, &w.au_pair_tmap);
      w.au_pair_tmap_ok = trc == 0;
      if (trc) return fail(e, R4_ERR_CUDA, "r4_finalize_weights: cuTensorMapEncodeTiled failed for the AUGRU pair weight image");
    }
    std::vector<float> vb1(ab1, ab1 + AH1), vw2(aw2, aw2 + AH1 * AH2), vb2(ab2, ab2 + AH2), vkv(akv, akv + AH2);
    if ((rc = upload(e, wx, &w.gru_wx)) || (rc = upload(e, bx, &w.gru_bx)) || (rc = upload(e, wgh, &w.gru_wgh)) ||
        (rc = upload(e, wch, &w.gru_wch)) || (rc = upload(e, awx, &w.au_wx)) || (rc = upload(e, abx, &w.au_bx)) ||
        (rc = upload(e, awgh, &w.au_wgh)) || (rc = upload(e, awch, &w.au_wch)) || (rc = upload(e, wqd, &w.wqd)) ||
        (rc = upload(e, wp, &w.wp)) || (rc = upload(e, vb1, &w.ab1)) || (rc = upload(e, vw2, &w.aw2)) ||
        (rc = upload(e, vb2, &w.ab2)) || (rc = upload(e, vkv, &w.akv)))
      return rc;
    w.abk = abk[0];
  }
  e->hw.clear();
  e->weights_ready = true;
  // SlateRecEnv's second sequence is the constant [0] (slate.py:75 -> 64 x id 0): cache it once.
  cudaStream_t st = S(stream);
  if ((rc = reserve(e, e->ws_ids1, (size_t)std::max(e->B, 1) * MAXLEN * 4))) return rc;
  R4_CUDA(e, cudaMemsetAsync(e->ws_ids1.p, 0, (size_t)MAXLEN * 4, st));
  if ((rc = build_cache(e, 1, reinterpret_cast<const int32_t*>(e->ws_ids1.p), 1, e->c1const, st))) return rc;
  return R4_OK;
}

int r4_load_log(r4_env* e, const int32_t* user_cat, const float* user_dense, const int32_t* user_seq,
                const int32_t* logged_items, const uint8_t* feedback, int64_t n_rows, int n_slots) {
  if (!e || !user_cat || !user_dense || !user_seq || !logged_items || !feedback || n_rows < 1 || n_slots < 1)
    return fail(e, R4_ERR_ARG, "r4_load_log: bad argument");
  if (n_rows > 0x7fffffffLL) return fail(e, R4_ERR_ARG, "r4_load_log: more than 2^31-1 rows");
  e->log_cat = user_cat; e->log_dense = user_dense; e->log_seq = user_seq; e->log_items = logged_items;
  e->log_fb = feedback; e->log_n = n_rows; e->log_slots = n_slots;
  e->has_reset = false;
  return R4_OK;
}

int r4_reset(r4_env* e, const int32_t* row_idx, const r4_out* out, void* stream) {
  if (!e || !row_idx) return fail(e, R4_ERR_ARG, "r4_reset: null argument");
  if (!e->weights_ready || !e->items_ready || !e->log_cat)
    return fail(e, R4_ERR_STATE, "r4_reset: load items, weights (+finalize) and log first");
  R4_CUDA(e, cudaSetDevice(e->device));
  cudaStream_t st = S(stream);
  int rc;
  const int B = e->B;
  R4_CUDA(e, cudaMemcpyAsync(e->row_idx, row_idx, (size_t)B * 4, cudaMemcpyDeviceToDevice, st));
  e->cur_steps = 0;
  e->c1_is_page = false;
  k_init_state<<<(B + 3) / 4, 128, 0, st>>>(B, e->T, e->A, e->words, e->prev_actions, e->amask, e->sflag,
                                             out ? out->action_mask : nullptr, 0);
  R4_LAUNCH_CHECK(e, "k_init_state");
  if ((rc = reserve(e, e->ws_ids0, (size_t)B * MAXLEN * 4))) return rc;
  k_seq_ids<<<(B * MAXLEN + 255) / 256, 256, 0, st>>>(B, e->T, 0, e->row_idx, e->log_seq, e->prev_actions,
                                                       (int32_t*)e->ws_ids0.p, nullptr, out ? out->seq : nullptr);
  R4_LAUNCH_CHECK(e, "k_seq_ids");
  e->has_reset = true;
  // user-history GRU-1 + input projections: once per episode (they do not depend on the actions); the dnn simulator
  // has no sequence branch
  if ((e->sim == R4_SIM_DIEN || e->sim == R4_SIM_LSTM) && (rc = build_cache(e, 0, (const int32_t*)e->ws_ids0.p, B, e->c0, st))) return rc;
  if ((rc = obs_pass(e, 0, 0, out, st))) return rc;
  if (out && out->reward) { k_fill_f64<<<(B + 255) / 256, 256, 0, st>>>(B, 0.0, out->reward); R4_LAUNCH_CHECK(e, "k_fill_f64"); }
  if (out && out->done) { k_fill_u8<<<(B + 255) / 256, 256, 0, st>>>(B, 0, out->done); R4_LAUNCH_CHECK(e, "k_fill_u8"); }
  if ((rc = write_masked_actions(e, out, st))) return rc;
  return R4_OK;
}

int r4_step(r4_env* e, const void* action, int action_is_f64, const r4_out* out, void* stream) {
  if (!e || !action) return fail(e, R4_ERR_ARG, "r4_step: null argument");
  if (!e->has_reset) return fail(e, R4_ERR_STATE, "r4_step: reset first");
  if (e->cur_steps >= e->T)   // the reference raises IndexError at slate.py:198
    return fail(e, R4_ERR_STATE, "r4_step: episode is over (cur_steps == max_steps)");
  R4_CUDA(e, cudaSetDevice(e->device));
  cudaStream_t st = S(stream);
  int rc;
  const int B = e->B, cur = e->cur_steps;
  bool conti = (e->cfg.flags & R4_FLAG_CONTI) != 0;
  // SeqSlate: entering a new page, the second sequence becomes the items of all previous pages
  // (seqslate.py:109-110) -> rebuild its GRU-1 cache once per page.
  if ((e->sim == R4_SIM_DIEN || e->sim == R4_SIM_LSTM) && e->seq && cur > 0 && cur % e->P == 0) {
    if ((rc = reserve(e, e->ws_ids1, (size_t)B * MAXLEN * 4))) return rc;
    k_seq_ids<<<(B * MAXLEN + 255) / 256, 256, 0, st>>>(B, e->T, cur, e->row_idx, e->log_seq, e->prev_actions,
                                                         nullptr, (int32_t*)e->ws_ids1.p, nullptr);
    R4_LAUNCH_CHECK(e, "k_seq_ids");
    if ((rc = build_cache(e, 1, (const int32_t*)e->ws_ids1.p, B, e->c1page, st))) return rc;
    e->c1_is_page = true;
  }
  ActParams ap{B, e->T, e->P, e->A, e->words, e->seq, conti ? 1 : 0, e->emb_dim, cur, action_is_f64};
  { ProfScope ps(e, SL_ACT, st, (double)B);
  k_act<<<(B + 3) / 4, 128, 0, st>>>(ap, action, e->action_emb, e->special, e->prev_actions, e->amask, e->sflag,
                                      out ? out->chosen : nullptr, out ? out->action_mask : nullptr); }
  R4_LAUNCH_CHECK(e, "k_act");
  e->cur_steps = cur + 1;
  if (out && out->seq) {
    int p0 = e->seq ? cur / e->P * e->P : 0;
    k_seq_ids<<<(B * MAXLEN + 255) / 256, 256, 0, st>>>(B, e->T, p0, e->row_idx, e->log_seq, e->prev_actions,
                                                         nullptr, nullptr, out->seq);
    R4_LAUNCH_CHECK(e, "k_seq_ids");
  }
  const bool pay = e->seq ? (e->cur_steps % e->P == 0) : (e->cur_steps >= e->T);
  // paying step with a network observation and no feature outputs: the reward pass delivers the observation as well
  const bool reuse = augru_opts().pay_obs_reuse && pay && out && out->reward && out->obs && !out->cat && !out->dense &&
                     !(e->cfg.flags & R4_FLAG_RAWSTATE);
  if (!reuse && (rc = obs_pass(e, 1, cur, out, st))) return rc;
  if (out && out->reward) {
    if (pay) { if ((rc = reward_pass(e, e->cur_steps, out, st, reuse ? out->obs : nullptr))) return rc; }
    else { k_fill_f64<<<(B + 255) / 256, 256, 0, st>>>(B, 0.0, out->reward); R4_LAUNCH_CHECK(e, "k_fill_f64"); }
  }
  if (out && out->done) {       // base.py:165-168 with the pre-increment step (Q1)
    k_fill_u8<<<(B + 255) / 256, 256, 0, st>>>(B, cur < e->T - 1 ? 0 : 1, out->done);
    R4_LAUNCH_CHECK(e, "k_fill_u8");
  }
  if ((rc = write_masked_actions(e, out, st))) return rc;
  return R4_OK;
}

int r4_offline_action(r4_env* e, int32_t* items, double* emb, void* stream) {
  if (!e || (!items && !emb)) return fail(e, R4_ERR_ARG, "r4_offline_action: null argument");
  if (!e->has_reset) return fail(e, R4_ERR_STATE, "r4_offline_action: reset first");
  R4_CUDA(e, cudaSetDevice(e->device));
  k_offline_action<<<(e->B + 3) / 4, 128, 0, S(stream)>>>(e->B, e->log_slots, e->cur_steps, e->T, e->emb_dim,
                                                         e->row_idx, e->log_items, e->action_emb, items, emb);
  R4_LAUNCH_CHECK(e, "k_offline_action");
  return R4_OK;
}

int r4_offline_reward(r4_env* e, double* reward, void* stream) {
  if (!e || !reward) return fail(e, R4_ERR_ARG, "r4_offline_reward: null argument");
  if (!e->has_reset) return fail(e, R4_ERR_STATE, "r4_offline_reward: reset first");
  R4_CUDA(e, cudaSetDevice(e->device));
  int c = e->cur_steps, lo = 0, hi = 0;
  if (e->seq) {                       // seqslate.py:71-86 (hard-coded 9 at :74)
    if (c % 9 == 0 && c > 0) { lo = c - e->P; hi = c; }
  } else if (c >= e->T) { lo = 0; hi = e->log_slots; }   // slate.py:164-174: every logged slot
  if (hi > e->log_slots) hi = e->log_slots;
  k_offline_reward<<<(e->B + 127) / 128, 128, 0, S(stream)>>>(e->B, e->log_slots, lo, hi, e->row_idx, e->log_items,
                                                              e->log_fb, e->price, reward);
  R4_LAUNCH_CHECK(e, "k_offline_reward");
  return R4_OK;
}

int r4_violation(r4_env* e, int32_t* out, void* stream) {
  if (!e || !out) return fail(e, R4_ERR_ARG, "r4_violation: null argument");
  if (!e->has_reset) return fail(e, R4_ERR_STATE, "r4_violation: reset first");
  R4_CUDA(e, cudaSetDevice(e->device));
  k_violation<<<(e->B + 127) / 128, 128, 0, S(stream)>>>(e->B, e->T, e->P, e->seq, e->cur_steps, e->prev_actions,
                                                         e->special, out);
  R4_LAUNCH_CHECK(e, "k_violation");
  return R4_OK;
}

int r4_features(r4_env* e, int32_t* cat, float* dense, int32_t* seq, void* stream) {
  if (!e || (!cat && !dense && !seq)) return fail(e, R4_ERR_ARG, "r4_features: null argument");
  if (!e->has_reset) return fail(e, R4_ERR_STATE, "r4_features: reset first");
  R4_CUDA(e, cudaSetDevice(e->device));
  cudaStream_t st = S(stream);
  int rc;
  const int B = e->B, cur = e->cur_steps;
  if (cat || dense) {
    int32_t* c = cat; float* d = dense;
    if (!c) { if ((rc = reserve(e, e->ws_cat, (size_t)B * NCAT * 4))) return rc; c = (int32_t*)e->ws_cat.p; }
    if (!d) { if ((rc = reserve(e, e->ws_dense, (size_t)B * NDENSE * 4))) return rc; d = (float*)e->ws_dense.p; }
    if ((rc = assemble(e, cur == 0 ? 0 : 1, cur == 0 ? 0 : cur - 1, 1, 0, B, c, d, st))) return rc;
  }
  if (seq) {
    const int p0 = (e->seq && cur > 0) ? (cur - 1) / e->P * e->P : 0;
    k_seq_ids<<<(B * MAXLEN + 255) / 256, 256, 0, st>>>(B, e->T, p0, e->row_idx, e->log_seq, e->prev_actions, nullptr, nullptr, seq);
    R4_LAUNCH_CHECK(e, "k_seq_ids");
  }
  return R4_OK;
}

int r4_nearest_neighbor(r4_env* e, const void* action, int action_is_f64, int n, int32_t* out, void* stream) {
  if (!e || !action || !out || n < 1) return fail(e, R4_ERR_ARG, "r4_nearest_neighbor: bad argument");
  if (!e->items_ready) return fail(e, R4_ERR_STATE, "r4_nearest_neighbor: load items first");
  R4_CUDA(e, cudaSetDevice(e->device));
  k_knn_plain<<<(n + 3) / 4, 128, 0, S(stream)>>>(n, e->A, e->emb_dim, action_is_f64, action, e->action_emb, out);
  R4_LAUNCH_CHECK(e, "k_knn_plain");
  return R4_OK;
}

int r4_cur_steps(const r4_env* e) { return e ? e->cur_steps : -1; }
const int32_t* r4_prev_actions(const r4_env* e) { return e ? e->prev_actions : nullptr; }
int64_t r4_launch_count(const r4_env* e) { return e ? e->launches : 0; }

int r4_set_option(const char* key, int value) {
  if (!key) return fail(nullptr, R4_ERR_ARG, "r4_set_option: null key");
  AugruOpts& o = augru_opts();
  const std::string k(key);
  if (k == "augru_kernel" && (value == 0 || value == 2 || value == 3)) o.force = value;
  else if (k == "augru_cost_pair" && value > 0) o.cost_pair = value;
  else if (k == "augru_cost_pp" && value > 0) o.cost_pp = value;
  else if (k == "pay_obs_reuse" && (value == 0 || value == 1)) o.pay_obs_reuse = value;
  else if (k == "scores_shared_pct" && value >= 10 && value <= 100) o.scores_shared_pct = value;
  else return fail(nullptr, R4_ERR_ARG, "r4_set_option: unknown key or value out of range: " + k);
  return R4_OK;
}

int r4_augru_kernel_for(int ctas, int sms) { return (ctas < 1 || sms < 2) ? 0 : augru_rule(ctas, sms); }

int r4_profile(r4_env* e, int mode) {
  if (!e || mode < 0 || mode > 2) return fail(e, R4_ERR_ARG, "r4_profile: mode must be 0, 1 or 2");
  R4_CUDA(e, cudaSetDevice(e->device));
  R4_CUDA(e, cudaDeviceSynchronize());
  for (auto& pe : e->pending) { e->evpool.push_back(pe.a); e->evpool.push_back(pe.b); }
  e->pending.clear();
  for (auto& sl : e->slots) sl = r4_env::ProfSlot();
  e->prof_mode = mode;
  return R4_OK;
}

int r4_profile_read(r4_env* e, int slot, const char** name, double* ms, int64_t* launches, double* work) {
  if (!e || slot < 0) return fail(e, R4_ERR_ARG, "r4_profile_read: bad argument");
  if (slot >= SL_COUNT) return 1;                               // end of the slot list
  R4_CUDA(e, cudaSetDevice(e->device));
  for (auto& pe : e->pending) {
    R4_CUDA(e, cudaEventSynchronize(pe.b));
    float t = 0.f;
    R4_CUDA(e, cudaEventElapsedTime(&t, pe.a, pe.b));
    e->slots[pe.slot].ms += t; e->slots[pe.slot].n += 1;
    e->evpool.push_back(pe.a); e->evpool.push_back(pe.b);
  }
  e->pending.clear();
  if (name) *name = SLOT_NAMES[slot];
  if (ms) *ms = e->slots[slot].ms;
  if (launches) *launches = e->slots[slot].n;
  if (work) *work = e->slots[slot].work;
  return R4_OK;
}

int r4_copy_prev_actions(r4_env* e, int32_t* out, void* stream) {
  if (!e || !out) return fail(e, R4_ERR_ARG, "r4_copy_prev_actions: null argument");
  R4_CUDA(e, cudaSetDevice(e->device));
  R4_CUDA(e, cudaMemcpyAsync(out, e->prev_actions, (size_t)e->B * e->T * 4, cudaMemcpyDeviceToDevice, S(stream)));
  return R4_OK;
}

// ---- K12: policy / learner kernels (stateless) ---------------------------------------------------
#define R4_PCHECK(name)                                                                     \
  do {                                                                                      \
    cudaError_t _st = cudaGetLastError();                                                   \
    if (_st != cudaSuccess) return fail(nullptr, R4_ERR_CUDA, std::string(name) + ": " + cudaGetErrorString(_st)); \
  } while (0)

int r4_policy_num_params(int action_size) { return r4ppo::make_layout(action_size).n; }

int r4_policy_act(const float* params, const float* obs, const uint8_t* mask, int n, int action_size, int explore,
                  uint64_t seed, uint64_t counter, int32_t* action, float* logp, float* value, float* logits,
                  void* stream) {
  if (!params || !obs || !mask || !action || !logp || !value || n < 1 || action_size < 2 || action_size > 512)
    return fail(nullptr, R4_ERR_ARG, "r4_policy_act: bad argument");
  r4ppo::Layout L = r4ppo::make_layout(action_size);
  size_t smem = (size_t)(r4ppo::TS * r4ppo::OBS + r4ppo::TS * r4ppo::HID + r4ppo::TS * action_size + r4ppo::TS) * 4;
  static bool attr = false;
  if (!attr) { cudaFuncSetAttribute(r4ppo::k_policy_act, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024); attr = true; }
  r4ppo::k_policy_act<<<(n + r4ppo::TS - 1) / r4ppo::TS, r4ppo::NT, smem, S(stream)>>>(
      L, params, obs, mask, n, explore, seed, counter, action, logp, value, logits);
  R4_PCHECK("k_policy_act");
  return R4_OK;
}

static int policy_grad_impl(int mode, const float* params, const float* obs, const uint8_t* mask, const int64_t* action,
                            const float* old_logp, const float* old_logits, const float* old_value, const float* adv,
                            const float* target, const int64_t* idx, int n, int action_size, float clip, float vf_clip,
                            float vf_coeff, float kl_coeff, float ent_coeff, float inv_n, float* scratch, int G,
                            float* flat_grad, float* stats_accum, float stat_scale, void* stream, bool reduce, bool pdl = false) {
  if (!params || !obs || !mask || !action || !old_logits || !adv || !target || !scratch || !flat_grad || n < 1 ||
      G < 1 || action_size < 2 || action_size > 512 || (mode == 0 && (!old_logp || !old_value)))
    return fail(nullptr, R4_ERR_ARG, "r4_policy_grad: bad argument");
  r4ppo::Layout L = r4ppo::make_layout(action_size);
  r4ppo::LossHyper hp{mode, clip, vf_clip, vf_coeff, kl_coeff, ent_coeff, inv_n};
  const bool single = ((n + r4ppo::TS - 1) / r4ppo::TS) == G;      // one tile per CTA (PPO minibatch)
  const size_t head = single ? (size_t)(r4ppo::OBS * r4ppo::HID + ((r4ppo::HID * action_size + 3) & ~3)) : (size_t)((L.n + 3) & ~3);
  size_t smem = (head + r4ppo::TS * r4ppo::OBS + 2 * r4ppo::TS * r4ppo::HID + r4ppo::TS * action_size + 2 * r4ppo::TS) * 4;
  if (smem > 226 * 1024) return fail(nullptr, R4_ERR_ARG, "r4_policy_grad: action_size too large for the shared-memory layout");
  static size_t attr[2] = {0, 0};
  if (smem > attr[single]) {
    cudaError_t st_ = single
        ? cudaFuncSetAttribute(r4ppo::k_policy_grad<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
        : cudaFuncSetAttribute(r4ppo::k_policy_grad<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (st_ != cudaSuccess) return fail(nullptr, R4_ERR_CUDA, std::string("cudaFuncSetAttribute(k_policy_grad): ") + cudaGetErrorString(st_));
    attr[single] = smem;
  }
  float* partial = scratch;
  float* stat_partial = scratch + (size_t)G * L.n;
  if (single && pdl) {
    cudaLaunchConfig_t lc = {};
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[0].val.programmaticStreamSerializationAllowed = 1;
    lc.gridDim = dim3(G); lc.blockDim = dim3(r4ppo::NT); lc.dynamicSmemBytes = smem; lc.stream = S(stream); lc.attrs = at; lc.numAttrs = 1;
    cudaLaunchKernelEx(&lc, r4ppo::k_policy_grad<true>, L, hp, params, obs, mask, action, old_logp, old_logits, old_value, adv, target, idx, n,
                       partial, stat_partial);
  } else if (single)
    r4ppo::k_policy_grad<true><<<G, r4ppo::NT, smem, S(stream)>>>(L, hp, params, obs, mask, action, old_logp, old_logits,
                                                                 old_value, adv, target, idx, n, partial, stat_partial);
  else
    r4ppo::k_policy_grad<false><<<G, r4ppo::NT, smem, S(stream)>>>(L, hp, params, obs, mask, action, old_logp, old_logits,
                                                                  old_value, adv, target, idx, n, partial, stat_partial);
  R4_PCHECK("k_policy_grad");
  if (!reduce) return R4_OK;       // the caller folds the reduction into its optimiser kernel (r4_ppo_epoch)
  r4ppo::k_grad_reduce<<<(L.n + 255) / 256, 256, 0, S(stream)>>>(L.n, G, partial, flat_grad, stat_partial, stats_accum, stat_scale);
  R4_PCHECK("k_grad_reduce");
  return R4_OK;
}

int r4_policy_grad(int mode, const float* params, const float* obs, const uint8_t* mask, const int64_t* action,
                   const float* old_logp, const float* old_logits, const float* old_value, const float* adv,
                   const float* target, const int64_t* idx, int n, int action_size, float clip, float vf_clip,
                   float vf_coeff, float kl_coeff, float ent_coeff, float inv_n, float* scratch, int G,
                   float* flat_grad, float* stats_accum, float stat_scale, void* stream) {
  return policy_grad_impl(mode, params, obs, mask, action, old_logp, old_logits, old_value, adv, target, idx, n, action_size,
                          clip, vf_clip, vf_coeff, kl_coeff, ent_coeff, inv_n, scratch, G, flat_grad, stats_accum, stat_scale,
                          stream, true);
}

int r4_gae(const float* reward, const float* value, int T, int B, float gamma, float gamma_lambda, float* adv, float* target, void* stream) {
  if (!reward || !value || !adv || !target || T < 1 || B < 1) return fail(nullptr, R4_ERR_ARG, "r4_gae: bad argument");
  r4ppo::k_gae<<<(B + 255) / 256, 256, 0, S(stream)>>>(T, B, reward, value, gamma, gamma_lambda, adv, target);
  R4_PCHECK("k_gae");
  return R4_OK;
}

int r4_adam_step(float* params, const float* grad, float* m, float* v, int n, int step, float lr, float beta1,
                 float beta2, float eps, float grad_scale, float clip, float* norm_scratch, void* stream) {
  if (!params || !grad || !m || !v || n < 1 || step < 1 || (clip > 0.f && !norm_scratch))
    return fail(nullptr, R4_ERR_ARG, "r4_adam_step: bad argument");
  if (clip > 0.f) {
    cudaMemsetAsync(norm_scratch, 0, 4, S(stream));
    r4ppo::k_sumsq<<<32, 256, 0, S(stream)>>>(n, grad, norm_scratch);
    R4_PCHECK("k_sumsq");
  }
  r4ppo::k_adam<<<(n + 255) / 256, 256, 0, S(stream)>>>(n, params, grad, m, v, step, lr, beta1, beta2, eps, grad_scale,
                                                         clip > 0.f ? norm_scratch : nullptr, clip);
  R4_PCHECK("k_adam");
  return R4_OK;
}

int r4_ppo_epoch(float* params, const float* obs, const uint8_t* mask, const int64_t* action, const float* old_logp,
                 const float* old_logits, const float* old_value, const float* adv, const float* target,
                 const int64_t* perm, int n, int mb, int action_size, float clip, float vf_clip, float vf_coeff,
                 float kl_coeff, float ent_coeff, float* scratch, float* flat_grad, float* stats_accum, float* m,
                 float* v, int step0, float lr, float beta1, float beta2, float eps, float grad_clip,
                 float* norm_scratch, void* stream) {
  if (!perm || n < 1 || mb < 1 || mb > n || step0 < 0) return fail(nullptr, R4_ERR_ARG, "r4_ppo_epoch: bad argument");
  const int G = std::max(1, std::min((mb + r4ppo::TS - 1) / r4ppo::TS, 148));
  const int np = r4ppo::make_layout(action_size).n;
  int steps = 0;
  const bool fused = !(grad_clip > 0.f);      // global-norm clipping needs the reduced gradient first
  // programmatic dependent launch for the grad / optimiser chain of the epoch (R4_NO_PDL=1: plain stream order)
  static const bool pdl = getenv("R4_NO_PDL") == nullptr;
  if (!params || !m || !v || !flat_grad || !scratch) return fail(nullptr, R4_ERR_ARG, "r4_ppo_epoch: bad argument");
  for (int s = 0; s + mb <= n; s += mb, ++steps) {
    int rc = policy_grad_impl(0, params, obs, mask, action, old_logp, old_logits, old_value, adv, target, perm + s, mb,
                              action_size, clip, vf_clip, vf_coeff, kl_coeff, ent_coeff, 1.0f / mb, scratch, G, flat_grad,
                              stats_accum, 1.0f / mb, stream, !fused, fused && pdl);
    if (rc) return rc;
    if (fused && pdl) {
      cudaLaunchConfig_t lc = {};
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[0].val.programmaticStreamSerializationAllowed = 1;
      lc.gridDim = dim3((np + 255) / 256); lc.blockDim = dim3(256); lc.dynamicSmemBytes = 0; lc.stream = S(stream); lc.attrs = at; lc.numAttrs = 1;
      cudaLaunchKernelEx(&lc, r4ppo::k_reduce_adam, np, G, (const float*)scratch, flat_grad, (const float*)(scratch + (size_t)G * np), stats_accum,
                         1.0f / mb, params, m, v, step0 + steps + 1, lr, beta1, beta2, eps);
      R4_PCHECK("k_reduce_adam");
    } else if (fused) {
      r4ppo::k_reduce_adam<<<(np + 255) / 256, 256, 0, S(stream)>>>(np, G, scratch, flat_grad, scratch + (size_t)G * np, stats_accum,
                                                                    1.0f / mb, params, m, v, step0 + steps + 1, lr, beta1, beta2, eps);
      R4_PCHECK("k_reduce_adam");
    } else {
      rc = r4_adam_step(params, flat_grad, m, v, np, step0 + steps + 1, lr, beta1, beta2, eps, 1.0f, grad_clip, norm_scratch, stream);
      if (rc) return rc;
    }
  }
  return steps;
}

// ---- data-parallel learner: peer-memory gradient exchange (r4_comm.cuh) -------------------------------------
}  // extern "C"

struct r4_comm {
  int rank = 0, world = 1, n = 0, nblk = 0, device = 0;
  void* base = nullptr;
  size_t inbox_bytes = 0, bytes = 0;
  r4comm::Peers peers{};
  std::vector<void*> opened;
  uint32_t seq = 0;
  bool ready = false;
};

extern "C" {

int r4_comm_create(int rank, int world, int n_params, r4_comm** out) {
  if (!out || world < 1 || world > r4comm::MAX_WORLD || rank < 0 || rank >= world || n_params < 1)
    return fail(nullptr, R4_ERR_ARG, "r4_comm_create: bad argument (world <= 16)");
  *out = nullptr;
  r4_comm* c = new r4_comm();
  c->rank = rank; c->world = world; c->n = n_params; c->nblk = (n_params + r4comm::BLK - 1) / r4comm::BLK;
  cudaGetDevice(&c->device);
  c->inbox_bytes = (((size_t)2 * world * n_params * 4) + 255) & ~(size_t)255;
  c->bytes = c->inbox_bytes + (size_t)2 * world * c->nblk * 4;
  cudaError_t st = cudaMalloc(&c->base, c->bytes);
  if (st == cudaSuccess) st = cudaMemset(c->base, 0, c->bytes);
  if (st == cudaSuccess) st = cudaDeviceSynchronize();
  if (st != cudaSuccess) { if (c->base) cudaFree(c->base); delete c; return fail(nullptr, R4_ERR_CUDA, std::string("r4_comm_create: ") + cudaGetErrorString(st)); }
  c->peers.inbox[rank] = reinterpret_cast<float*>(c->base);
  c->peers.flags[rank] = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(c->base) + c->inbox_bytes);
  c->ready = world == 1;
  *out = c;
  return R4_OK;
}

int r4_comm_handle(r4_comm* c, void* handle_out_64) {
  if (!c || !handle_out_64) return fail(nullptr, R4_ERR_ARG, "r4_comm_handle: null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  cudaIpcMemHandle_t h;
  cudaError_t st = cudaIpcGetMemHandle(&h, c->base);
  if (st != cudaSuccess) return fail(nullptr, R4_ERR_CUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(st));
  memcpy(handle_out_64, &h, 64);
  return R4_OK;
}

int r4_comm_open(r4_comm* c, const void* handles, int n_handles) {
  if (!c || !handles || n_handles != c->world) return fail(nullptr, R4_ERR_ARG, "r4_comm_open: need one handle per rank");
  cudaSetDevice(c->device);
  for (int r = 0; r < c->world; ++r) {
    if (r == c->rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, reinterpret_cast<const uint8_t*>(handles) + (size_t)r * 64, 64);
    void* p = nullptr;
    cudaError_t st = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (st != cudaSuccess) {
      cudaGetLastError();
      return fail(nullptr, R4_ERR_CUDA, std::string("cudaIpcOpenMemHandle(rank ") + std::to_string(r) + "): " + cudaGetErrorString(st));
    }
    c->opened.push_back(p);
    c->peers.inbox[r] = reinterpret_cast<float*>(p);
    c->peers.flags[r] = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(p) + c->inbox_bytes);
  }
  c->ready = true;
  return R4_OK;
}

void r4_comm_destroy(r4_comm* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  for (void* p : c->opened) cudaIpcCloseMemHandle(p);
  if (c->base) cudaFree(c->base);
  delete c;
}

int r4_policy_grad_partial(int mode, const float* params, const float* obs, const uint8_t* mask, const int64_t* action,
                           const float* old_logp, const float* old_logits, const float* old_value, const float* adv,
                           const float* target, const int64_t* idx, int n, int action_size, float clip, float vf_clip,
                           float vf_coeff, float kl_coeff, float ent_coeff, float inv_n, float* scratch, int G,
                           void* stream) {
  return policy_grad_impl(mode, params, obs, mask, action, old_logp, old_logits, old_value, adv, target, idx, n, action_size,
                          clip, vf_clip, vf_coeff, kl_coeff, ent_coeff, inv_n, scratch, G, scratch /*unused*/, nullptr, 0.f,
                          stream, false);
}

static int exchange_launch(r4_comm* c, const float* scratch, int G, int np, float* flat, float* stats_accum, float stat_scale,
                           int do_adam, float* params, float* m, float* v, int step, float lr, float b1, float b2, float eps,
                           void* stream) {
  if (!c->ready) return fail(nullptr, R4_ERR_STATE, "r4_comm: open the peers' handles first (r4_comm_open)");
  if (np != c->n) return fail(nullptr, R4_ERR_ARG, "r4_comm: parameter count differs from the communicator's");
  ++c->seq;
  r4comm::k_exchange_adam<<<c->nblk, r4comm::BLK, 0, S(stream)>>>(np, G, scratch, flat, scratch + (size_t)G * np, stats_accum,
                                                                  stat_scale, c->peers, c->rank, c->world, c->seq, do_adam,
                                                                  params, m, v, step, lr, b1, b2, eps);
  R4_PCHECK("k_exchange_adam");
  return R4_OK;
}

int r4_grad_exchange(r4_comm* c, const float* scratch, int G, int action_size, float* flat_grad, float* stats_accum,
                     float stat_scale, void* stream) {
  if (!c || !scratch || !flat_grad || G < 1) return fail(nullptr, R4_ERR_ARG, "r4_grad_exchange: bad argument");
  return exchange_launch(c, scratch, G, r4ppo::make_layout(action_size).n, flat_grad, stats_accum, stat_scale, 0, nullptr, nullptr,
                         nullptr, 0, 0.f, 0.f, 0.f, 0.f, stream);
}

int r4_ppo_epoch_dist(r4_comm* c, float* params, const float* obs, const uint8_t* mask, const int64_t* action,
                      const float* old_logp, const float* old_logits, const float* old_value, const float* adv,
                      const float* target, const int64_t* perm, int n, int mb, int action_size, float clip,
                      float vf_clip, float vf_coeff, float kl_coeff, float ent_coeff, float* scratch, float* flat_grad,
                      float* stats_accum, float* m, float* v, int step0, float lr, float beta1, float beta2, float eps,
                      void* stream) {
  if (!c || !params || !perm || !m || !v || !scratch || n < 1 || mb < 1 || mb > n || step0 < 0)
    return fail(nullptr, R4_ERR_ARG, "r4_ppo_epoch_dist: bad argument");
  const int G = std::max(1, std::min((mb + r4ppo::TS - 1) / r4ppo::TS, 148));
  const int np = r4ppo::make_layout(action_size).n;
  const float inv = 1.0f / ((float)mb * (float)c->world);
  int steps = 0;
  for (int s = 0; s + mb <= n; s += mb, ++steps) {
    int rc = policy_grad_impl(0, params, obs, mask, action, old_logp, old_logits, old_value, adv, target, perm + s, mb,
                              action_size, clip, vf_clip, vf_coeff, kl_coeff, ent_coeff, inv, scratch, G, scratch, nullptr, 0.f,
                              stream, false);
    if (rc) return rc;
    // statistics stay per-rank means over this rank's mb samples (the trainer averages them over the ranks)
    rc = exchange_launch(c, scratch, G, np, flat_grad, stats_accum, 1.0f / (float)mb, 1, params, m, v, step0 + steps + 1, lr, beta1, beta2,
                         eps, stream);
    if (rc) return rc;
  }
  return steps;
}

int r4_dien_forward(r4_env* e, const int32_t* seq, const float* dense, const int32_t* cat, int n_rows,
                    float* obs, float* probs, void* stream) {
  if (!e || !seq || !dense || !cat || n_rows < 1) return fail(e, R4_ERR_ARG, "r4_dien_forward: bad argument");
  if (!e->weights_ready) return fail(e, R4_ERR_STATE, "r4_dien_forward: load + finalize weights first");
  R4_CUDA(e, cudaSetDevice(e->device));
  cudaStream_t st = S(stream);
  int rc;
  if (e->sim == R4_SIM_DNN || e->sim == R4_SIM_WIDEDEEP) {          // dnn: no sequence branch; widedeep: raw ids, no sequence cache
    rc = R4_OK;
    int chunk = std::min(n_rows, e->max_rows);
    for (int r0 = 0; !rc && r0 < n_rows; r0 += chunk) {
      int nr = std::min(chunk, n_rows - r0);
      if (e->sim == R4_SIM_WIDEDEEP) {
        if ((rc = reserve(e, e->ws_seq, (size_t)nr * 2 * MAXLEN * 4))) return rc;
        R4_CUDA(e, cudaMemcpyAsync(e->ws_seq.p, seq + (size_t)r0 * 2 * MAXLEN, (size_t)nr * 2 * MAXLEN * 4, cudaMemcpyDeviceToDevice, st));
      }
      rc = forward_rows(e, nr, r0, 1, cat + (size_t)r0 * NCAT, dense + (size_t)r0 * NDENSE, e->c0, 0, e->c0, 0,
                        obs ? obs + (size_t)r0 * e->obs_dim : nullptr, nullptr, probs ? probs + (size_t)r0 * 2 : nullptr, st);
    }
    return rc;
  }
  SeqCache t0, t1;
  DevBuf ids;
  if ((rc = reserve(e, ids, (size_t)2 * n_rows * MAXLEN * 4))) return rc;
  int32_t* i0 = (int32_t*)ids.p;
  int32_t* i1 = i0 + (size_t)n_rows * MAXLEN;
  R4_CUDA(e, cudaMemcpy2DAsync(i0, MAXLEN * 4, seq, 2 * MAXLEN * 4, MAXLEN * 4, n_rows, cudaMemcpyDeviceToDevice, st));
  R4_CUDA(e, cudaMemcpy2DAsync(i1, MAXLEN * 4, seq + MAXLEN, 2 * MAXLEN * 4, MAXLEN * 4, n_rows, cudaMemcpyDeviceToDevice, st));
  rc = build_cache(e, 0, i0, n_rows, t0, st);
  if (!rc) rc = build_cache(e, 1, i1, n_rows, t1, st);
  int chunk = std::min(n_rows, e->max_rows);
  for (int r0 = 0; !rc && r0 < n_rows; r0 += chunk) {
    int nr = std::min(chunk, n_rows - r0);
    rc = forward_rows(e, nr, r0, 1, cat + (size_t)r0 * NCAT, dense + (size_t)r0 * NDENSE, t0, 0, t1, 0,
                      obs ? obs + (size_t)r0 * OBSD : nullptr, nullptr, probs ? probs + (size_t)r0 * 2 : nullptr, st);
  }
  cudaStreamSynchronize(st);
  DevBuf* tmp[] = {&t0.H, &t0.Kp, &t0.XT, &t1.H, &t1.Kp, &t1.XT, &ids};
  for (DevBuf* b : tmp) if (b->p) cudaFree(b->p);
  return rc;
}

}  // extern "C"
