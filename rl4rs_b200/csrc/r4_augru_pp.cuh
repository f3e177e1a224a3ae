// r4_augru_pp.cuh -- the 2-CTA AUGRU recurrence with TWO independent recurrences in flight per CTA pair ("ping-pong"):
// both sequences of one 128-row tile share the pair's tensor pipe, TMEM, shared memory and epilogue warps.
//
// Why (ncu + in-kernel clocks on k_augru_pair2, round 2): one recurrence is a dependency chain
//     h -> [r,u gates] -> r*h -> [c gate] -> h'
// and a pair that works on one tile alternates between "tensor pipe waits for the epilogue" and "epilogue waits for the
// tensor pipe": 16.6 k cycles per step for 9.2 k cycles of MMAs (tensor pipe 58 % active), the epilogue warps 70 % busy.
// With two recurrences A, B the leader issues  [r,u]A [r,u]B [c]A [c]B  and the epilogue runs  R,U(A) R,U(B) C(A) C(B):
// whatever one side produces is consumed while the other side already has work queued, so neither waits in steady state.
// Cost model from the measured phase times (R 4.0 k + U 2.3 k + C 4.5 k per recurrence): ~21.6 k cycles per step for
// TWO tile-steps against 2 x 16.6 k -- 1.5x the throughput per SM pair.  It wins wherever a launch has more tiles than
// CTA pairs (reward passes, 8192-row batches); a 4096-row observation pass (32 tiles) still prefers k_augru_pair2, which
// spreads over 128 SMs (r4_capi.cu: augru_choice).
//
// What had to change against k_augru_pair2 to fit two recurrences into one SM pair:
//   * shared memory: r*h ALIASES h (one 64 KB A operand per recurrence and CTA, 2 x 64 KB + the 96 KB weight ring).  The
//     epilogue therefore writes r*h only after the u gate has retired (its MMAs read h): phase R waits for the commit of
//     [r,u] as a whole -- free in steady state, the epilogue is busy with the other recurrence meanwhile;
//   * TMEM: 256 columns per recurrence, c aliases r (r is consumed by phase R before the c gate starts), u keeps its own.
//     Because of the alias the next r gate may not start under the second half of phase C (it would overwrite c
//     accumulators that are still being read): ONE hand-over barrier per state instead of pair2's early/late halves --
//     the other recurrence fills the gap;
//   * registers: a thread owns one row x 64 columns of BOTH states (128 registers); gate inputs are walked in 8-column
//     chunks with a 3-deep rolling prefetch that runs across phase boundaries (32 registers), 16 + 16 for accumulators;
//   * the weight ring carries 48 stages per step (16 revolutions of the 3 stages: stage and parity stay compile-time).
// Same arithmetic, weight image and hand-over as k_augru_pair2 (r4_augru_pair2.cuh).  The weight ring is fed by
// tensor-map TMA: both CTAs issue cp.async.bulk.tensor.2d.cta_group::2 for their own half of the stage with the LEADER's
// "full" barrier as the completion target, and the leader's producer posts one expect_tx for both halves -- no relay
// thread, no remote arrive: the transaction count is the signal.
#pragma once
#include "r4_augru_pair2.cuh"

namespace r4tc {

constexpr int PP_SLOT_BYTES = 2 * P_A_BYTES;                     // one recurrence: A operand hi + lo (h, then r*h, then h')
constexpr int PP_SMEM_BYTES = 2 * PP_SLOT_BYTES + P_NST * P_STAGE_BYTES + 128;
constexpr int PP_USES = 2 * P_STAGES_PER_STEP;                   // 48 ring uses per step
static_assert(PP_USES % (2 * P_NST) == 0, "stage parity must repeat every step");
constexpr int PP_CH = 8, PP_NCH = 64 / PP_CH, PP_XD = 3;        // chunk width, chunks per phase, prefetch distance
constexpr int P2_TM_ROW_BYTES = 1024;                             // tensor-map row = 256 x u32
constexpr int P2_TM_BOX_ROWS = P_STAGE_BYTES / P2_TM_ROW_BYTES;   // 16 rows per ring stage

// this CTA's 16 KB box of the weight image -> own shared memory, completion bytes -> the barrier at `mbar_cluster`
// (a shared::cluster address: the leader's "full" barrier for both CTAs of the pair)
__device__ __forceinline__ void tma_box_cg2(uint32_t dst_smem, const CUtensorMap* tm, int c0, int c1, uint32_t mbar_cluster) {
  asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
               :: "r"(dst_smem), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(mbar_cluster) : "memory");
}

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
  uint32_t* u = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7])
               : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float* v) {
  const uint32_t* u = reinterpret_cast<const uint32_t*>(v);
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               :: "r"(taddr), "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]) : "memory");
}
// 8 consecutive columns (colbase % 8 == 0) of one lane, quad layout: two 128-bit loads
__device__ __forceinline__ void load_x8(float* dst, const float* ts, int colbase, int ln4) {
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(ts + (size_t)(colbase + 4 * g) * TM + ln4));
    dst[4 * g] = v.x; dst[4 * g + 1] = v.y; dst[4 * g + 2] = v.z; dst[4 * g + 3] = v.w;
  }
}

// One gate (8 ring stages) of the leader's issue stream; U0 = index of its first ring use inside the step.
template <int U0>
__device__ __forceinline__ void issue_gate_pp(uint32_t leader, uint32_t d_tmem, uint32_t aHi_lo, uint32_t aLo_lo, uint32_t b_lo,
                                              uint64_t* bar_full, uint64_t* bar_empty, uint64_t* half_bar, uint32_t half_par) {
  constexpr uint32_t idesc = make_idesc(TM, HID);
  constexpr uint32_t a_hi = desc_hi(A_SBO), b_hi = desc_hi(B_SBO);
#pragma unroll
  for (int s8 = 0; s8 < NKB; ++s8) {
    const int u = U0 + s8;
    const int stage = u % P_NST;
    const uint32_t par = (uint32_t)((u / P_NST) & 1);
    const int kb = pair_kb(s8);                     // the weight image's order (build_pair_image), every gate
    if (half_bar != nullptr && s8 == NKB / 2) { mbar_wait_cl(half_bar, half_par); tc_fence_after(); }
    mbar_wait(&bar_full[stage], par);
    if (leader) {
#pragma unroll
      for (int j = 0; j < KB / 16; ++j) {
        const uint32_t bo = (uint32_t)(stage * P_STAGE_BYTES + j * 2 * LBO) >> 4;
        const uint32_t ao = (uint32_t)((kb * (KB / 16) + j) * 2 * LBO) >> 4;
        const uint64_t dbh = desc_of(b_lo + bo, b_hi), dbl = desc_of(b_lo + bo + (P_HALF_BYTES >> 4), b_hi);
        const uint64_t dah = desc_of(aHi_lo + ao, a_hi), dal = desc_of(aLo_lo + ao, a_hi);
        mma2_bf16(d_tmem, dah, dbh, idesc, (s8 | j) ? 1u : 0u);
        mma2_bf16(d_tmem, dal, dbh, idesc, 1u);
        mma2_bf16(d_tmem, dah, dbl, idesc, 1u);
      }
      commit2(&bar_empty[stage]);
    }
    __syncwarp();
  }
}

// per-recurrence view of an epilogue thread
struct PpLane {
  const float* xt;      // tile base of the cached input halves of this recurrence
  const float* st;      // this row's attention scores, step stride TM
  int ln4;              // lane * 4 inside the quad layout
  uint8_t *aHi, *aLo;   // A operand of this recurrence (this CTA)
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NTHREADS, 1) k_augru_pp(const __grid_constant__ AugruPairParams pp) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bar_full[P_NST], bar_empty[P_NST], bar_h[2], bar_rh[2], bar_u[2], bar_c[2];
  __shared__ uint32_t tmem_base_s;
  const AugruTcParams& p = pp.b;
  uint8_t* smem = smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u);
  uint8_t* sB = smem + 2 * PP_SLOT_BYTES;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  const int m0 = (blockIdx.x >> 1) * TM;      // the pair's 128-row tile; recurrence s = sequence s of that tile

  if (tid == 0) {
    for (int i = 0; i < P_NST; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], 1); }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&bar_h[s], 16); mbar_init(&bar_rh[s], 16);
      mbar_init(&bar_u[s], 1); mbar_init(&bar_c[s], 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 8) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tbase = tmem_base_s;

  if (warp >= 8) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (warp == 9) {
      // ===== TMA producer: per step  [r,u](seq 0)  [r,u](seq 1)  [c](seq 0)  [c](seq 1)  of this CTA's column half =====
      if (lane == 0) {
        const uint32_t full0_leader = mapa_rank(smem_u32(&bar_full[0]), 0);
        const uint32_t sB_u = smem_u32(sB);
        int stage = 0; uint32_t phase = 0;
        for (int t = 0; t < STEPS; ++t) {
#pragma unroll 1
          for (int u = 0; u < PP_USES; ++u) {
            const int slot = u < 32 ? (u >> 4) : ((u - 32) >> 3);
            const int gs = u < 32 ? (u & 15) : 16 + ((u - 32) & 7);            // stage inside the sequence's 24-stage image
            mbar_wait(&bar_empty[stage], phase ^ 1);
            if (rank == 0) mbar_expect_tx(&bar_full[stage], 2 * P_STAGE_BYTES);
            tma_box_cg2(sB_u + stage * P_STAGE_BYTES, &pp.tmap[slot], 0, ((int)rank * P_STAGES_PER_STEP + gs) * P2_TM_BOX_ROWS,
                        full0_leader + stage * 8);
            if (++stage == P_NST) { stage = 0; phase ^= 1; }
          }
        }
      }
    } else if (warp == 8 && rank == 0) {
      // ===== MMA issuer (leader CTA): uniform control flow, one elected lane issues =====
      const uint32_t leader = elect_one();
      uint32_t a0h = desc_lo(smem_u32(smem), LBO), a0l = desc_lo(smem_u32(smem + P_A_BYTES), LBO),
               a1h = desc_lo(smem_u32(smem + PP_SLOT_BYTES), LBO), a1l = desc_lo(smem_u32(smem + PP_SLOT_BYTES + P_A_BYTES), LBO),
               b_d = desc_lo(smem_u32(sB), LBO);
      for (int t = 0; t < STEPS; ++t) {
        const uint32_t par = t & 1;
        long long* dbg = (p.dbg && blockIdx.x == 0 && leader) ? p.dbg + t * 16 : nullptr;
        asm volatile("" : "+r"(a0h), "+r"(a0l), "+r"(a1h), "+r"(a1l), "+r"(b_d));
        if (dbg) dbg[0] = clock64();
        mbar_wait_cl(&bar_h[0], par); tc_fence_after();
        if (dbg) dbg[1] = clock64();
        issue_gate_pp<0>(leader, tbase + 0, a0h, a0l, b_d, bar_full, bar_empty, nullptr, 0);
        issue_gate_pp<8>(leader, tbase + 128, a0h, a0l, b_d, bar_full, bar_empty, nullptr, 0);
        if (leader) commit2(&bar_u[0]);
        if (dbg) dbg[2] = clock64();
        mbar_wait_cl(&bar_h[1], par); tc_fence_after();
        if (dbg) dbg[3] = clock64();
        issue_gate_pp<16>(leader, tbase + 256, a1h, a1l, b_d, bar_full, bar_empty, nullptr, 0);
        issue_gate_pp<24>(leader, tbase + 384, a1h, a1l, b_d, bar_full, bar_empty, nullptr, 0);
        if (leader) commit2(&bar_u[1]);
        if (dbg) dbg[4] = clock64();
        mbar_wait_cl(&bar_rh[0], par); tc_fence_after();
        if (dbg) dbg[5] = clock64();
        issue_gate_pp<32>(leader, tbase + 0, a0h, a0l, b_d, bar_full, bar_empty, nullptr, 0);
        if (leader) commit2(&bar_c[0]);
        if (dbg) dbg[6] = clock64();
        mbar_wait_cl(&bar_rh[1], par); tc_fence_after();
        if (dbg) dbg[7] = clock64();
        issue_gate_pp<40>(leader, tbase + 256, a1h, a1l, b_d, bar_full, bar_empty, nullptr, 0);
        if (leader) commit2(&bar_c[1]);
        if (dbg) dbg[8] = clock64();
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    // ===== epilogue warps: thread = (row of this CTA, 64 hidden columns) of BOTH recurrences =====
    const int q = warp & 3, sub = warp >> 2;
    const int rl = (q & 1) * 32 + lane;
    const int prow = (int)rank * P_RC + rl;
    const int hc0 = (q >> 1) * 128 + sub * 64;
    const uint32_t tcol = (uint32_t)sub * 64;
    int r = m0 + prow;
    const bool valid = r < p.R;
    if (!valid) r = p.R - 1;
    const uint32_t tlane = tbase + ((uint32_t)(q * 32) << 16);
    const uint32_t a_row_off = (uint32_t)(rl / 8) * A_SBO + (uint32_t)(rl % 8) * 16;
    PpLane L[2];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      const AugruTcSeq& S = p.s[s];
      const int ci = S.shared ? 0 : (p.row0 + r) / p.div;
      L[s].xt = S.XT + ((size_t)(ci / TM) * STEPS) * XT_COLS * TM;
      L[s].ln4 = (ci % TM) * 4;
      L[s].st = S.scoresT + ((size_t)(m0 / TM) * STEPS) * TM + prow;
      L[s].aHi = smem + s * PP_SLOT_BYTES;
      L[s].aLo = L[s].aHi + P_A_BYTES;
    }
    uint32_t h_leader[2], rh_leader[2];
#pragma unroll
    for (int s = 0; s < 2; ++s) { h_leader[s] = mapa_rank(smem_u32(&bar_h[s]), 0); rh_leader[s] = mapa_rank(smem_u32(&bar_rh[s]), 0); }
    auto arrive = [&](uint64_t* local, uint32_t remote) {      // lane 0, after proxy_fence + __syncwarp
      if (rank == 0) mbar_arrive(local); else arrive_remote(remote);
    };
    float h[2][64], x[PP_XD + 1][PP_CH];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
#pragma unroll
      for (int i = 0; i < 64; ++i) h[s][i] = 0.f;
#pragma unroll
      for (int g = 0; g < 8; ++g) {                          // h0 = 0 into the A operands
        const uint32_t off = a_row_off + (uint32_t)((hc0 + g * 8) / 8) * LBO;
        *reinterpret_cast<uint4*>(L[s].aHi + off) = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4*>(L[s].aLo + off) = make_uint4(0, 0, 0, 0);
      }
    }
    proxy_fence();
    __syncwarp();
    if (lane == 0) {
#pragma unroll
      for (int s = 0; s < 2; ++s) arrive(&bar_h[s], h_leader[s]);
    }
    // the rolling input buffer always holds the first PP_XD chunks of the NEXT phase: prime it for R of recurrence 0
#pragma unroll
    for (int c = 0; c < PP_XD; ++c) load_x8(x[c], L[0].xt, hc0 + c * PP_CH, L[0].ln4);

    for (int t = 0; t < STEPS; ++t) {
      const uint32_t par = t & 1;
      const bool more = t + 1 < STEPS;
      float oms[2];
#pragma unroll
      for (int s = 0; s < 2; ++s) oms[s] = 1.0f - __ldg(L[s].st + (size_t)t * TM);
      if (more) {          // next step's input lines of this CTA's 64 rows: HBM -> L2 (a shared sequence is one cached row)
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          if (p.s[s].shared) continue;
          const float* xn = L[s].xt + (size_t)(t + 1) * XT_COLS * TM;
#pragma unroll
          for (int i = 0; i < 6; ++i) {
            const int id = i * 256 + tid;
            asm volatile("prefetch.global.L2 [%0];" :: "l"(xn + (size_t)(id >> 3) * 4 * TM + rank * (P_RC * 4) + (id & 7) * 32));
          }
        }
      }
      // ---- phases R and U of each recurrence ----
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        const float* xs = L[s].xt + (size_t)t * XT_COLS * TM;
        const uint32_t tr = tlane + (uint32_t)(s * 256) + tcol, tu = tr + 128;
        mbar_wait(&bar_u[s], par);                          // r AND u retired: h may be overwritten by r*h
        tc_fence_after();
        {
          float a[2][PP_CH];
          tmem_ld8(tr, a[0]);
#pragma unroll
          for (int ch = 0; ch < PP_NCH; ++ch) {
            const int cur = ch & 1;
            tmem_wait_ld();
            if (ch + 1 < PP_NCH) tmem_ld8(tr + (ch + 1) * PP_CH, a[cur ^ 1]);
            if (ch + PP_XD < PP_NCH) load_x8(x[(ch + PP_XD) % (PP_XD + 1)], xs, hc0 + (ch + PP_XD) * PP_CH, L[s].ln4);
#pragma unroll
            for (int j = 0; j < PP_CH; ++j)
              a[cur][j] = rcp_approx(1.0f + ex2_approx(fminf(P2_NL2E * (a[cur][j] + x[ch % (PP_XD + 1)][j]), 60.0f))) * h[s][ch * PP_CH + j];
            split_store8(a[cur], L[s].aHi, L[s].aLo, a_row_off + (uint32_t)((hc0 + ch * PP_CH) / 8) * LBO);
          }
        }
#pragma unroll
        for (int c = 0; c < PP_XD; ++c) load_x8(x[(PP_NCH + c) % (PP_XD + 1)], xs, HID + hc0 + c * PP_CH, L[s].ln4);   // prime U
        tc_fence_before();
        proxy_fence();
        __syncwarp();
        if (lane == 0) arrive(&bar_rh[s], rh_leader[s]);
        {
          float a[2][PP_CH];
          tmem_ld8(tu, a[0]);
#pragma unroll
          for (int ch = 0; ch < PP_NCH; ++ch) {
            const int cur = ch & 1, xi = (PP_NCH + ch) % (PP_XD + 1);
            tmem_wait_ld();
            if (ch + 1 < PP_NCH) tmem_ld8(tu + (ch + 1) * PP_CH, a[cur ^ 1]);
            if (ch + PP_XD < PP_NCH) load_x8(x[(PP_NCH + ch + PP_XD) % (PP_XD + 1)], xs, HID + hc0 + (ch + PP_XD) * PP_CH, L[s].ln4);
#pragma unroll
            for (int j = 0; j < PP_CH; ++j)
              a[cur][j] = 1.0f + ex2_approx(fminf(P2_NL2E * (a[cur][j] + x[xi][j]), 60.0f));
            tmem_st8(tu + ch * PP_CH, a[cur]);
          }
          tmem_wait_st();
        }
        // prime the next phase: R of recurrence 1 (same step), or C of recurrence 0
        {
          const float* nb = s == 0 ? L[1].xt + (size_t)t * XT_COLS * TM : L[0].xt + (size_t)t * XT_COLS * TM;
          const int ncol = s == 0 ? hc0 : 2 * HID + hc0;
          const int nl = s == 0 ? L[1].ln4 : L[0].ln4;
#pragma unroll
          for (int c = 0; c < PP_XD; ++c) load_x8(x[(2 * PP_NCH + c) % (PP_XD + 1)], nb, ncol + c * PP_CH, nl);
        }
      }
      // ---- phase C of each recurrence ----
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        const float* xs = L[s].xt + (size_t)t * XT_COLS * TM;
        const uint32_t tc = tlane + (uint32_t)(s * 256) + tcol, tu = tc + 128;
        mbar_wait(&bar_c[s], par);
        tc_fence_after();
        {
          float a[2][PP_CH], u[2][PP_CH];
          tmem_ld8(tc, a[0]);
          tmem_ld8(tu, u[0]);
#pragma unroll
          for (int ch = 0; ch < PP_NCH; ++ch) {
            const int cur = ch & 1, xi = (2 * PP_NCH + ch) % (PP_XD + 1);
            tmem_wait_ld();
            if (ch + 1 < PP_NCH) { tmem_ld8(tc + (ch + 1) * PP_CH, a[cur ^ 1]); tmem_ld8(tu + (ch + 1) * PP_CH, u[cur ^ 1]); }
            if (ch + PP_XD < PP_NCH)
              load_x8(x[(2 * PP_NCH + ch + PP_XD) % (PP_XD + 1)], xs, 2 * HID + hc0 + (ch + PP_XD) * PP_CH, L[s].ln4);
#pragma unroll
            for (int j = 0; j < PP_CH; ++j) {
              const float F = 1.0f + ex2_approx(fminf(P2_2L2E * (a[cur][j] + x[xi][j]), 60.0f));
              const float E = u[cur][j];
              const float rc = rcp_approx(E * F);
              const float c = fmaf(-2.0f, rc * E, 1.0f);
              const float up = oms[s] * (rc * F);
              const float hn = fmaf(up, h[s][ch * PP_CH + j] - c, c);
              h[s][ch * PP_CH + j] = hn;
              a[cur][j] = hn;
            }
            split_store8(a[cur], L[s].aHi, L[s].aLo, a_row_off + (uint32_t)((hc0 + ch * PP_CH) / 8) * LBO);
          }
        }
        // prime the next phase: C of recurrence 1, or R of recurrence 0 of the NEXT step
        {
          const float* nb = s == 0 ? L[1].xt + (size_t)t * XT_COLS * TM : L[0].xt + (size_t)(more ? t + 1 : t) * XT_COLS * TM;
          const int ncol = s == 0 ? 2 * HID + hc0 : hc0;
          const int nl = s == 0 ? L[1].ln4 : L[0].ln4;
#pragma unroll
          for (int c = 0; c < PP_XD; ++c) load_x8(x[(3 * PP_NCH + c) % (PP_XD + 1)], nb, ncol + c * PP_CH, nl);
        }
        tc_fence_before();
        proxy_fence();
        __syncwarp();
        if (lane == 0) arrive(&bar_h[s], h_leader[s]);
      }
    }
    if (valid) {
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        float* o = p.s[s].out + (size_t)(m0 + prow) * p.out_ld + hc0;
#pragma unroll
        for (int i = 0; i < 64; i += 4) *reinterpret_cast<float4*>(o + i) = make_float4(h[s][i], h[s][i + 1], h[s][i + 2], h[s][i + 3]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 8) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" :: "r"(tbase), "r"(512));
}

// host: the pair weight image of one sequence (2 ranks x 24 stages x 16 KB, device pointer) as a tensor map of
// [768 rows][256 x u32]; box = 256 x 16 = one ring stage.  cuTensorMapEncodeTiled is fetched through the runtime
// (cudaGetDriverEntryPoint), so the library does not link libcuda.  Returns 0 on success.
inline int make_pair_tensor_map(const void* dev_img, CUtensorMap* out) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &qr) != cudaSuccess || qr != cudaDriverEntryPointSuccess)
      f = nullptr;
    return reinterpret_cast<EncodeFn>(f);
  }();
  if (!fn) return 1;
  const cuuint64_t gdim[2] = {256, (cuuint64_t)(2 * P_RANK_IMAGE_BYTES / P2_TM_ROW_BYTES)};
  const cuuint64_t gstride[1] = {P2_TM_ROW_BYTES};
  const cuuint32_t box[2] = {256, (cuuint32_t)P2_TM_BOX_ROWS};
  const cuuint32_t estr[2] = {1, 1};
  CUresult rc = fn(out, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<void*>(dev_img), gdim, gstride, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return rc == CUDA_SUCCESS ? 0 : 2;
}

}  // namespace r4tc
