// r4_augru_pair2.cuh -- the AUGRU recurrence (deepctr VecAttGRUCell, nets/utils.py:123-124) as ONE tensor-core instruction
// stream per 2-CTA cluster: tcgen05.mma.cta_group::2, M = 128 (64 feature rows per CTA), N = 256, bf16 hi/lo operands, fp32
// accumulators in both CTAs' TMEM.  The arithmetic (r4_tc_common.cuh):
//     r = sigmoid(Xr_t + h Wr)      u = sigmoid(Xu_t + h Wu)      c = tanh(Xc_t + (r*h) Wc)
//     u' = (1 - score_t) u ;  h <- u' h + (1 - u') c              (3 bf16 products per fp32 product)
// What the pair buys (measured with tools/pair_probe.cu): a 128x256x16 MMA takes 64 cycles instead of 128, each CTA streams
// only its half of the weight columns, each CTA's epilogue owns 64 rows instead of 128 (so a 4096-row batch x 2 sequences
// fills 128 SMs instead of 64), and the accumulators of one gate take 128 TMEM columns per CTA -- r, u and c do not alias,
// and r*h gets its own A buffer, so the gate epilogues overlap the next gate's MMAs.
// TMEM layout of a pair MMA (cute tmem_frg_2sm "2x2" atom, confirmed by the probe): in each CTA, lanes 0-63 hold
// accumulator columns 0-127 of the CTA's 64 rows and lanes 64-127 hold columns 128-255.
//
// Per CTA: shared memory = A(h) hi/lo 64 KB + A(r*h) hi/lo 64 KB + a 3-stage ring of 16 KB weight stages (one 32-deep K
// block of the CTA's 128 weight columns, hi then lo split, pre-tiled on the host so a stage is one bulk copy).  Both CTAs'
// stages must have landed before the leader issues: the peer's control warp relays its local "full" barrier to the leader
// with a remote mbarrier arrive (~460 cycles one way, hidden by the ring).
// Warp roles: 0-7 epilogue (TMEM lane quarter q = warp & 3, column half = warp >> 2; thread = one row x 64 hidden
// columns), 8 = MMA issuer (leader) / ring relay (peer), 9 = TMA producer, 10-11 idle.
//
// Around the tensor pipe, each item answering a measurement of round 1:
//   * issue loop: the whole MMA warp walks the step in uniform control flow, ONE lane elected once (elect.sync) issues,
//     ring stage / mbarrier parity / operand offsets are compile-time constants (a step = 24 ring uses = 8 revolutions
//     of the 3 stages, so they repeat every step).  Round 1: ~100 SASS instructions of descriptor arithmetic + an
//     ELECT/BRA.U.ANY wrapper per MMA paced the pair MMAs at ~105 cycles; this form issues at 52-65.
//   * rolling input prefetch: the epilogue keeps the inputs of the NEXT gate phase in registers (x[4][16]); a chunk is
//     reloaded with the next phase's columns the moment it has been consumed, so every L2 load has a whole phase
//     (~2 k cycles) to land.  Round 1: a 1-deep pipeline over 16-column chunks left each phase (R 5.3 k, U 4.8 k,
//     C 5.5 k cycles) bound by L2 latency, and the phases run back to back on the same 8 warps.
//   * hand-over: every epilogue warp of BOTH CTAs publishes a finished operand quarter with st.shared ->
//     fence.proxy.async -> __syncwarp -> one mbarrier.arrive.release.cta on the LEADER's barrier (a shared::cluster address
//     for the peer: the instruction CUTLASS's ClusterBarrier::arrive(cta_id) issues for the peer-epilogue -> leader-MMA
//     signals of its 2-SM kernels).  The data a peer warp publishes stays in the PEER's shared memory and is read by the
//     peer SM's half of the cta_group::2 MMA; what crosses the cluster is only the arrival.
// Measured alternatives (tools/augru_probe.cu, round 2, cycles per step; DESIGN.md section 4): a relayed release.cluster
// hand-over 19.3 k and a tensor-map weight ring 17.2 k, against 15.5 k for this kernel.
#pragma once
#include <cuda.h>
#include "r4_tc_common.cuh"

namespace r4tc {

constexpr int P_RC = 64;                              // rows per CTA
constexpr int P_NB = 128;                             // weight columns (B rows) per CTA
constexpr int P_HALF_BYTES = P_NB * KB * 2;           // 8192: one split of one 32-deep K block of the CTA's 128 columns
constexpr int P_STAGE_BYTES = 2 * P_HALF_BYTES;       // 16384: ring stage = [hi | lo] of one K block (6 MMAs, 384 cycles)
constexpr int P_STAGES_PER_STEP = 3 * NKB;            // 24
// Ring depth.  Measured (tools/augru_probe.cu, round 2, cycles per step of k_augru_pair2 / k_augru_pp): 6 stages 17.1 k /
// 31.3 k, 4 stages 16.0 k / 31.4 k, 3 stages 15.7 k / 29.6 k, 2 stages 20.5 k.  A deep ring refills in bursts that compete
// with the gate epilogues for the shared-memory port (the MMA warp's own clocks: with 6 stages it waits 7-8 k cycles per
// step for operand quarters, i.e. for the epilogue, with 3 stages 2.7 k); 3 stages = 48 KB keeps the weight stream just
// ahead of the MMAs.  24 % (2 * P_NST) == 0 keeps stage and parity compile-time.
constexpr int P_NST = 3;
constexpr int P_A_BYTES = P_RC * HID * 2;             // 32768 per split
constexpr int P_SMEM_BYTES = 4 * P_A_BYTES + P_NST * P_STAGE_BYTES + 128;
constexpr int P_RANK_IMAGE_BYTES = P_STAGES_PER_STEP * P_STAGE_BYTES; // 393216 per CTA rank
constexpr int P_TC_R = 0, P_TC_U = 128, P_TC_C = 256;                  // TMEM column bases of the gates

__device__ __forceinline__ void mma2_bf16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
               :: "r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(acc) : "memory");
}
// completion of all earlier MMAs of this thread -> one arrival on the barrier at this offset in BOTH CTAs
__device__ __forceinline__ void commit2(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               :: "r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
// acquire.cluster try_wait is expensive (a producer loop built on it issued one stage per ~450 cycles); it is used
// only for the barriers the leader's MMA thread waits on, which collect remote arrivals.
__device__ __forceinline__ void mbar_wait_cl(uint64_t* bar, uint32_t parity) {
  asm volatile("{\n\t.reg .pred p;\n\tWAIT_LOOP:\n\t"
               "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n\t"
               "@p bra DONE;\n\tbra WAIT_LOOP;\n\tDONE:\n\t}\n" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ uint32_t mapa_rank(uint32_t laddr, uint32_t rank) {
  uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(laddr), "r"(rank)); return r;
}
// Arrival on a barrier of the other CTA of the pair: mbarrier.arrive.release.cta (the default semantics of
// mbarrier.arrive: CUTLASS's ClusterBarrier::arrive(cta_id)).  It is enough where the data being published lives in the
// ARRIVING CTA's own shared memory and has already been made visible to the async proxy (TMA completion, or
// fence.proxy.async by every writer + __syncwarp): the consumer is this SM's tensor core, started by the leader only after
// it has observed the arrival.  Measured (cycles per step): .relaxed.cluster 15.5 k, .release.cta 15.5 k, .release.cluster
// 30.1 k (it blocks its thread ~320 cycles, tools/pair_probe.cu).
__device__ __forceinline__ void arrive_remote(uint32_t caddr) {
  asm volatile("mbarrier.arrive.release.cta.shared::cluster.b64 _, [%0];" :: "r"(caddr) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// Ring stage s8 (0..7) of every gate holds K block 0,4,1,5,2,6,3,7: the epilogue of k_augru_pair2 completes the blocks
// {q, 4 + q} of an A operand with its q-th column chunk, and the MMAs follow it in that order.
__host__ __device__ constexpr int pair_kb(int s8) { return (s8 & 1) * 4 + (s8 >> 1); }

// host: fp32 recurrent weights -> [rank 2][mat r,u,c][8 K blocks][hi, lo] stages of 128 columns x 32 K (8 KB).
// Wg: [256][512] rows = h index, columns [r | u];  Wc: [256][256].
inline void build_pair_image(const float* Wg, const float* Wc, uint8_t* img) {
  for (int rank = 0; rank < 2; ++rank)
    for (int mat = 0; mat < 3; ++mat)
      for (int kb = 0; kb < NKB; ++kb)
        for (int sp = 0; sp < 2; ++sp) {
          const int kbsrc = pair_kb(kb);               // the order in which the kernels walk the K blocks of a gate
          uint8_t* st = img + (size_t)rank * P_RANK_IMAGE_BYTES + (size_t)((mat * NKB + kb) * 2 + sp) * P_HALF_BYTES;
          for (int nl = 0; nl < P_NB; ++nl)
            for (int kk = 0; kk < KB; ++kk) {
              const int k = kbsrc * KB + kk, n = rank * P_NB + nl;
              float w = mat == 0 ? Wg[(size_t)k * 2 * HID + n] : (mat == 1 ? Wg[(size_t)k * 2 * HID + HID + n] : Wc[(size_t)k * HID + n]);
              uint16_t hi = host_bf16_bits(w);
              uint16_t v = sp == 0 ? hi : host_bf16_bits(w - host_bf16_val(hi));
              memcpy(st + (nl / 8) * B_SBO + (kk / 8) * LBO + (nl % 8) * 16 + (kk % 8) * 2, &v, 2);
            }
        }
}

struct AugruPairParams {
  AugruTcParams b;
  CUtensorMap tmap[2];        // per sequence: the pair weight image as [rows of 1 KB][256 x u32] (k_augru_pp's weight ring)
};

// Descriptor of a SWIZZLE_NONE K-major operand split into its two words: `lo` carries the start address (>> 4, 14 bits)
// and LBO, `hi` carries SBO and the version bit.  Advancing the operand by `bytes` is `lo + (bytes >> 4)` (shared
// memory is < 256 KB, the address field cannot carry out), so a descriptor costs ONE add in the issue loop.
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr, uint32_t lbo) { return ((saddr >> 4) & 0x3fffu) | ((lbo >> 4) << 16); }
__device__ __forceinline__ constexpr uint32_t desc_hi(uint32_t sbo) { return ((sbo >> 4) & 0x3fffu) | (1u << 14); }
__device__ __forceinline__ uint64_t desc_of(uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; }

// tcgen05.commit -> one arrival on the barrier at this offset in every CTA of `mask`
__device__ __forceinline__ void commit2_mask(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               :: "r"(smem_u32(bar)), "h"(mask) : "memory");
}

// One gate of one step: 8 ring stages x 2 K16 slices x (A_hi*B_hi + A_lo*B_hi + A_hi*B_lo).  Every gate walks the K
// blocks of its A operand in the order pair_kb() = 0,4,1,5,2,6,3,7: the epilogue finishes blocks {q, 4 + q} with its
// q-th column chunk and publishes them on quarter barrier q, so the gate's MMAs chase the epilogue that produces their
// operand, 12 MMAs behind it (`qbar` = the 4 quarter barriers of the A operand, nullptr when it is already complete).
// build_pair_image lays the weights out in the same order.  No tcgen05 fence per stage: the weights come from TMA.
template <int GATE>
__device__ __forceinline__ void issue_gate2(uint32_t leader, uint32_t tbase, uint32_t aHi_lo, uint32_t aLo_lo, uint32_t b_lo,
                                            uint64_t* bar_full, uint64_t* bar_empty, uint64_t* qbar, uint32_t qpar,
                                            long long* wait_acc = nullptr) {
  constexpr uint32_t idesc = make_idesc(TM, HID);
  constexpr uint32_t dcol = GATE == 0 ? P_TC_R : (GATE == 1 ? P_TC_U : P_TC_C);
  constexpr uint32_t a_hi = desc_hi(A_SBO), b_hi = desc_hi(B_SBO);
#pragma unroll
  for (int s8 = 0; s8 < NKB; ++s8) {
    const int u = GATE * NKB + s8;
    const int stage = u % P_NST;
    const uint32_t par = (uint32_t)((u / P_NST) & 1);
    const int kb = pair_kb(s8);
    // wait_acc (probe builds only): [0] cycles waiting for operand quarters, [1] cycles waiting for ring stages
    long long w0 = wait_acc ? clock64() : 0;
    if (qbar != nullptr && (s8 & 1) == 0) { mbar_wait_cl(&qbar[s8 >> 1], qpar); tc_fence_after(); }
    long long w1 = wait_acc ? clock64() : 0;
    mbar_wait(&bar_full[stage], par);
    if (wait_acc) { wait_acc[0] += w1 - w0; wait_acc[1] += clock64() - w1; }
    if (leader) {
#pragma unroll
      for (int j = 0; j < KB / 16; ++j) {
        const uint32_t bo = (uint32_t)(stage * P_STAGE_BYTES + j * 2 * LBO) >> 4;
        const uint32_t ao = (uint32_t)((kb * (KB / 16) + j) * 2 * LBO) >> 4;
        const uint64_t dbh = desc_of(b_lo + bo, b_hi), dbl = desc_of(b_lo + bo + (P_HALF_BYTES >> 4), b_hi);
        const uint64_t dah = desc_of(aHi_lo + ao, a_hi), dal = desc_of(aLo_lo + ao, a_hi);
        mma2_bf16(tbase + dcol, dah, dbh, idesc, (s8 | j) ? 1u : 0u);
        mma2_bf16(tbase + dcol, dal, dbh, idesc, 1u);
        mma2_bf16(tbase + dcol, dah, dbl, idesc, 1u);
      }
      commit2(&bar_empty[stage]);
    }
    __syncwarp();
  }
}

constexpr float P2_NL2E = -1.4426950408889634f, P2_2L2E = 2.8853900817779268f;   // gate pre-activations in the exp2 domain
// 8 fp32 -> bf16 hi / lo core-matrix rows of an A operand
__device__ __forceinline__ void split_store8(const float* v, uint8_t* hi_base, uint8_t* lo_base, uint32_t off) {
  uint4 hi, lo;
  split8(v, hi, lo);
  *reinterpret_cast<uint4*>(hi_base + off) = hi;
  *reinterpret_cast<uint4*>(lo_base + off) = lo;
}

// Launched in clusters of 2 CTAs (cudaLaunchAttributeClusterDimension): one CTA pair per 128-row tile and sequence.
__global__ void __launch_bounds__(NTHREADS, 1) k_augru_pair2(const __grid_constant__ AugruPairParams pp) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bar_full[P_NST], bar_empty[P_NST], bar_h[4], bar_rh[4], bar_r, bar_u, bar_c;
  __shared__ uint32_t tmem_base_s;
  const AugruTcParams& p = pp.b;
  uint8_t* smem = smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u);
  uint8_t* sHhi = smem;                       // A operand: h
  uint8_t* sHlo = smem + P_A_BYTES;
  uint8_t* sRhi = smem + 2 * P_A_BYTES;       // A operand: r*h
  uint8_t* sRlo = smem + 3 * P_A_BYTES;
  uint8_t* sB = smem + 4 * P_A_BYTES;
  const AugruTcSeq& S = p.s[blockIdx.y];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // The leader's cluster rank and the tile are derived for a general cluster shape although a cluster is one pair here
  // (lead = 0, every pair has a tile): written as constants, they reorder the machine code of the whole kernel.
  const uint32_t crank = cluster_ctarank();
  const uint32_t rank = crank & 1;             // rank inside the CTA pair: 0 = leader (issues the MMAs)
  const uint32_t lead = crank & ~1u;           // cluster rank of this pair's leader
  const int n_tiles = (p.R + TM - 1) / TM;
  const int tile = min((int)(blockIdx.x >> 1), n_tiles - 1);
  const bool pad_pair = (int)(blockIdx.x >> 1) >= n_tiles;   // a pair past the last tile would redo it, unseen
  const int m0 = tile * TM;                    // the pair's 128-row tile
  const uint16_t pair_mask = (uint16_t)(3u << lead);

  if (tid == 0) {
    // "full": the leader's collects its own TMA (expect_tx arrival) and the peer's relay arrival
    for (int i = 0; i < P_NST; ++i) { mbar_init(&bar_full[i], rank == 0 ? 2 : 1); mbar_init(&bar_empty[i], 1); }
    // hand-over barriers: 8 warps x 2 CTAs on the leader
    for (int i = 0; i < 4; ++i) { mbar_init(&bar_h[i], 16); mbar_init(&bar_rh[i], 16); }
    mbar_init(&bar_r, 1); mbar_init(&bar_u, 1); mbar_init(&bar_c, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 8) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                         // the peer's barriers exist before anyone arrives remotely
  tc_fence_after();
  const uint32_t tbase = tmem_base_s;
  const uint32_t bar_h_leader = mapa_rank(smem_u32(&bar_h[0]), lead), bar_rh_leader = mapa_rank(smem_u32(&bar_rh[0]), lead);

  if (warp >= 8) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");   // frees 128 x 128 registers = what 232 for the 256 epilogue threads takes
    if (warp == 9) {
      // ===== TMA producer: this CTA's half of the 24-stage weight stream of a step, 64 times =====
      if (lane == 0) {
        int stage = 0; uint32_t phase = 0;
        const uint8_t* img = S.Wimg + (size_t)rank * P_RANK_IMAGE_BYTES;
        for (int t = 0; t < STEPS; ++t) {
          const uint8_t* src = img;
          for (int i = 0; i < P_STAGES_PER_STEP; ++i, src += P_STAGE_BYTES) {
            mbar_wait(&bar_empty[stage], phase ^ 1);
            mbar_expect_tx(&bar_full[stage], P_STAGE_BYTES);
            bulk_g2s(sB + stage * P_STAGE_BYTES, src, P_STAGE_BYTES, &bar_full[stage]);
            if (++stage == P_NST) { stage = 0; phase ^= 1; }
          }
        }
      }
    } else if (warp == 8 && rank == 1) {
      // ===== ring relay: tell the leader that this CTA's copy of stage s has landed =====
      if (lane == 0) {
        const uint32_t remote0 = mapa_rank(smem_u32(&bar_full[0]), lead);
        int stage = 0; uint32_t phase = 0;
        for (int i = 0; i < STEPS * P_STAGES_PER_STEP; ++i) {
          mbar_wait(&bar_full[stage], phase);
          arrive_remote(remote0 + stage * 8);
          if (++stage == P_NST) { stage = 0; phase ^= 1; }
        }
      }
    } else if (warp == 8) {
      // ===== MMA issuer (leader CTA): uniform control flow, one elected lane issues =====
      const uint32_t leader = elect_one();
      uint32_t hHi_d = desc_lo(smem_u32(sHhi), LBO), hLo_d = desc_lo(smem_u32(sHlo), LBO), rHi_d = desc_lo(smem_u32(sRhi), LBO),
               rLo_d = desc_lo(smem_u32(sRlo), LBO), b_d = desc_lo(smem_u32(sB), LBO);
      for (int t = 0; t < STEPS; ++t) {
        const uint32_t par = t & 1;
        long long* dbg = (p.dbg && blockIdx.x == 0 && blockIdx.y == 0 && leader) ? p.dbg + t * 16 : nullptr;
        if (dbg) dbg[0] = clock64();
        // keep the 144 descriptors of a step OUT of the loop-invariant set: hoisted, they live in local memory (this warp
        // has 40 registers) and every MMA pays a local load; rebuilt from these five words each costs one add
        asm volatile("" : "+r"(hHi_d), "+r"(hLo_d), "+r"(rHi_d), "+r"(rLo_d), "+r"(b_d));
        long long wacc[2] = {0, 0};
        long long* wa = dbg ? wacc : nullptr;
        if (dbg) dbg[1] = clock64();
        issue_gate2<0>(leader, tbase, hHi_d, hLo_d, b_d, bar_full, bar_empty, bar_h, par, wa);   // chases phase C of step t-1
        if (leader) commit2_mask(&bar_r, pair_mask);
        if (dbg) dbg[2] = clock64();
        issue_gate2<1>(leader, tbase, hHi_d, hLo_d, b_d, bar_full, bar_empty, nullptr, 0, wa);
        if (leader) commit2_mask(&bar_u, pair_mask);
        if (dbg) dbg[3] = clock64();
        if (dbg) dbg[4] = clock64();
        issue_gate2<2>(leader, tbase, rHi_d, rLo_d, b_d, bar_full, bar_empty, bar_rh, par, wa);  // chases phase R of this step
        if (leader) commit2_mask(&bar_c, pair_mask);
        if (dbg) { dbg[5] = clock64(); dbg[6] = wacc[0]; dbg[7] = wacc[1]; }
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    // ===== epilogue warps: thread = (row of this CTA, 4 chunks of 16 hidden columns) =====
    // Chunk ch of a thread covers hidden columns half * 128 + ch * 32 + sub * 16 .. + 15: the two warps (sub = 0, 1) of a
    // lane quarter together finish the 32-wide K block half * 4 + ch with their ch-th chunk, so over the CTA pair chunk ch
    // completes K blocks {ch, 4 + ch} of the A operand -- quarter barrier ch, the unit the MMA warp chases.
    const int q = warp & 3, sub = warp >> 2;
    const int rl = (q & 1) * 32 + lane;                    // row inside this CTA
    const int prow = (int)rank * P_RC + rl;                // row inside the pair's 128-row tile
    const int hcb = (q >> 1) * 128 + sub * 16;             // hidden column of chunk ch: hcb + ch * 32
    const uint32_t tcb = (uint32_t)sub * 16;               // TMEM column inside a gate of chunk ch: tcb + ch * 32
    int r = m0 + prow;
    const bool valid = r < p.R && !pad_pair;
    if (r >= p.R) r = p.R - 1;
    const int ci = S.shared ? 0 : (p.row0 + r) / p.div;
    const float* xt = S.XT + ((size_t)(ci / TM) * STEPS) * XT_COLS * TM;
    const int ln4 = (ci % TM) * 4;
    const float* st = S.scoresT + ((size_t)(m0 / TM) * STEPS) * TM + prow;
    const uint32_t tlane = tbase + ((uint32_t)(q * 32) << 16);
    const uint32_t a_row_off = (uint32_t)(rl / 8) * A_SBO + (uint32_t)(rl % 8) * 16 + (uint32_t)(hcb / 8) * LBO;
    // publish quarter `i` of an A operand: this thread's stores -> async proxy, then one arrival per warp on the leader's
    // barrier
    auto publish = [&](uint64_t* bars, uint32_t bars_leader, int i) {
      tc_fence_before();
      proxy_fence();
      __syncwarp();
      if (lane == 0) { if (rank == 0) mbar_arrive(&bars[i]); else arrive_remote(bars_leader + i * 8); }
    };
    float h[64], x[4][16];
#pragma unroll
    for (int i = 0; i < 64; ++i) h[i] = 0.f;
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) {                       // h0 = 0 into the A operand
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        const uint32_t off = a_row_off + (uint32_t)(ch * 4 + g) * LBO;
        *reinterpret_cast<uint4*>(sHhi + off) = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4*>(sHlo + off) = make_uint4(0, 0, 0, 0);
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) publish(bar_h, bar_h_leader, i);
    // rolling input buffer: x[ch] always holds chunk ch of the NEXT phase to run (here: the r gate of step 0)
#pragma unroll
    for (int c4 = 0; c4 < 4; ++c4) load_x16(x[c4], xt, hcb + c4 * 32, ln4);
    float one_minus_s = 1.0f - __ldg(st);

    for (int t = 0; t < STEPS; ++t) {
      const uint32_t par = t & 1;
      long long* dbg = (p.dbg && blockIdx.x == 0 && blockIdx.y == 0 && tid == 0) ? p.dbg + t * 16 : nullptr;
      const float* xs = xt + (size_t)t * XT_COLS * TM;
      const bool more = t + 1 < STEPS;
      const float* xs_next = xs + (more ? (size_t)XT_COLS * TM : 0);
      const float oms_next = 1.0f - __ldg(st + (size_t)(more ? t + 1 : t) * TM);
      // Pull this CTA's half of the NEXT step's input lines (768 columns x 2 lines) from HBM into L2.
      if (more) {
        const float* xn = S.XT + (((size_t)(ci / TM) * STEPS + (t + 1)) * XT_COLS) * TM;
#pragma unroll
        for (int i = 0; i < 6; ++i) {
          const int id = i * 256 + tid;                    // 1536 lines: (column quad, 8 lines of this CTA's 64 lanes x 16 B)
          asm volatile("prefetch.global.L2 [%0];" :: "l"(xn + (size_t)(id >> 3) * 4 * TM + rank * (P_RC * 4) + (id & 7) * 32));
        }
      }
      // ---- phase R (overlaps the u MMAs; the c MMAs chase it quarter by quarter): r*h -> its own A operand;
      //      x[] <- the u gate's inputs ----
      {
        float a[2][16];
        if (dbg) dbg[8] = clock64();
        mbar_wait(&bar_r, par);
        if (dbg) dbg[9] = clock64();
        tc_fence_after();
        tmem_ld16(tlane + P_TC_R + tcb, a[0]);
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          const int cur = ch & 1, nxt = cur ^ 1;
          tmem_wait_ld();
          if (ch < 3) tmem_ld16(tlane + P_TC_R + tcb + (ch + 1) * 32, a[nxt]);
#pragma unroll
          for (int j = 0; j < 16; ++j)
            a[cur][j] = rcp_approx(1.0f + ex2_approx(fminf(P2_NL2E * (a[cur][j] + x[ch][j]), 60.0f))) * h[ch * 16 + j];
          load_x16(x[ch], xs, HID + hcb + ch * 32, ln4);
#pragma unroll
          for (int g = 0; g < 2; ++g)
            split_store8(a[cur] + g * 8, sRhi, sRlo, a_row_off + (uint32_t)(ch * 4 + g) * LBO);
          publish(bar_rh, bar_rh_leader, ch);
        }
      }
      if (dbg) dbg[10] = clock64();
      // ---- phase U (overlaps the c MMAs): E = 1 + exp(-(acc_u + Xu)) back into TMEM; x[] <- the c gate's inputs ----
      {
        float a[2][16];
        mbar_wait(&bar_u, par);
        if (dbg) dbg[11] = clock64();
        tc_fence_after();
        tmem_ld16(tlane + P_TC_U + tcb, a[0]);
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          const int cur = ch & 1, nxt = cur ^ 1;
          tmem_wait_ld();
          if (ch < 3) tmem_ld16(tlane + P_TC_U + tcb + (ch + 1) * 32, a[nxt]);
#pragma unroll
          for (int j = 0; j < 16; ++j)
            a[cur][j] = 1.0f + ex2_approx(fminf(P2_NL2E * (a[cur][j] + x[ch][j]), 60.0f));
          load_x16(x[ch], xs, 2 * HID + hcb + ch * 32, ln4);
          tmem_st16(tlane + P_TC_U + tcb + ch * 32, a[cur]);
        }
        tmem_wait_st();
      }
      if (dbg) dbg[12] = clock64();
      // ---- phase C (the next step's r MMAs chase it quarter by quarter): c = tanh(acc_c + Xc) = 1 - 2/(1 + F), u = 1/E
      //      with ONE reciprocal of E*F; x[] <- next step's r inputs ----
      {
        float a[2][16], u[2][16];
        mbar_wait(&bar_c, par);
        if (dbg) dbg[13] = clock64();
        tc_fence_after();
        tmem_ld16(tlane + P_TC_C + tcb, a[0]);
        tmem_ld16(tlane + P_TC_U + tcb, u[0]);
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          const int cur = ch & 1, nxt = cur ^ 1;
          tmem_wait_ld();
          if (ch < 3) {
            tmem_ld16(tlane + P_TC_C + tcb + (ch + 1) * 32, a[nxt]);
            tmem_ld16(tlane + P_TC_U + tcb + (ch + 1) * 32, u[nxt]);
          }
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float F = 1.0f + ex2_approx(fminf(P2_2L2E * (a[cur][j] + x[ch][j]), 60.0f));
            const float E = u[cur][j];
            const float rc = rcp_approx(E * F);                      // E, F <= 1 + 2^60: the product is finite
            const float c = fmaf(-2.0f, rc * E, 1.0f);               // tanh
            const float up = one_minus_s * (rc * F);                 // (1 - s) sigmoid
            const float hn = fmaf(up, h[ch * 16 + j] - c, c);        // u' h + (1 - u') c
            h[ch * 16 + j] = hn;
            a[cur][j] = hn;
          }
          load_x16(x[ch], xs_next, hcb + ch * 32, ln4);      // (last step: a harmless re-read of this step's lines)
#pragma unroll
          for (int g = 0; g < 2; ++g)
            split_store8(a[cur] + g * 8, sHhi, sHlo, a_row_off + (uint32_t)(ch * 4 + g) * LBO);
          publish(bar_h, bar_h_leader, ch);
        }
      }
      if (dbg) dbg[14] = clock64();
      one_minus_s = oms_next;
    }
    if (valid) {
      float* o = S.out + (size_t)(m0 + prow) * p.out_ld + hcb;
#pragma unroll
      for (int ch = 0; ch < 4; ++ch)
#pragma unroll
        for (int i = 0; i < 16; i += 4)
          *reinterpret_cast<float4*>(o + ch * 32 + i) = make_float4(h[ch * 16 + i], h[ch * 16 + i + 1], h[ch * 16 + i + 2], h[ch * 16 + i + 3]);
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                         // neither CTA frees TMEM / exits while the pair's MMAs or arrivals are in flight
  if (warp == 8) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" :: "r"(tbase), "r"(512));
}

}  // namespace r4tc
