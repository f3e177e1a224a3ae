// r4_tc_common.cuh -- what every tcgen05 kernel of the library includes (AUGRU pair / ping-pong kernels, GRU-1, attention
// scores, GEMM): constants of the AUGRU problem, the PTX wrappers (mbarrier, bulk copy, tcgen05.mma / ld / st / commit,
// descriptors, elect.sync), the bf16 hi/lo split, the quad-layout input loads and the parameter structs of the AUGRU kernels.
//
// The AUGRU recurrence (deepctr VecAttGRUCell, nets/utils.py:123-124), per step, with h the 256-wide state:
//     u = sigmoid(Xu_t + h Wu)      r = sigmoid(Xr_t + h Wr)      c = tanh(Xc_t + (r*h) Wc)
//     u' = (1 - score_t) u ;  h <- u' h + (1 - u') c
// fp32 parity on a bf16 tensor pipe: every fp32 operand x is split x = hi + lo (both bf16, lo =
// bf16(x - hi)) and each product is issued as hi*hi + lo*hi + hi*lo (3 MMAs, fp32 accumulate):
// relative error ~2^-16 per term, measured 1e-5..3e-5 of rms on the 64-step recurrence against
// f64 (tools/split_sim.py) -- inside the 1e-4 parity bound.  The state h itself stays fp32 in the
// epilogue threads' registers; only the MMA operand copies are rounded.
//
// The kernels: r4_augru_pair2.cuh (one recurrence per CTA pair) and r4_augru_pp.cuh (two per pair).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <string.h>
#include <algorithm>

namespace r4tc {

constexpr int TM = 128;                 // rows per CTA tile (UMMA_M)
constexpr int HID = 256;                // AUGRU hidden = GEMM N and K
constexpr int STEPS = 64;
constexpr int KB = 32;                  // K elements per B stage
constexpr int NKB = HID / KB;           // 8 K blocks per matrix
constexpr int STAGE_BYTES = HID * KB * 2;            // 16384
constexpr int A_BYTES = TM * HID * 2;                // 65536 per split
constexpr int LBO = 128;                             // K-adjacent core matrices
constexpr int A_SBO = (HID / 8) * 128;               // 4096: 8-row groups of the A operand
constexpr int B_SBO = (KB / 8) * 128;                // 512:  8-row groups inside a B stage
constexpr int W_IMAGE_BYTES = 3 * NKB * 2 * STAGE_BYTES;   // 786432 per sequence: r, u, c x 8 K blocks x (hi, lo)
constexpr int XT_COLS = 3 * HID;                     // transposed input halves: [r | u | c] rows of 128 lanes
constexpr int NTHREADS = 384;               // 8 epilogue warps + one control warpgroup (MMA, TMA, 2 idle)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((saddr >> 4) & 0x3fff) | ((uint64_t)((lbo >> 4) & 0x3fff) << 16) |
         ((uint64_t)((sbo >> 4) & 0x3fff) << 32) | ((uint64_t)1 << 46);   // version 1, SWIZZLE_NONE
}
__device__ __forceinline__ constexpr uint32_t make_idesc(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void mma_bf16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
               :: "r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile("{\n\t.reg .pred p;\n\tWAIT_LOOP:\n\t"
               "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
               "@p bra DONE;\n\tbra WAIT_LOOP;\n\tDONE:\n\t}\n"
               :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void proxy_fence() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// 1 in exactly one lane of the (converged) warp: an MMA warp that walks its loop in uniform control flow and lets the
// elected lane issue avoids the ELECT / BRA.U.ANY convergence loop an `if (lane == 0)` body costs per tcgen05.mma
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .b32 r;\n\t.reg .pred p;\n\telect.sync r|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}\n" : "=r"(pred));
  return pred;
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t* u = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
               : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
                 "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
               : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float* v) {
  const uint32_t* u = reinterpret_cast<const uint32_t*>(v);
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
               :: "r"(taddr), "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]),
                  "r"(u[8]), "r"(u[9]), "r"(u[10]), "r"(u[11]), "r"(u[12]), "r"(u[13]), "r"(u[14]), "r"(u[15]) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// MUFU-based gate functions: ex2.approx (rel. error 2^-22) + rcp.approx (1 ulp); saturate correctly
// (ex2 -> +inf gives rcp -> 0).  No slow-path calls (the IEEE __frcp_rn costs a CALL per element).
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fast_sigmoid(float x) { return rcp_approx(1.0f + ex2_approx(-1.4426950408889634f * x)); }
__device__ __forceinline__ float fast_tanh(float x) { return fmaf(-2.0f, rcp_approx(1.0f + ex2_approx(2.8853900817779268f * x)), 1.0f); }

// split 8 consecutive fp32 into bf16 hi / lo vectors (16 B each)
__device__ __forceinline__ void split8(const float* x, uint4& hi, uint4& lo) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __nv_bfloat162 hh = __floats2bfloat162_rn(x[2 * i], x[2 * i + 1]);
    float r0 = x[2 * i] - __bfloat162float(hh.x), r1 = x[2 * i + 1] - __bfloat162float(hh.y);
    __nv_bfloat162 ll = __floats2bfloat162_rn(r0, r1);
    h[i] = *reinterpret_cast<uint32_t*>(&hh);
    l[i] = *reinterpret_cast<uint32_t*>(&ll);
  }
  hi = make_uint4(h[0], h[1], h[2], h[3]);
  lo = make_uint4(l[0], l[1], l[2], l[3]);
}

// 16 consecutive columns (colbase % 16 == 0) of one lane of a lane-major tile-step in the quad layout
// [col / 4][lane][col % 4] (r4_gemm_tc.cuh: xt_index): four 128-bit loads.  `ts` = tile-step base, `ln4` = lane * 4.
__device__ __forceinline__ void load_x16(float* dst, const float* ts, int colbase, int ln4) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(ts + (size_t)(colbase + 4 * g) * TM + ln4));
    dst[4 * g] = v.x; dst[4 * g + 1] = v.y; dst[4 * g + 2] = v.z; dst[4 * g + 3] = v.w;
  }
}

struct AugruTcSeq {
  const float* XT;        // transposed input halves [n_tiles_cached, 64, 768 / 4, 128, 4]  (tile, step, column quad, lane, column % 4)
  const uint8_t* Wimg;    // pre-tiled bf16 hi/lo weight image of the pair kernels (r4_augru_pair2.cuh: build_pair_image)
  const float* scoresT;   // [n_row_tiles, 64, 128]
  float* out;             // final state, row stride out_ld
  int shared;             // 1: every row reads cached sequence 0
};
struct AugruTcParams {
  AugruTcSeq s[2];
  int R, row0, div, out_ld;
  long long* dbg;         // optional: per-step phase timestamps of CTA 0 (development probe), else null
};

// host-side bf16 rounding (round to nearest even) shared by the weight-image builders
inline uint16_t host_bf16_bits(float x) {
  uint32_t u; memcpy(&u, &x, 4);
  if ((u & 0x7f800000u) == 0x7f800000u) return (uint16_t)(u >> 16);
  u = (u + 0x7fffu + ((u >> 16) & 1u)) >> 16; return (uint16_t)u;
}
inline float host_bf16_val(uint16_t b) { uint32_t u = (uint32_t)b << 16; float f; memcpy(&f, &u, 4); return f; }
}  // namespace r4tc
