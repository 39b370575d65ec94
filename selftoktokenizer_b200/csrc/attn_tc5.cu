// Joint attention of the MMDiT on tcgen05 tensor cores with TMEM accumulators (sm_100a), head_dim 64, fp32 softmax.
// Operands: single-pass 16-bit (IEEE half or bf16), or split bf16 ("bf16x3": hi*hi + hi*lo + lo*hi into the same TMEM
// accumulators for both products, fp32-faithful).  The split mode keeps 2 CTAs per SM by giving up the second Q buffer and
// two of the four K/V stages (one CTA per SM with deeper buffers measured 1362 ms vs 1025 ms per 50-step decode).
//
//   grid           persistent: 2 CTAs per SM (100 KiB smem, 256 TMEM columns each) walk the work items (image, head, 128-query
//                  tile), query tile fastest so that co-running CTAs share one (image, head)'s K / V in L2.  All roles follow
//                  the same item sequence with a CTA-global tile counter that drives ring stages and barrier parities, so
//                  the TMA / MMA warps run into the next item while the softmax warps finish the current one.
//   warp 0         TMA producer: Q tile of the NEXT item (double-buffered), K and V tiles (64 keys x 64 dims) through a 4-stage ring
//   warp 1         MMA issuer (one thread):  S = Q K^T  -> TMEM cols [0,64) / [64,128), double-buffered by tile parity, so
//                                                         Q K^T of tile g+1 overlaps the softmax of tile g (UMMA 128x64x16 x4)
//                                            O += P V   -> TMEM cols [128,192) / [192,256), double-buffered by ITEM parity
//                                                         (A = P from TMEM, B = V MN-major straight from the TMA tile)
//   warps 2-9      two threads per query row (TMEM lane quarter = warp % 4, 32 of the 64 keys / dims each): tcgen05.ld the
//                  half row of S; online softmax in registers (row max exchanged through smem + a 64-thread named barrier;
//                  scale / subtract and row sums on the packed fp32 pipe, ex2.approx, packed cvt); LAZY rescale (the
//                  reference maximum only moves when the running maximum grew by > 2^8, so the O correction pass is rare);
//                  P goes back to TMEM with tcgen05.st as 16-bit pairs IN PLACE of the S columns the thread just read and is
//                  consumed by tcgen05.mma as a TMEM A operand -- no shared-memory round trip, no proxy fence;
//                  the item epilogue (O / l -> A-operand planes of the proj GEMM) is deferred until after the first tile of
//                  the next item, when its wait on the last P V is already satisfied.
//   waits          every mbarrier wait carries a suspend-time hint (the warp sleeps in hardware instead of spinning)
//
// Measured at S = 768, batch 64, 24 heads: 520 us (first version: one CTA per item, P through smem) -> 410-445 us.
//
// Contract (sd3/mmdit.py:521-531, sd3/other_impls.py:37-45): dense non-causal attention over the joint
// [context prefix ; image] sequence; rows < ctx_rows only see keys < ctx_keys (renderer rule, mmdit.py:1581).
// PREFIX variant (decode from a token prefix): image b also ignores the context keys [min(kc, n_ctx[b]), kc), where kc is the
// number of context rows of the launch (image keys start there); key tiles wholly inside that hole are skipped by every role.
#include "common.cuh"
#include "kernels.h"

#include <cuda.h>

#include <algorithm>
#include <cstdlib>

namespace stk {

// provided by gemm_tc.cu
int make_tensor_map_2d(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows, uint32_t box_cols,
                       int fp16);

namespace {

constexpr int HD = 64, BQ = 128, BKV = 64;
// S buffers in TMEM: 2 = S double-buffered + O double-buffered by item parity (deferred item epilogue);
//                    3 = S triple-buffered (Q K^T runs two tiles ahead of the softmax) + ONE O buffer (immediate epilogue)
#ifndef SELFTOK_ATTN5_NSB
#define SELFTOK_ATTN5_NSB 2
#endif
constexpr int NSB = SELFTOK_ATTN5_NSB;
// 1 = the Q K^T instructions are issued by the TMA thread (warp 0), warp 1 issues only P V: neither issuer waits behind the
//     other one's blocking tcgen05.mma issue, and Q K^T of tile g + NSB is launched the moment P V of tile g retires
#ifndef SELFTOK_ATTN5_SPLIT_ISSUE
#define SELFTOK_ATTN5_SPLIT_ISSUE 0
#endif
constexpr bool SPLIT_ISSUE = SELFTOK_ATTN5_SPLIT_ISSUE != 0;
constexpr int Q_BYTES = BQ * HD * 2, KV_TILE_BYTES = BKV * HD * 2;
constexpr int XCH_BYTES = 6 * BQ * 4;               // row-max exchange (2 parities x 2 halves) + partial-sum exchange (2 halves)
// NSPLIT == 1: single-pass 16-bit operands, 2 CTAs per SM.  NSPLIT == 3 ("bf16x3", fp32-faithful): every product is
// hi*hi + hi*lo + lo*hi of bf16 planes accumulated into the same TMEM tile -- Q, K, V arrive as hi and lo planes (twice the
// shared memory: one CTA per SM, three K/V stages), P is split in registers and its lo half goes into the S columns the hi
// half leaves free.
// split mode at 2 CTAs per SM: one Q buffer and two K/V stages (100 KiB per CTA) instead of 2 + 3 (160 KiB, one CTA per SM)
#ifndef SELFTOK_ATTN5_SPLIT_CTAS
#define SELFTOK_ATTN5_SPLIT_CTAS 2
#endif
template <int NSPLIT> struct A5 {
  static constexpr int PL = NSPLIT == 3 ? 2 : 1;                        // operand planes
  static constexpr int MIN_CTAS = NSPLIT == 3 ? SELFTOK_ATTN5_SPLIT_CTAS : 2;
  static constexpr int KV_STAGES = NSPLIT == 3 ? (MIN_CTAS == 2 ? 2 : 3) : 4;
  static constexpr int Q_STAGES = (NSPLIT == 3 && MIN_CTAS == 2) ? 1 : 2;
  static constexpr int Q_STAGE = PL * Q_BYTES;                          // [hi | lo]
  static constexpr int KV_STAGE = PL * 2 * KV_TILE_BYTES;               // [K hi | V hi | K lo | V lo]
  static constexpr int SMEM_TILES = Q_STAGES * Q_STAGE + KV_STAGES * KV_STAGE;   // 96 KiB (P lives in TMEM)
  static constexpr int SMEM_BYTES = SMEM_TILES + 1024 + 256 + XCH_BYTES;   // tiles + alignment slack + barriers + exchange
};
constexpr int TMEM_COLS = 256;      // S0 [0,64) | S1 [64,128) | O0 [128,192) | O1 [192,256); P_g overwrites half of S_g in place
constexpr int NUM_THREADS = 64 + 8 * 32;        // TMA warp, MMA warp, 8 softmax warps
constexpr float kRescaleThreshold = 8.0f;       // log2 units

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// suspend-time hint: a waiting warp sleeps in hardware until the phase flips (or the hint expires) instead of spinning through
// the issue slots that the exp / convert chain of the other warps needs
constexpr uint32_t kSuspendHintNs = 20000;
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(bar), "r"(parity), "r"(kSuspendHintNs) : "memory");
  return ok != 0;
}
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {      // non-blocking
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3ff) == 0 && clock64() - t0 > 8000000000LL) {
      printf("selftok attn_tc5: mbarrier timeout (block %d,%d,%d thread %d bar %u parity %u)\n", blockIdx.x, blockIdx.y, blockIdx.z,
             threadIdx.x, bar, parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// A operand from tensor memory (P of the P V product), B from shared memory
__device__ __forceinline__ void tc_mma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
        "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
        "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// SWIZZLE_128B shared-memory descriptors (cute::UMMA::SmemDescriptor): 8 rows x 128 B atoms, SBO = 1024 B between atoms.
// The same encoding serves the K-major operands (Q, K, P: 64 K-elements per 128 B row) and the MN-major V tile (64 head
// dims contiguous per key row, 8 keys per atom); the major-ness is selected in the instruction descriptor.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// kind::f16 instruction descriptor: D fp32, A/B format (0 = F16, 1 = BF16), a_major bit 15, b_major bit 16 (1 = MN-major)
__device__ __forceinline__ uint32_t make_idesc(int m, int n, int fp16, int b_mn_major) {
  const uint32_t fmt = fp16 ? 0u : 1u;
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// packed fp32 pipe: (x0, x1) = (s0, s1) * scale + nsub;  (a0, a1) += (e0, e1)
__device__ __forceinline__ void scale_sub2(uint32_t s0, uint32_t s1, float scale, float nsub, float& x0, float& x1) {
  asm("{\n\t.reg .b64 x, sc, sb;\n\t"
      "mov.b64 x, {%2, %3};\n\t"
      "mov.b64 sc, {%4, %4};\n\t"
      "mov.b64 sb, {%5, %5};\n\t"
      "fma.rn.f32x2 x, x, sc, sb;\n\t"
      "mov.b64 {%0, %1}, x;\n\t}"
      : "=f"(x0), "=f"(x1) : "r"(s0), "r"(s1), "f"(scale), "f"(nsub));
}
__device__ __forceinline__ void add2(float& a0, float& a1, float e0, float e1) {
  asm("{\n\t.reg .b64 a, b;\n\t"
      "mov.b64 a, {%0, %1};\n\t"
      "mov.b64 b, {%2, %3};\n\t"
      "add.f32x2 a, a, b;\n\t"
      "mov.b64 {%0, %1}, a;\n\t}"
      : "+f"(a0), "+f"(a1) : "f"(e0), "f"(e1));
}
// two fp32 -> packed 16-bit pair (IEEE half or bf16), one cvt instruction
__device__ __forceinline__ uint32_t pack2_16(float lo, float hi, bool fp16) {
  uint32_t r;
  if (fp16) asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  else asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

struct Attn5Params {
  AttnOut out;
  int B, S, H, ctx_rows, ctx_keys, fp16;
  float scale_log2e;
  const int32_t* n_ctx;         // PREFIX: visible context tokens per image [B]
  int kc;                       // PREFIX: context rows of the joint sequence
};

// PREFIX tile map of one item whose image sees context keys [0, hole0) and image keys [kc, S): the n1 key tiles from key 0,
// then the tiles from h1 on (those in between lie wholly inside the hole); kmax_cta = the item's key limit (kc for an item of
// context rows only)
__device__ __forceinline__ int prefix_tiles(int kmax_cta, int hole0, int kc) {
  const int n1 = (min(hole0, kmax_cta) + BKV - 1) / BKV, h1 = max(n1, kc / BKV);
  return n1 + (kmax_cta > kc ? max(0, (kmax_cta + BKV - 1) / BKV - h1) : 0);
}
__device__ __forceinline__ int prefix_key0(int j, int hole0, int kc) {        // first key of the item's j-th tile
  const int n1 = (hole0 + BKV - 1) / BKV;
  return (j < n1 ? j : max(n1, kc / BKV) + (j - n1)) * BKV;
}

template <bool FP16, int NSPLIT, bool PREFIX>
__global__ void __launch_bounds__(NUM_THREADS, A5<NSPLIT>::MIN_CTAS)
attention_tc5_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_kv,
                     const __grid_constant__ CUtensorMap map_q_lo, const __grid_constant__ CUtensorMap map_kv_lo, const Attn5Params p) {
  static_assert(NSPLIT == 1 || (NSPLIT == 3 && !FP16), "split mode uses bf16 planes");
  using C = A5<NSPLIT>;
  constexpr int KV_STAGES = C::KV_STAGES;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t q_s = base;                                  // Q buffer qb at q_s + qb * Q_STAGE (hi plane, lo plane)
  constexpr int QS = C::Q_STAGES;
  static_assert(!SPLIT_ISSUE || QS == 2, "the two-issuer experiment prefetches Q one item ahead");
  const uint32_t kv_s = base + QS * C::Q_STAGE;               // stage st at kv_s + st * KV_STAGE: K hi, V hi (, K lo, V lo)
  const uint32_t bars = kv_s + KV_STAGES * C::KV_STAGE;
  // every per-tile barrier exists twice (tile parity) so that no waiter can be lapped by two phases
  auto q_full = [&](int qb) { return bars + 8u * qb; };
  auto q_empty = [&](int qb) { return bars + 16 + 8u * qb; };
  auto p_ready = [&](int pb) { return bars + 32 + 8u * pb; };               // per S buffer (up to 3)
  auto pv_done = [&](int pb) { return bars + 56 + 8u * pb; };
  auto s_full = [&](int sb) { return bars + 80 + 8u * sb; };
  auto kv_full = [&](int st) { return bars + 104 + 8u * st; };
  auto kv_empty = [&](int st) { return bars + 104 + 8u * KV_STAGES + 8u * st; };
  const uint32_t tmem_slot = bars + 104 + 16u * KV_STAGES;
  // tile g lives in S buffer SB(g), phase SPH(g) of that buffer's barriers; item n accumulates in O buffer OB(n)
  auto SB = [](int g) { return g % NSB; };
  auto SPH = [](int g) { return (uint32_t)((g / NSB) & 1); };
  auto OB = [](int n) { return NSB == 2 ? (n & 1) : 0; };
  const uint32_t xch_s = tmem_slot + 16;
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int S = p.S;
  // persistent CTA: work items (image b, head h, query tile qt), qt fastest, so that the CTAs running side by side share
  // the K / V tiles of one (b, h) in L2.  All roles walk the same item sequence with a CTA-global tile counter g that
  // drives the ring stages and barrier parities, so the TMA / MMA warps run ahead into the next item while the softmax
  // warps finish the current one (no per-item prologue bubble).
  const int nq = (S + BQ - 1) / BQ;
  const int n_items = nq * p.H * p.B;
  // PREFIX: the item's image sees context keys [0, kcb) and image keys [kc, S); its tile sequence is the n1 tiles from key 0
  // followed by the tiles from h1 on (the tiles in between lie wholly inside the hole)
  auto item_tiles = [&](int qt) {
    const int kmax_cta = ((qt + 1) * BQ <= p.ctx_rows) ? p.ctx_keys : S;  // every row of the tile is a context row
    return (kmax_cta + BKV - 1) / BKV;
  };
#define PREFIX_HOLE(item) min(p.kc, __ldg(p.n_ctx + (item) / (nq * p.H)))
#define PREFIX_TILES(item) \
  prefix_tiles((((item) % nq + 1) * BQ <= p.ctx_rows) ? p.ctx_keys : S, PREFIX_HOLE(item), p.kc)

  if (warp == 1 && lane == 0) {
    for (int i = 0; i < 2; ++i) { mbar_init(q_full(i), 1); mbar_init(q_empty(i), 1); }
    for (int i = 0; i < NSB; ++i) { mbar_init(s_full(i), 1); mbar_init(p_ready(i), 8); mbar_init(pv_done(i), 1); }
    for (int st = 0; st < KV_STAGES; ++st) { mbar_init(kv_full(st), 1); mbar_init(kv_empty(st), 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  // S buffer sb at s_tmem0 + 64 * sb; O buffer (item parity) ob at o_tmem0 + 64 * ob.  P_g (16-bit pairs, two keys per
  // column) replaces S_g in place: the thread that loaded S columns [32 half, 32 half + 32) writes its 32 keys into columns
  // [32 half, 32 half + 16) -- nobody else reads those, and Q K^T of tile g+2 (same buffer) is issued after P V of tile g.
  const uint32_t s_tmem0 = tmem_base, o_tmem0 = tmem_base + 64 * NSB;

  // The issuing threads walk the (item, tile) sequence with cursors: the Q K^T cursor runs ahead of the P V cursor (across
  // item boundaries), so S_{g + NSB - 1} is being computed while the softmax warps work on S_g.
  struct Cur { int item, n, j, nt; };
  auto cur_first = [&]() {
    Cur c{(int)blockIdx.x, 0, 0, 0};
    c.nt = c.item < n_items ? (PREFIX ? PREFIX_TILES(c.item) : item_tiles(c.item % nq)) : 0;
    return c;
  };
  auto cur_next = [&](Cur& c) {
    if (++c.j == c.nt) {
      c.item += gridDim.x; ++c.n; c.j = 0;
      c.nt = c.item < n_items ? (PREFIX ? PREFIX_TILES(c.item) : item_tiles(c.item % nq)) : 0;
    }
  };
  Cur cq = cur_first();
  int gq = 0;
  const uint32_t idesc_qk = make_idesc(BQ, BKV, FP16 ? 1 : 0, 0);              // S[128 x 64 keys]: B = K tile, K-major (d contiguous)
  // S[SB(gq)] = Q K_gq^T, then advance the cursor.  wait_free: the caller is not the P V issuer, so the buffer's previous
  // occupant (tile gq - NSB) must be seen retired explicitly instead of through the issue order of one thread.
  auto issue_qk = [&](bool wait_free) {
    const int qb = cq.n % QS, st = gq % KV_STAGES;
    if (cq.j == 0) mbar_wait(q_full(qb), (cq.n / QS) & 1);
    mbar_wait(kv_full(st), (gq / KV_STAGES) & 1);
    if (wait_free && gq >= NSB) mbar_wait(pv_done(SB(gq)), SPH(gq - NSB));
    tc_fence_after();
    const uint32_t ks = kv_s + st * C::KV_STAGE, qs = q_s + qb * C::Q_STAGE;
#pragma unroll
    for (int k = 0; k < HD / 16; ++k) {                                  // K dimension = head dim: 32 B per k-step inside the row
      tc_mma_f16(s_tmem0 + 64 * SB(gq), make_smem_desc(qs + k * 32), make_smem_desc(ks + k * 32), idesc_qk, k > 0 ? 1u : 0u);
      if (NSPLIT == 3) {                                                 // + Q_hi K_lo^T + Q_lo K_hi^T
        tc_mma_f16(s_tmem0 + 64 * SB(gq), make_smem_desc(qs + k * 32), make_smem_desc(ks + 2 * KV_TILE_BYTES + k * 32), idesc_qk, 1u);
        tc_mma_f16(s_tmem0 + 64 * SB(gq), make_smem_desc(qs + Q_BYTES + k * 32), make_smem_desc(ks + k * 32), idesc_qk, 1u);
      }
    }
    tc_commit(s_full(SB(gq)));
    if (cq.j == cq.nt - 1) tc_commit(q_empty(qb));                      // last tile of the item: Q buffer reusable
    cur_next(cq);
    ++gq;
  };

  if (warp == 0) {
    // =========================================================== TMA producer
    if (lane == 0) {
      auto load_q = [&](int item, int n) {                              // n = CTA-local item number
        const int qt = item % nq, h = (item / nq) % p.H, b = item / (nq * p.H);
        const int qb = n % QS;
        mbar_wait(q_empty(qb), ((n / QS) & 1) ^ 1);
        mbar_expect_tx(q_full(qb), C::Q_STAGE);
        tma_load_2d(q_s + qb * C::Q_STAGE, &map_q, q_full(qb), h * HD, b * S + qt * BQ);
        if (NSPLIT == 3) tma_load_2d(q_s + qb * C::Q_STAGE + Q_BYTES, &map_q_lo, q_full(qb), h * HD, b * S + qt * BQ);
      };
      auto load_kv = [&](int item, int j, int g) {
        const int h = (item / nq) % p.H, b = item / (nq * p.H);
        const int row0 = b * S;                                           // first row of this image in the [B*S, 3*H*64] matrix
        const int st = g % KV_STAGES;
        mbar_wait(kv_empty(st), ((g / KV_STAGES) & 1) ^ 1);
        const uint32_t ks = kv_s + st * C::KV_STAGE;
        mbar_expect_tx(kv_full(st), C::KV_STAGE);
        const int key0 = PREFIX ? prefix_key0(j, PREFIX_HOLE(item), p.kc) : j * BKV;
        tma_load_2d(ks, &map_kv, kv_full(st), (p.H + h) * HD, row0 + key0);
        tma_load_2d(ks + KV_TILE_BYTES, &map_kv, kv_full(st), (2 * p.H + h) * HD, row0 + key0);
        if (NSPLIT == 3) {
          tma_load_2d(ks + 2 * KV_TILE_BYTES, &map_kv_lo, kv_full(st), (p.H + h) * HD, row0 + key0);
          tma_load_2d(ks + 3 * KV_TILE_BYTES, &map_kv_lo, kv_full(st), (2 * p.H + h) * HD, row0 + key0);
        }
      };
      if (SPLIT_ISSUE) {
        // this thread also issues Q K^T, two tiles behind its own K/V loads (the loads stay a tile period ahead of their use).
        // The next item's Q is fetched as soon as its buffer is seen free (non-blocking test), at the latest right before the
        // Q K^T that needs it -- a blocking wait at the item start would wait for a Q K^T this thread has not issued yet.
        Cur ct = cur_first();
        int gt = 0, pend_item = -1, pend_n = 0;
        if (ct.item < n_items) load_q(ct.item, 0);
        while (cq.item < n_items) {
          if (pend_item >= 0 && mbar_test(q_empty(pend_n % QS), ((pend_n / QS) & 1) ^ 1)) { load_q(pend_item, pend_n); pend_item = -1; }
          if (ct.item < n_items) {
            if (ct.j == 0 && ct.item + (int)gridDim.x < n_items) {
              while (pend_item >= 0) {                                    // short items: the previous prefetch is still owed
                if (gq < gt && pend_n != cq.n) issue_qk(true);
                else { load_q(pend_item, pend_n); pend_item = -1; }
                if (pend_item >= 0 && mbar_test(q_empty(pend_n % QS), ((pend_n / QS) & 1) ^ 1)) { load_q(pend_item, pend_n); pend_item = -1; }
              }
              pend_item = ct.item + gridDim.x; pend_n = ct.n + 1;
            }
            load_kv(ct.item, ct.j, gt);
            cur_next(ct);
            ++gt;
          }
          if (gq + 2 < gt || ct.item >= n_items) {
            if (pend_item >= 0 && pend_n == cq.n) { load_q(pend_item, pend_n); pend_item = -1; }
            issue_qk(true);
          }
        }
      }
      int g = 0, n = 0;
      if (!SPLIT_ISSUE && (int)blockIdx.x < n_items) load_q(blockIdx.x, 0);
      for (int item = blockIdx.x; !SPLIT_ISSUE && item < n_items; item += gridDim.x, ++n) {
        const int n_tiles = PREFIX ? PREFIX_TILES(item) : item_tiles(item % nq);
        const bool more = item + (int)gridDim.x < n_items;
        if (QS == 2 && more) load_q(item + gridDim.x, n + 1);            // next item's Q, one item ahead
        for (int j = 0; j < n_tiles; ++j, ++g) load_kv(item, j, g);
        if (QS == 1 && more) load_q(item + gridDim.x, n + 1);            // one Q buffer: free once this item's last Q K^T retired
      }
    }
  } else if (warp == 1) {
    // =========================================================== MMA issuer
    if (lane == 0) {
      const uint32_t idesc_pv = make_idesc(BQ, HD, FP16 ? 1 : 0, 1);           // O[128 x 64 dims]: B = V tile, MN-major (d contiguous)
      if (!SPLIT_ISSUE)
        for (int i = 0; i < NSB - 1 && cq.item < n_items; ++i) issue_qk(false);
      Cur cp = cur_first();
      for (int g = 0; cp.item < n_items; ++g) {
        if (!SPLIT_ISSUE && cq.item < n_items) issue_qk(false);          // look-ahead Q K^T (its S buffer was freed by P V_{g-1})
        const int st = g % KV_STAGES;
        const uint32_t vs = kv_s + st * C::KV_STAGE + KV_TILE_BYTES;
        mbar_wait(p_ready(SB(g)), SPH(g));                               // P_g in TMEM, O rescaled (or read out), S[SB(g)] consumed
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < BKV / 16; ++k) {                             // K dimension = keys: 16 keys = 2 atoms of 8 key rows
          const uint32_t pa = s_tmem0 + 64 * SB(g) + 32 * (k >> 1) + 8 * (k & 1);      // P hi; P lo 16 columns further
          tc_mma_f16_ts(o_tmem0 + 64 * OB(cp.n), pa, make_smem_desc(vs + k * 2048), idesc_pv, (cp.j > 0 || k > 0) ? 1u : 0u);
          if (NSPLIT == 3) {                                             // + P_hi V_lo + P_lo V_hi
            tc_mma_f16_ts(o_tmem0 + 64 * OB(cp.n), pa, make_smem_desc(vs + 2 * KV_TILE_BYTES + k * 2048), idesc_pv, 1u);
            tc_mma_f16_ts(o_tmem0 + 64 * OB(cp.n), pa + 16, make_smem_desc(vs + k * 2048), idesc_pv, 1u);
          }
        }
        tc_commit(kv_empty(st));                                         // K/V stage reusable once QK_g and PV_g retire
        tc_commit(pv_done(SB(g)));                                       // O holds tiles 0..j of the item
        cur_next(cp);
      }
    }
  } else {
    // =========================================================== softmax / correction / epilogue
    // 8 warps: TMEM lane quarter = warp % 4 (hardware rule), column half = (warp - 2) / 4.  Two threads share a query row,
    // each owning 32 of the tile's 64 keys (and 32 of the 64 output dims); they exchange only the row maximum per tile
    // (shared memory + a 64-thread named barrier); the row sums stay partial until the end.  Twice the warps of the
    // thread-per-row version hide the fixed-latency stalls of the exp / convert chain.
    const int quarter = warp & 3, half = (warp - 2) >> 2;
    const int rl = quarter * 32 + lane;                                  // row inside the tile = TMEM lane
    const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
    float* xch = reinterpret_cast<float*>(smem_raw + (xch_s - smem_u32(smem_raw)));   // [2 halves][128 rows]
    // Item epilogue (O / l -> 16-bit planes of the proj GEMM and / or fp32), deferred until after the first tile of the
    // NEXT item so that its wait on the last P V is already satisfied and the tensor core keeps running: O is
    // double-buffered by item parity, and the P V that overwrites O[n & 1] (first tile of item n + 2) waits for a p_ready
    // that every softmax warp arrives at only after this read.
    auto epilogue = [&](int item, int n, int g_last, float l_run) {
      const int qt = item % nq, h = (item / nq) % p.H, b = item / (nq * p.H);
      const int row = qt * BQ + rl;
      mbar_wait(pv_done(SB(g_last)), SPH(g_last));
      tc_fence_after();
      uint32_t r0[32];
      tmem_ld32(o_tmem0 + 64 * OB(n) + 32 * half + lane_addr, r0);
      tmem_ld_wait();
      if (row < S) {
        const float inv = 1.0f / l_run;
        const AttnOut& t = p.out;
        const bool inA = row < t.split;
        const int64_t orow = inA ? ((int64_t)b * t.split + row) : ((int64_t)b * (S - t.split) + (row - t.split));
        float* of = inA ? t.f32_a : t.f32_b;
        uint16_t* oh = reinterpret_cast<uint16_t*>(inA ? t.hi_a : t.hi_b);
        uint16_t* ol = reinterpret_cast<uint16_t*>(inA ? t.lo_a : t.lo_b);
        const int64_t o = orow * t.ld + (int64_t)h * HD + 32 * half;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float y[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) y[q] = __uint_as_float(r0[c * 8 + q]) * inv;
          if (of) {
            *reinterpret_cast<float4*>(of + o + c * 8) = make_float4(y[0], y[1], y[2], y[3]);
            *reinterpret_cast<float4*>(of + o + c * 8 + 4) = make_float4(y[4], y[5], y[6], y[7]);
          }
          if (oh) {
            uint32_t hp[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) hp[q] = pack2_sat16(y[2 * q], y[2 * q + 1], FP16);
            *reinterpret_cast<uint4*>(oh + o + c * 8) = make_uint4(hp[0], hp[1], hp[2], hp[3]);
            if (!FP16 && ol) {                                               // bf16 residual planes (split-bf16 consumers)
              uint32_t lp[4];
#pragma unroll
              for (int q = 0; q < 4; ++q) lp[q] = pack2_resid_bf16(y[2 * q], y[2 * q + 1], hp[q]);
              *reinterpret_cast<uint4*>(ol + o + c * 8) = make_uint4(lp[0], lp[1], lp[2], lp[3]);
            }
          }
        }
      }
    };
    int g = 0, n = 0, pend_item = -1, pend_g = 0;
    float pend_l = 1.f;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++n) {
      const int qt = item % nq;
      const int n_tiles = PREFIX ? PREFIX_TILES(item) : item_tiles(qt);
      const int row = qt * BQ + rl;
      const int kmax = (row < p.ctx_rows) ? p.ctx_keys : S;
      const int hole0 = PREFIX ? PREFIX_HOLE(item) : 0;                  // PREFIX: keys [hole0, kc) are hidden
      float m_run = -INFINITY, l_part = 0.f;
      for (int j = 0; j < n_tiles; ++j, ++g) {
        mbar_wait(s_full(SB(g)), SPH(g));
        tc_fence_after();
        uint32_t r0[32];
        tmem_ld32(s_tmem0 + 64 * SB(g) + 32 * half + lane_addr, r0);
        tmem_ld_wait();
        const int k0 = (PREFIX ? prefix_key0(j, hole0, p.kc) : j * BKV) + 32 * half;
        if (k0 + 32 > kmax || (PREFIX && k0 + 32 > hole0 && k0 < p.kc)) {  // tile straddles this row's key limit (or the hole)
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (k0 + i >= kmax || (PREFIX && k0 + i >= hole0 && k0 + i < p.kc)) r0[i] = 0xff800000u;   // -inf
        }
        float mx;
        {
          float mp[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) mp[i] = __uint_as_float(r0[i]);
#pragma unroll
          for (int i = 4; i < 32; ++i) mp[i & 3] = fmaxf(mp[i & 3], __uint_as_float(r0[i]));
          mx = fmaxf(fmaxf(mp[0], mp[1]), fmaxf(mp[2], mp[3]));
        }
        // exchange the half-row maxima (double-buffered by tile parity: no second barrier needed)
        xch[((g & 1) * 2 + half) * BQ + rl] = mx;
        asm volatile("bar.sync %0, 64;" ::"r"(1 + quarter) : "memory");
        mx = fmaxf(mx, xch[((g & 1) * 2 + (half ^ 1)) * BQ + rl]);
        // lazy rescale: the reference maximum only moves when the running maximum grew by more than 2^8 (P <= 256 stays
        // exact enough in 16 bits and the final O / l normalisation cancels the stale offset), so the O correction pass and
        // its wait on the previous P V are rare instead of per tile.  (-inf - -inf = NaN keeps m_run: comparison is false.)
        float m_new = fmaxf(m_run, mx * p.scale_log2e);
        if (m_new - m_run <= kRescaleThreshold) m_new = m_run;
        const float sub = (m_new == -INFINITY) ? 0.f : m_new;
        const float corr = (m_new == m_run || m_new == -INFINITY) ? 1.f : ex2_approx(m_run - m_new);
        // scale / subtract and the row sum run on the packed fp32 pipe (two keys per FFMA2 / FADD2): the softmax warps are
        // co-limited by issue slots and the MUFU pipe, so every instruction saved around the 32 ex2 counts
        uint32_t w[16], wl[16];
        float rsp[4] = {0.f, 0.f, 0.f, 0.f};
        const float nsub = -sub;
#pragma unroll
        for (int q = 0; q < 16; ++q) {
          float x0, x1;
          scale_sub2(r0[2 * q], r0[2 * q + 1], p.scale_log2e, nsub, x0, x1);
          const float e0 = ex2_approx(x0), e1 = ex2_approx(x1);
          add2(rsp[2 * (q & 1)], rsp[2 * (q & 1) + 1], e0, e1);
          w[q] = pack2_16(e0, e1, FP16);
          if (NSPLIT == 3) wl[q] = pack2_resid_bf16(e0, e1, w[q]);          // lo plane: rn(p - rn_bf16(p))
        }
        const float rs = (rsp[0] + rsp[1]) + (rsp[2] + rsp[3]);
        // this thread's 32 keys = 16 packed columns of row rl (TMEM lane) of the A operand of P V, in place of its S columns
        // (split mode: the lo plane takes the other 16 columns of the thread's 32)
        tmem_st16(s_tmem0 + 64 * SB(g) + 32 * half + lane_addr, w);
        if (NSPLIT == 3) tmem_st16(s_tmem0 + 64 * SB(g) + 32 * half + 16 + lane_addr, wl);
        l_part = l_part * corr + rs;
        m_run = m_new;
        // rescale this thread's 32 output dims only when some row of the warp moved its maximum
        if (j > 0 && !__all_sync(0xffffffffu, corr == 1.0f)) {
          mbar_wait(pv_done(SB(g - 1)), SPH(g - 1));                      // PV of the previous tile retired: O is stable
          tc_fence_after();
          tmem_ld32(o_tmem0 + 64 * OB(n) + 32 * half + lane_addr, r0);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i) r0[i] = __float_as_uint(__uint_as_float(r0[i]) * corr);
          tmem_st32(o_tmem0 + 64 * OB(n) + 32 * half + lane_addr, r0);
        }
        tmem_st_wait();                                                   // P (and the rescaled O) are in TMEM
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_ready(SB(g)));
        if (NSB == 2 && j == 0 && pend_item >= 0) {
          epilogue(pend_item, n - 1, pend_g, pend_l);
          pend_item = -1;
        }
      }
      // ---- item end: combine the partial row sums now, leave the read-out of O for after the next item's first tile
      xch[(4 + half) * BQ + rl] = l_part;
      asm volatile("bar.sync %0, 64;" ::"r"(1 + quarter) : "memory");
      pend_l = l_part + xch[(4 + (half ^ 1)) * BQ + rl];
      pend_item = item;
      pend_g = g - 1;
      if (NSB != 2) {                   // one O buffer: read it out now (the next item's first P V waits for our next p_ready)
        epilogue(pend_item, n, pend_g, pend_l);
        pend_item = -1;
      }
    }
    if (pend_item >= 0) epilogue(pend_item, n - 1, pend_g, pend_l);
  }
#undef PREFIX_TILES
#undef PREFIX_HOLE
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS) : "memory");
  }
}

int g_num_sms_dev[64];
bool g_attr_dev[64];       // cudaFuncSetAttribute is per device: one handle per GPU may live in the same process

}  // namespace

int launch_attention_tc5(const __nv_bfloat16* qkv16, int B, int S, int H, int ctx_rows, int ctx_keys, const AttnOut& out,
                         cudaStream_t s, int fp16, const __nv_bfloat16* qkv_lo, const int32_t* n_ctx, int kc) {
  STK_CHECK(qkv16 && B > 0 && S > 0 && H > 0, -1, "attention_tc5: bad arguments");
  STK_CHECK(!n_ctx || (kc > 0 && kc < S && (ctx_keys == 0 || ctx_keys == kc)), -1, "attention_tc5: bad context-prefix window");
  STK_CHECK(out.ld % 8 == 0, -1, "attention_tc5: output pitch must be a multiple of 8");
  STK_CHECK(ctx_keys <= S && ctx_rows <= S && ctx_keys >= 0 && ctx_rows >= 0, -1, "attention_tc5: context limits exceed the sequence");
  STK_CHECK(!(fp16 && qkv_lo), -1, "attention_tc5: the split mode uses bf16 planes");
  STK_TRY(gemm_tc_init());
  int dev = 0;
  STK_CUDA(cudaGetDevice(&dev));
  STK_CHECK(dev >= 0 && dev < 64, -1, "attention_tc5: device ordinal out of range");
  if (!g_attr_dev[dev]) {
    STK_CUDA(cudaDeviceGetAttribute(&g_num_sms_dev[dev], cudaDevAttrMultiProcessorCount, dev));
    STK_CUDA(cudaFuncSetAttribute(attention_tc5_kernel<true, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, A5<1>::SMEM_BYTES));
    STK_CUDA(cudaFuncSetAttribute(attention_tc5_kernel<false, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, A5<1>::SMEM_BYTES));
    STK_CUDA(cudaFuncSetAttribute(attention_tc5_kernel<false, 3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, A5<3>::SMEM_BYTES));
    STK_CUDA(cudaFuncSetAttribute(attention_tc5_kernel<true, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, A5<1>::SMEM_BYTES));
    STK_CUDA(cudaFuncSetAttribute(attention_tc5_kernel<false, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, A5<1>::SMEM_BYTES));
    STK_CUDA(cudaFuncSetAttribute(attention_tc5_kernel<false, 3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, A5<3>::SMEM_BYTES));
    g_attr_dev[dev] = true;
  }
  const int g_num_sms = g_num_sms_dev[dev];
  CUtensorMap mq, mkv, mql, mkvl;
  const uint64_t rows = (uint64_t)B * S, cols = (uint64_t)3 * H * HD;
  STK_TRY(make_tensor_map_2d(&mq, qkv16, rows, cols, BQ, HD, fp16));
  STK_TRY(make_tensor_map_2d(&mkv, qkv16, rows, cols, BKV, HD, fp16));
  mql = mq; mkvl = mkv;
  if (qkv_lo) {
    STK_TRY(make_tensor_map_2d(&mql, qkv_lo, rows, cols, BQ, HD, 0));
    STK_TRY(make_tensor_map_2d(&mkvl, qkv_lo, rows, cols, BKV, HD, 0));
  }
  Attn5Params p{out, B, S, H, ctx_rows, ctx_keys, fp16, 0.125f * 1.4426950408889634f, n_ctx, kc};
  const int n_items = ((S + BQ - 1) / BQ) * H * B;
  if (qkv_lo) {
    dim3 grid(std::min(n_items, A5<3>::MIN_CTAS * g_num_sms));
    if (n_ctx) attention_tc5_kernel<false, 3, true><<<grid, NUM_THREADS, A5<3>::SMEM_BYTES, s>>>(mq, mkv, mql, mkvl, p);
    else attention_tc5_kernel<false, 3, false><<<grid, NUM_THREADS, A5<3>::SMEM_BYTES, s>>>(mq, mkv, mql, mkvl, p);
  } else {
    // persistent: two CTAs per SM walk the item list.  SELFTOK_ATTN5_CTAS_PER_SM=1 is a measurement knob (how much a CTA is
    // slowed by its co-resident twin: profiles/r2_attention_investigation.md); it never changes results.
    static const int ctas_per_sm = [] { const char* e = getenv("SELFTOK_ATTN5_CTAS_PER_SM"); return (e && e[0] == '1') ? 1 : 2; }();
    dim3 grid(std::min(n_items, ctas_per_sm * g_num_sms));
    if (n_ctx) {
      if (fp16) attention_tc5_kernel<true, 1, true><<<grid, NUM_THREADS, A5<1>::SMEM_BYTES, s>>>(mq, mkv, mql, mkvl, p);
      else attention_tc5_kernel<false, 1, true><<<grid, NUM_THREADS, A5<1>::SMEM_BYTES, s>>>(mq, mkv, mql, mkvl, p);
    } else if (fp16) {
      attention_tc5_kernel<true, 1, false><<<grid, NUM_THREADS, A5<1>::SMEM_BYTES, s>>>(mq, mkv, mql, mkvl, p);
    } else {
      attention_tc5_kernel<false, 1, false><<<grid, NUM_THREADS, A5<1>::SMEM_BYTES, s>>>(mq, mkv, mql, mkvl, p);
    }
  }
  count_launch();
  STK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace stk
