// fp32 FFMA kernels of the Selftok path (sm_100a): the encoder's fp32-faithful GEMMs and attention, the fused
// VQ argmax, LayerNorm+modulate, and the small layout kernels.  These also serve as the bisecting reference for
// the tcgen05 kernels (SELFTOK_PREC_FP32_SIMT).
//
// Reference semantics restated here (file:line under /root/reference/mimogpt/models/selftok):
//   linear  : nn.Linear everywhere (modules.py:147-162; sd3/mmdit.py:266-301; sd3/other_impls.py:82-84)
//   ln_mod  : LayerNorm(elementwise_affine=False, eps=1e-6) + modulate (sd3/mmdit.py:78-83,386,407; modules.py:29-32)
//   attn    : F.scaled_dot_product_attention (sd3/other_impls.py:44; modules.py:235-238,263-266)
//   vq      : VectorQuantize eval (vector_quantize_pytorch.py:844-876) -> CosineSimCodebook (:525-563,580),
//             l2norm (:51-52), argmax (:135), final_layer_norm3 (models_ours.py:88,241-242)
#include "common.cuh"
#include "kernels.h"

namespace stk {

// =================================================================================================== linear
// y = act(A W^T + b); tile BM x BN x 16, 256 threads, (BM/16) x (BN/16) micro-tile per thread.  The K loop is a
// sequential FMA chain per output (no split-K): results do not depend on M, the grid or the batch size.
struct LinParams {
  const float* A; int64_t lda;
  const float* W; int64_t ldw;
  int64_t M; int N; int K;
  Epilogue ep;
};

template <int BM, int BN>
__global__ void __launch_bounds__(256, 2) linear_f32_kernel(const LinParams p) {
  constexpr int BK = 16;
  constexpr int TM = BM / 16, TN = BN / 16;          // 4 or 8
  constexpr int CM = TM / 4, CN = TN / 4;            // float4 chunks per thread
  __shared__ __align__(16) float As[2][BK][BM + 4];
  __shared__ __align__(16) float Ws[2][BK][BN + 4];
  const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
  const int64_t m0 = (int64_t)blockIdx.y * BM;
  const int n0 = blockIdx.x * BN;
  constexpr int LA = BM * BK / 4 / 256;              // float4 loads per thread for A (1 or 2)
  constexpr int LW = BN * BK / 4 / 256;
  float4 ra[LA], rw[LW];
  auto gload = [&](int k0) {
#pragma unroll
    for (int i = 0; i < LA; ++i) {
      int f = tid + i * 256; int r = f / 4, kq = (f % 4) * 4;
      int64_t m = m0 + r; int k = k0 + kq;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (m < p.M && k < p.K) v = *reinterpret_cast<const float4*>(p.A + m * p.lda + k);
      ra[i] = v;
    }
#pragma unroll
    for (int i = 0; i < LW; ++i) {
      int f = tid + i * 256; int r = f / 4, kq = (f % 4) * 4;
      int n = n0 + r; int k = k0 + kq;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (n < p.N && k < p.K) v = *reinterpret_cast<const float4*>(p.W + (int64_t)n * p.ldw + k);
      rw[i] = v;
    }
  };
  auto sstore = [&](int buf) {
#pragma unroll
    for (int i = 0; i < LA; ++i) {
      int f = tid + i * 256; int r = f / 4, kq = (f % 4) * 4;
      As[buf][kq + 0][r] = ra[i].x; As[buf][kq + 1][r] = ra[i].y; As[buf][kq + 2][r] = ra[i].z; As[buf][kq + 3][r] = ra[i].w;
    }
#pragma unroll
    for (int i = 0; i < LW; ++i) {
      int f = tid + i * 256; int r = f / 4, kq = (f % 4) * 4;
      Ws[buf][kq + 0][r] = rw[i].x; Ws[buf][kq + 1][r] = rw[i].y; Ws[buf][kq + 2][r] = rw[i].z; Ws[buf][kq + 3][r] = rw[i].w;
    }
  };
  // accumulators as packed pairs (acc[i][2 j2], acc[i][2 j2 + 1]): the inner product runs on FFMA2 (fma.rn.f32x2: two independent
  // round-to-nearest FMAs per issue slot, bit-identical to fmaf per element, same k order), which leaves every other issue slot
  // to the shared-memory loads -- the scalar version spent all of them on FFMA and sat at half the FMA-pipe rate
  unsigned long long acc2[TM][TN / 2];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN / 2; ++j) acc2[i][j] = 0ull;

  const int nk = (p.K + BK - 1) / BK;
  gload(0);
  sstore(0);
  __syncthreads();
  for (int kb = 0; kb < nk; ++kb) {
    const int buf = kb & 1;
    if (kb + 1 < nk) gload((kb + 1) * BK);
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float a[TM];
      unsigned long long w2[TN / 2];
#pragma unroll
      for (int c = 0; c < CM; ++c) {
        float4 v = *reinterpret_cast<const float4*>(&As[buf][k][c * (BM / CM) + ty * 4]);
        a[c * 4 + 0] = v.x; a[c * 4 + 1] = v.y; a[c * 4 + 2] = v.z; a[c * 4 + 3] = v.w;
      }
#pragma unroll
      for (int c = 0; c < CN; ++c) {
        const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(&Ws[buf][k][c * (BN / CN) + tx * 4]);
        w2[c * 2 + 0] = v.x; w2[c * 2 + 1] = v.y;
      }
#pragma unroll
      for (int i = 0; i < TM; ++i) {
        unsigned long long ad;
        asm("mov.b64 %0, {%1, %1};" : "=l"(ad) : "f"(a[i]));
#pragma unroll
        for (int j = 0; j < TN / 2; ++j) asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc2[i][j]) : "l"(ad), "l"(w2[j]));
      }
    }
    if (kb + 1 < nk) {
      sstore(buf ^ 1);
      __syncthreads();
    }
  }
  // ---- epilogue
  const Epilogue& e = p.ep;
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int64_t m = m0 + (i / 4) * (BM / CM) + ty * 4 + (i % 4);
    if (m >= p.M) continue;
    int64_t orow = m;
    if (e.rpb_in > 0) orow = (m / e.rpb_in) * e.rpb_out + e.row_off + (m % e.rpb_in);
#pragma unroll
    for (int c = 0; c < CN; ++c) {
      const int n = n0 + c * (BN / CN) + tx * 4;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int nn = n + j;
        if (nn >= p.N) continue;
        const unsigned long long pr = acc2[i][c * 2 + (j >> 1)];
        float y = __uint_as_float((j & 1) ? (uint32_t)(pr >> 32) : (uint32_t)pr);
        if (e.bias) y += e.bias[nn];
        y = apply_act(y, e.act);
        if (e.mode == EPI_STORE) {
          if (e.addtab) y += e.addtab[(m % e.add_period) * e.add_ld + nn];
          e.out[orow * e.ldo + nn] = y;
        } else if (e.mode == EPI_RESID) {
          float g = e.gate ? e.gate[(m % e.gate_period) * e.gate_ld + nn] : 1.0f;
          e.out[orow * e.ldo + nn] = e.resid[orow * e.ldo + nn] + g * y;
        } else {
          uint16_t hi, lo;
          split16(y, e.fp16, hi, lo);
          reinterpret_cast<uint16_t*>(e.out_hi)[orow * e.ldo + nn] = hi;
          if (e.out_lo) reinterpret_cast<uint16_t*>(e.out_lo)[orow * e.ldo + nn] = lo;
        }
      }
    }
  }
}

int launch_linear_f32(const float* A, int64_t lda, const float* W, int64_t ldw, int64_t M, int N, int K,
                      const Epilogue& ep, cudaStream_t s) {
  STK_CHECK(A && W && M > 0 && N > 0 && K > 0, -1, "linear_f32: bad arguments");
  STK_CHECK(K % 4 == 0 && lda % 4 == 0 && ldw % 4 == 0, -2, "linear_f32: K and leading dims must be multiples of 4");
  STK_CHECK((reinterpret_cast<uintptr_t>(A) % 16 == 0) && (reinterpret_cast<uintptr_t>(W) % 16 == 0), -1,
            "linear_f32: operands must be 16-byte aligned");
  LinParams p{A, lda, W, ldw, M, N, K, ep};
  if (N > 64 && M > 64) {
    dim3 grid((N + 127) / 128, (unsigned)((M + 127) / 128));
    linear_f32_kernel<128, 128><<<grid, 256, 0, s>>>(p);
  } else {
    dim3 grid((N + 63) / 64, (unsigned)((M + 63) / 64));
    linear_f32_kernel<64, 64><<<grid, 256, 0, s>>>(p);
  }
  count_launch();
  STK_CUDA(cudaGetLastError());
  return 0;
}

// =================================================================================================== ln_mod
// One warp per row.  mean and biased variance in two register-resident passes (matches F.layer_norm semantics),
// out = xn * (1 + scale[m % period]) + shift[m % period].
// Per-position tables (period > 1, the context stream): the 8 warps of a CTA take the SAME position of 8 different images
// (imgs > 0), so one shift / scale row (12 KB at D = 1536) serves the whole CTA; it is staged in shared memory with cp.async
// while the x loads are in flight.  With the natural row order every row pulled its own table rows through L2 (2x the
// bytes of x itself), one dependent pair at a time.  Measured on the 96 LN launches of sampler step 0 (batch 64):
// 8.6 ms -> 6.95 ms (position-major) -> 6.1 ms (staged); the context LN moves 302 MB in 65 us (4.6 TB/s, 71 % of the measured
// HBM copy peak), the image LN 151 MB in 34.6 us.  x is streamed (evict-first).
// (A persistent variant with the next row prefetched into registers -- 16 resident warps instead of 24 -- was slower.)
template <int MAXV, bool STAGED>   // STAGED: all 8 rows of the CTA use ONE shift / scale row, staged in shared memory
__global__ void __launch_bounds__(256) ln_mod_kernel(const float* __restrict__ x, int64_t ldx,
                                                     const float* __restrict__ shift, const float* __restrict__ scale,
                                                     int64_t ld_mod, int period, float* __restrict__ out_f32,
                                                     __nv_bfloat16* __restrict__ out_hi, __nv_bfloat16* __restrict__ out_lo,
                                                     int64_t ldo, int64_t M, int D, float eps, int fp16, int imgs) {
  __shared__ __align__(16) float4 tab[STAGED ? 2 * MAXV * 32 : 1];     // [shift | scale] of the CTA's table row
  const int lane = threadIdx.x & 31;
  const int nv = D >> 2;                              // float4 per row
  int64_t m;
  bool active = true;
  if (imgs > 0) {
    const int64_t img = (int64_t)(blockIdx.x / period) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    active = img < imgs;
    m = img * period + (blockIdx.x % period);
  } else {
    m = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    active = m < M;
  }
  if (STAGED) {
    // The table row goes global -> shared with cp.async (no registers), issued BEFORE the x loads so that both latencies
    // overlap; read from L2 once per CTA.  Without this every row walked its 24 table float4 through L1/L2 one dependent
    // pair at a time (12 serial round trips per row) and the kernel sat at 60 % of the HBM roofline.
    const int64_t trow = (imgs > 0) ? (blockIdx.x % period) : 0;
    const float4* sh = reinterpret_cast<const float4*>(shift + trow * ld_mod);
    const float4* sc = reinterpret_cast<const float4*>(scale + trow * ld_mod);
    for (int t = threadIdx.x; t < nv; t += blockDim.x) {
      const uint32_t d0 = (uint32_t)__cvta_generic_to_shared(&tab[t]), d1 = (uint32_t)__cvta_generic_to_shared(&tab[MAXV * 32 + t]);
      asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(d0), "l"(sh + t) : "memory");
      asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(d1), "l"(sc + t) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  } else if (!active) {
    return;
  }
  const float4* xr = reinterpret_cast<const float4*>(x + (active ? m : 0) * ldx);
  float4 v[MAXV];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    int idx = lane + i * 32;
    if (idx < nv) {
      v[i] = __ldcs(xr + idx);
      sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
  }
  const float mean = warp_sum(sum) / (float)D;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    int idx = lane + i * 32;
    if (idx < nv) {
      float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
      sq += (a * a + b * b) + (c * c + d * d);
    }
  }
  const float rstd = rsqrtf(warp_sum(sq) / (float)D + eps);
  const float4 *sh = nullptr, *sc = nullptr;
  if (STAGED) {
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    if (!active) return;
  } else if (shift) {
    const int64_t mrow = (period > 0) ? (m % period) : 0;
    sh = reinterpret_cast<const float4*>(shift + mrow * ld_mod);
    sc = reinterpret_cast<const float4*>(scale + mrow * ld_mod);
  }
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    int idx = lane + i * 32;
    if (idx < nv) {
      float4 y;
      y.x = (v[i].x - mean) * rstd; y.y = (v[i].y - mean) * rstd; y.z = (v[i].z - mean) * rstd; y.w = (v[i].w - mean) * rstd;
      if (STAGED || sc) {
        const float4 h4 = STAGED ? tab[idx] : sh[idx], s4 = STAGED ? tab[MAXV * 32 + idx] : sc[idx];
        y.x = y.x * (1.f + s4.x) + h4.x; y.y = y.y * (1.f + s4.y) + h4.y;
        y.z = y.z * (1.f + s4.z) + h4.z; y.w = y.w * (1.f + s4.w) + h4.w;
      }
      if (out_f32) reinterpret_cast<float4*>(out_f32 + m * ldo)[idx] = y;
      if (out_hi) {
        uint16_t h0, h1, h2, h3, l0, l1, l2, l3;
        split16(y.x, fp16, h0, l0); split16(y.y, fp16, h1, l1); split16(y.z, fp16, h2, l2); split16(y.w, fp16, h3, l3);
        reinterpret_cast<uint2*>(out_hi + m * ldo)[idx] = make_uint2(h0 | ((uint32_t)h1 << 16), h2 | ((uint32_t)h3 << 16));
        if (out_lo) reinterpret_cast<uint2*>(out_lo + m * ldo)[idx] = make_uint2(l0 | ((uint32_t)l1 << 16), l2 | ((uint32_t)l3 << 16));
      }
    }
  }
}

int launch_ln_mod(const float* x, int64_t ldx, const float* shift, const float* scale, int64_t ld_mod, int period,
                  float* out_f32, __nv_bfloat16* out_hi, __nv_bfloat16* out_lo, int64_t ldo, int64_t M, int D,
                  float eps, cudaStream_t s, int fp16) {
  STK_CHECK(x && M > 0 && D > 0 && D % 4 == 0 && ldx % 4 == 0 && ldo % 4 == 0 && ld_mod % 4 == 0, -1, "ln_mod: bad arguments");
  STK_CHECK((shift == nullptr) == (scale == nullptr), -1, "ln_mod: shift and scale must both be given or both NULL");
  STK_CHECK(D <= 2048, -2, "ln_mod: D > 2048 unsupported");
  const int wpb = 8;
  // position-major mapping when the rows are [image][position] with per-position tables (see the kernel comment)
  const int imgs = (period > 1 && shift && M % period == 0 && M / period >= 2) ? (int)(M / period) : 0;
  dim3 grid(imgs ? (unsigned)(period * ((imgs + wpb - 1) / wpb)) : (unsigned)((M + wpb - 1) / wpb));
  const bool staged = shift && (imgs > 0 || period <= 1);            // one table row per CTA
#define STK_LN(MAXV, ST)                                                                                                      \
  ln_mod_kernel<MAXV, ST><<<grid, wpb * 32, 0, s>>>(x, ldx, shift, scale, ld_mod, period, out_f32, out_hi, out_lo, ldo, M, D, eps, \
                                                    fp16, imgs)
  if (D <= 512) { if (staged) STK_LN(4, true); else STK_LN(4, false); }
  else if (D <= 1536) { if (staged) STK_LN(12, true); else STK_LN(12, false); }
  else { if (staged) STK_LN(16, true); else STK_LN(16, false); }
#undef STK_LN
  count_launch();
  STK_CUDA(cudaGetLastError());
  return 0;
}

// ---- the two LN + modulate passes of an MMDiT layer stage (context rows, image rows) in ONE launch, 16-bit plane output.
// Each CTA = 8 rows that share one shift / scale table row (staged in shared memory with cp.async under the x loads):
// context problem position-major (the same position of 8 images), image problem natural order with its single per-step row.
// One launch instead of two keeps the small late-schedule launches (B * Kc rows with Kc down to 20) from each leaving most
// of the 148 SMs idle, and the output mode is compile-time (no per-element branches; one saturating F2FP per pair).
struct LnPairParams {
  LnProblem pr[2];
  int nblk0;               // CTAs of problem 0 (problem 1 owns the rest of the grid)
  int D;
  float eps;
};

// FULL: D == MAXV * 128 exactly (1536 with MAXV 12: the MMDiT), so that no per-chunk bounds predicate is compiled in.
// ROWS: rows per warp (the CTA covers 8 * ROWS rows that share one table row): the prologue -- index arithmetic, the staged table,
// the CTA launch itself -- is ~370 of the ~590 instructions a warp spends on its first row.
template <int MAXV, bool FP16, bool LO, bool FULL, int ROWS>
__global__ void __launch_bounds__(256) ln_mod_pair_kernel(const LnPairParams p) {
  __shared__ __align__(16) float4 tab[2 * MAXV * 32];
  const bool second = (int)blockIdx.x >= p.nblk0;
  const LnProblem& q = second ? p.pr[1] : p.pr[0];
  const int blk = second ? (int)blockIdx.x - p.nblk0 : (int)blockIdx.x;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int nv = p.D >> 2;
  // row r of this warp: position-major (imgs > 0): image (blk / period) * 8 ROWS + wid + 8 r at position blk % period;
  // natural order: row blk * 8 ROWS + wid + 8 r, one table row for the whole problem
  const bool pos_major = q.imgs > 0;
  const int64_t first = pos_major ? (int64_t)(blk / q.period) * (8 * ROWS) + wid : (int64_t)blk * (8 * ROWS) + wid;
  const int64_t trow = pos_major ? blk % q.period : 0;
  const int64_t limit = pos_major ? q.imgs : q.M;
  {
    const float4* sh = reinterpret_cast<const float4*>(q.shift + trow * q.ld_mod);
    const float4* sc = reinterpret_cast<const float4*>(q.scale + trow * q.ld_mod);
    for (int t = threadIdx.x; t < nv; t += 256) {
      const uint32_t d0 = (uint32_t)__cvta_generic_to_shared(&tab[t]), d1 = (uint32_t)__cvta_generic_to_shared(&tab[MAXV * 32 + t]);
      asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(d0), "l"(sh + t) : "memory");
      asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(d1), "l"(sc + t) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  // All row arithmetic runs on the packed fp32 pipe (FADD2 / FFMA2, two elements per issue slot): under the 1 kW cap the SMs
  // clock at ~1.35 GHz and this kernel is bound by instruction issue, not by HBM (91 % of the copy rate at burst clocks,
  // 69 % in situ before this change).
#pragma unroll 1
  for (int r = 0; r < ROWS; ++r) {
    const int64_t unit = first + 8 * r;
    const bool active = unit < limit;                                  // warp-uniform
    const int64_t m = pos_major ? unit * q.period + trow : unit;
    float4 v[MAXV];
    float rstd = 0.f, nmr = 0.f;
    if (active) {
      const float4* xr = reinterpret_cast<const float4*>(q.x + m * (int64_t)p.D);
      float s0 = 0.f, s1 = 0.f;
#pragma unroll
      for (int i = 0; i < MAXV; ++i) {
        const int idx = lane + i * 32;
        if (FULL || idx < nv) {
          v[i] = __ldcs(xr + idx);
          fadd2(s0, s1, v[i].x, v[i].y, s0, s1);
          fadd2(s0, s1, v[i].z, v[i].w, s0, s1);
        }
      }
      const float mean = warp_sum(s0 + s1) / (float)p.D;
      const float nmean = -mean;
      float q0 = 0.f, q1 = 0.f;
#pragma unroll
      for (int i = 0; i < MAXV; ++i) {
        const int idx = lane + i * 32;
        if (FULL || idx < nv) {
          float a, b, c, d;
          fadd2(v[i].x, v[i].y, nmean, nmean, a, b);
          fadd2(v[i].z, v[i].w, nmean, nmean, c, d);
          ffma2(a, b, a, b, q0, q1, q0, q1);
          ffma2(c, d, c, d, q0, q1, q0, q1);
        }
      }
      rstd = rsqrtf(warp_sum(q0 + q1) / (float)p.D + p.eps);
      nmr = nmean * rstd;                                              // xn = x * rstd - mean * rstd
    }
    if (r == 0) {                                                      // the table is needed from here on; every warp passes once
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      __syncthreads();
    }
    if (!active) continue;
    uint2* oh = reinterpret_cast<uint2*>(q.out_hi + m * (int64_t)p.D);
    uint2* ol = LO ? reinterpret_cast<uint2*>(q.out_lo + m * (int64_t)p.D) : nullptr;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int idx = lane + i * 32;
      if (FULL || idx < nv) {
        const float4 h4 = tab[idx], s4 = tab[MAXV * 32 + idx];
        float4 y, g;
        ffma2(v[i].x, v[i].y, rstd, rstd, nmr, nmr, y.x, y.y);
        ffma2(v[i].z, v[i].w, rstd, rstd, nmr, nmr, y.z, y.w);
        fadd2(s4.x, s4.y, 1.f, 1.f, g.x, g.y);
        fadd2(s4.z, s4.w, 1.f, 1.f, g.z, g.w);
        ffma2(y.x, y.y, g.x, g.y, h4.x, h4.y, y.x, y.y);
        ffma2(y.z, y.w, g.z, g.w, h4.z, h4.w, y.z, y.w);
        const uint32_t p0 = pack2_sat16(y.x, y.y, FP16), p1 = pack2_sat16(y.z, y.w, FP16);
        oh[idx] = make_uint2(p0, p1);
        if (LO) ol[idx] = make_uint2(pack2_resid_bf16(y.x, y.y, p0), pack2_resid_bf16(y.z, y.w, p1));
      }
    }
  }
}

int launch_ln_mod_pair(const LnProblem* probs, int n, int D, float eps, cudaStream_t s, int fp16) {
  STK_CHECK(probs && (n == 1 || n == 2) && D > 0 && D % 4 == 0 && D <= 2048, -1, "ln_mod_pair: bad arguments");
  LnPairParams p;
  p.D = D; p.eps = eps;
  int nblk[2] = {0, 0};
  bool lo = false;
  // two rows per warp when that still leaves >= 4 CTAs per SM of a B200 (halves the per-row share of the prologue); else one
  auto ctas_for = [&](int rows_per_warp) {
    int64_t c = 0;
    for (int i = 0; i < n; ++i) {
      const LnProblem& q = probs[i];
      const int64_t units = q.period > 1 ? q.M / q.period : q.M;
      c += (q.period > 1 ? q.period : 1) * ((units + 8 * rows_per_warp - 1) / (8 * rows_per_warp));
    }
    return c;
  };
  const int rows = ctas_for(2) >= 4 * 148 ? 2 : 1;
  for (int i = 0; i < 2; ++i) {
    if (i >= n) { p.pr[i] = probs[0]; p.pr[i].M = 0; continue; }
    LnProblem q = probs[i];
    STK_CHECK(q.x && q.shift && q.scale && q.out_hi && q.M > 0 && q.ld_mod % 4 == 0, -1, "ln_mod_pair: bad problem");
    STK_CHECK(i == 0 || (q.out_lo != nullptr) == lo, -1, "ln_mod_pair: both problems must use the same plane set");
    lo = q.out_lo != nullptr;
    if (q.period > 1) {                                // per-position table: position-major, needs whole images
      STK_CHECK(q.M % q.period == 0, -1, "ln_mod_pair: rows must be whole images of `period` positions");
      q.imgs = (int)(q.M / q.period);
      nblk[i] = q.period * ((q.imgs + 8 * rows - 1) / (8 * rows));
    } else {
      q.period = 1; q.imgs = 0;
      nblk[i] = (int)((q.M + 8 * rows - 1) / (8 * rows));
    }
    p.pr[i] = q;
  }
  STK_CHECK(!(fp16 && lo), -1, "ln_mod_pair: the fp16 mode has no residual planes");
  p.nblk0 = nblk[0];
  const unsigned grid = (unsigned)(nblk[0] + nblk[1]);
#define STK_LNP3(MAXV, FULL, ROWS)                                                          \
  do {                                                                                      \
    if (fp16) ln_mod_pair_kernel<MAXV, true, false, FULL, ROWS><<<grid, 256, 0, s>>>(p);    \
    else if (lo) ln_mod_pair_kernel<MAXV, false, true, FULL, ROWS><<<grid, 256, 0, s>>>(p); \
    else ln_mod_pair_kernel<MAXV, false, false, FULL, ROWS><<<grid, 256, 0, s>>>(p);        \
  } while (0)
#define STK_LNP(MAXV)                                                                       \
  do {                                                                                      \
    if (D == MAXV * 128) {                                                                  \
      if (rows == 2) STK_LNP3(MAXV, true, 2); else STK_LNP3(MAXV, true, 1);                 \
    } else {                                                                                \
      if (rows == 2) STK_LNP3(MAXV, false, 2); else STK_LNP3(MAXV, false, 1);               \
    }                                                                                       \
  } while (0)
  if (D <= 512) STK_LNP(4);
  else if (D <= 1536) STK_LNP(12);
  else STK_LNP(16);
#undef STK_LNP
#undef STK_LNP3
  count_launch();
  STK_CUDA(cudaGetLastError());
  return 0;
}

// =================================================================================================== attention (fp32)
// One CTA = 64 queries of one (batch, head); 256 threads as 16 x 16; keys streamed in tiles of 64 with an online
// softmax.  S-phase: thread (ty,tx) owns rows ty*4..+3 x keys tx*4..+3; PV-phase: rows ty*4..+3 x dims tx*(HD/16)..
struct AttnParams {
  const float* q; int64_t q_ld, q_bs;
  const float* k1; const float* v1; int64_t kv1_ld, kv1_bs; int S1;
  const float* k2; const float* v2; int64_t kv2_ld, kv2_bs; int S2;
  AttnOut out;
  int Sq, H, ctx_rows, ctx_keys;
  float scale;
  const int32_t* n_ctx;   // PREFIX: visible context tokens per image [B]
  int kc;                 // PREFIX: context keys; image b ignores keys [min(kc, n_ctx[b]), kc)
};

template <int HD, bool PREFIX = false>
__global__ void __launch_bounds__(256) attention_f32_kernel(const AttnParams p) {
  constexpr int BQ = 64, BKV = 64, DV = HD / 16;
  extern __shared__ __align__(16) float smem[];
  float* Qt = smem;                          // [HD][BQ+4]
  float* Kt = Qt + HD * (BQ + 4);            // [HD][BKV+4]
  float* Vs = Kt + HD * (BKV + 4);           // [BKV][HD]
  float* Pt = Vs + BKV * HD;                 // [BKV][BQ+4]
  const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
  const int q0 = blockIdx.x * BQ, h = blockIdx.y, b = blockIdx.z;
  const int Sk = p.S1 + p.S2;
  // ---- Q tile -> smem (transposed), pre-scaled
  for (int f = tid; f < BQ * HD / 4; f += 256) {
    int r = f / (HD / 4), d4 = (f % (HD / 4)) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (q0 + r < p.Sq) v = *reinterpret_cast<const float4*>(p.q + (int64_t)b * p.q_bs + (int64_t)(q0 + r) * p.q_ld + h * HD + d4);
    Qt[(d4 + 0) * (BQ + 4) + r] = v.x * p.scale; Qt[(d4 + 1) * (BQ + 4) + r] = v.y * p.scale;
    Qt[(d4 + 2) * (BQ + 4) + r] = v.z * p.scale; Qt[(d4 + 3) * (BQ + 4) + r] = v.w * p.scale;
  }
  float m_i[4], l_i[4], o[4][DV];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    m_i[i] = -INFINITY; l_i[i] = 0.f;
#pragma unroll
    for (int d = 0; d < DV; ++d) o[i][d] = 0.f;
  }
  // keys a row may see
  int kmax_row[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) kmax_row[i] = (q0 + ty * 4 + i < p.ctx_rows) ? p.ctx_keys : Sk;
  int kmax_cta = (q0 + BQ <= p.ctx_rows) ? p.ctx_keys : Sk;        // all rows of this CTA are context rows
  const int hole0 = PREFIX ? min(p.kc, p.n_ctx[b]) : 0;            // PREFIX: keys [hole0, kc) are hidden
  for (int k0 = 0; k0 < kmax_cta; k0 += BKV) {
    if (PREFIX && k0 >= hole0 && k0 + BKV <= p.kc) continue;      // tile wholly inside the hole
    __syncthreads();                                              // previous tile fully consumed (also covers Qt)
    for (int f = tid; f < BKV * HD / 4; f += 256) {
      int r = f / (HD / 4), d4 = (f % (HD / 4)) * 4;
      int key = k0 + r;
      float4 kv = make_float4(0.f, 0.f, 0.f, 0.f), vv = kv;
      if (key < Sk) {
        const float *kp, *vp;
        if (key < p.S1) {
          int64_t off = (int64_t)b * p.kv1_bs + (int64_t)key * p.kv1_ld + h * HD + d4;
          kp = p.k1 + off; vp = p.v1 + off;
        } else {
          int64_t off = (int64_t)b * p.kv2_bs + (int64_t)(key - p.S1) * p.kv2_ld + h * HD + d4;
          kp = p.k2 + off; vp = p.v2 + off;
        }
        kv = *reinterpret_cast<const float4*>(kp);
        vv = *reinterpret_cast<const float4*>(vp);
      }
      Kt[(d4 + 0) * (BKV + 4) + r] = kv.x; Kt[(d4 + 1) * (BKV + 4) + r] = kv.y;
      Kt[(d4 + 2) * (BKV + 4) + r] = kv.z; Kt[(d4 + 3) * (BKV + 4) + r] = kv.w;
      *reinterpret_cast<float4*>(&Vs[r * HD + d4]) = vv;
    }
    __syncthreads();
    // ---- S = Q K^T (4 x 4 per thread)
    // packed fp32 pipe (FFMA2: two independent round-to-nearest FMAs per issue slot, bit-identical to fmaf per element and in the
    // same d order): accumulators as key pairs, the query element duplicated into both lanes
    float sacc[4][4];
    {
      unsigned long long s2[4][2];
#pragma unroll
      for (int i = 0; i < 4; ++i) s2[i][0] = s2[i][1] = 0ull;
#pragma unroll 8
      for (int d = 0; d < HD; ++d) {
        const float4 a = *reinterpret_cast<const float4*>(&Qt[d * (BQ + 4) + ty * 4]);
        const ulonglong2 kk = *reinterpret_cast<const ulonglong2*>(&Kt[d * (BKV + 4) + tx * 4]);
        const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          unsigned long long ad;
          asm("mov.b64 %0, {%1, %1};" : "=l"(ad) : "f"(av[i]));
          asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(s2[i][0]) : "l"(ad), "l"(kk.x));
          asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(s2[i][1]) : "l"(ad), "l"(kk.y));
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          sacc[i][2 * j] = __uint_as_float((uint32_t)s2[i][j]);
          sacc[i][2 * j + 1] = __uint_as_float((uint32_t)(s2[i][j] >> 32));
        }
    }
    // ---- online softmax over this tile (row statistics shared by the 16 threads of a half-warp)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        int key = k0 + tx * 4 + j;
        if (key >= kmax_row[i] || (PREFIX && key >= hole0 && key < p.kc)) sacc[i][j] = -INFINITY;
        mx = fmaxf(mx, sacc[i][j]);
      }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
      const float m_new = fmaxf(m_i[i], mx);
      const float corr = (m_new == -INFINITY) ? 1.f : expf(m_i[i] - m_new);
      float rs = 0.f;
      float pv[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        pv[j] = (sacc[i][j] == -INFINITY) ? 0.f : expf(sacc[i][j] - m_new);
        rs += pv[j];
      }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) rs += __shfl_xor_sync(0xffffffffu, rs, off);
      l_i[i] = l_i[i] * corr + rs;
      m_i[i] = m_new;
#pragma unroll
      for (int d = 0; d < DV; ++d) o[i][d] *= corr;
#pragma unroll
      for (int j = 0; j < 4; ++j) Pt[(tx * 4 + j) * (BQ + 4) + ty * 4 + i] = pv[j];
    }
    __syncthreads();
    // ---- O += P V
    if (DV % 2 == 0) {                                     // head dims 32 / 64: output-dim pairs on FFMA2, P duplicated
      constexpr int DP = DV / 2 > 0 ? DV / 2 : 1;
      unsigned long long o2[4][DP];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int d = 0; d < DP; ++d) asm("mov.b64 %0, {%1, %2};" : "=l"(o2[i][d]) : "f"(o[i][2 * d]), "f"(o[i][(2 * d + 1) % DV]));
#pragma unroll 8
      for (int key = 0; key < BKV; ++key) {
        const float4 pp = *reinterpret_cast<const float4*>(&Pt[key * (BQ + 4) + ty * 4]);
        const float pr[4] = {pp.x, pp.y, pp.z, pp.w};
        unsigned long long v2[DP];
#pragma unroll
        for (int d = 0; d < DP; ++d) v2[d] = *reinterpret_cast<const unsigned long long*>(&Vs[key * HD + tx * DV + 2 * d]);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          unsigned long long pd;
          asm("mov.b64 %0, {%1, %1};" : "=l"(pd) : "f"(pr[i]));
#pragma unroll
          for (int d = 0; d < DP; ++d) asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(o2[i][d]) : "l"(pd), "l"(v2[d]));
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int d = 0; d < DP; ++d) {
          o[i][2 * d] = __uint_as_float((uint32_t)o2[i][d]);
          if (2 * d + 1 < DV) o[i][2 * d + 1] = __uint_as_float((uint32_t)(o2[i][d] >> 32));
        }
    } else {
#pragma unroll 8
      for (int key = 0; key < BKV; ++key) {
        float4 pp = *reinterpret_cast<const float4*>(&Pt[key * (BQ + 4) + ty * 4]);
        float pr[4] = {pp.x, pp.y, pp.z, pp.w};
        float vv[DV];
#pragma unroll
        for (int d = 0; d < DV; ++d) vv[d] = Vs[key * HD + tx * DV + d];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int d = 0; d < DV; ++d) o[i][d] = fmaf(pr[i], vv[d], o[i][d]);
      }
    }
  }
  // ---- normalise + store
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int row = q0 + ty * 4 + i;
    if (row >= p.Sq) continue;
    const float inv = 1.0f / l_i[i];
    const AttnOut& t = p.out;
    const bool inA = row < t.split;
    const int64_t orow = inA ? ((int64_t)b * t.split + row) : ((int64_t)b * (p.Sq - t.split) + (row - t.split));
    float* of = inA ? t.f32_a : t.f32_b;
    __nv_bfloat16* oh = inA ? t.hi_a : t.hi_b;
    __nv_bfloat16* ol = inA ? t.lo_a : t.lo_b;
#pragma unroll
    for (int d = 0; d < DV; ++d) {
      const float y = o[i][d] * inv;
      const int64_t idx = orow * t.ld + h * HD + tx * DV + d;
      if (of) of[idx] = y;
      if (oh) {
        uint16_t hi, lo;
        split16(y, t.fp16, hi, lo);
        reinterpret_cast<uint16_t*>(oh)[idx] = hi;
        if (ol) reinterpret_cast<uint16_t*>(ol)[idx] = lo;
      }
    }
  }
}

int launch_attention_f32(const float* q, int64_t q_ld, int64_t q_bs, const float* k1, const float* v1, int64_t kv1_ld,
                         int64_t kv1_bs, int S1, const float* k2, const float* v2, int64_t kv2_ld, int64_t kv2_bs,
                         int S2, const AttnOut& out, int B, int Sq, int H, int hd, int ctx_rows, int ctx_keys,
                         cudaStream_t s, const int32_t* n_ctx, int kc) {
  STK_CHECK(q && k1 && v1 && B > 0 && Sq > 0 && H > 0 && S1 > 0 && S2 >= 0, -1, "attention_f32: bad arguments");
  STK_CHECK(!n_ctx || (hd == 64 && kc > 0 && kc < S1 + S2 && (ctx_keys == 0 || ctx_keys == kc)), -1,
            "attention_f32: bad context-prefix window");
  STK_CHECK(hd == 16 || hd == 32 || hd == 64, -2, "attention_f32: head_dim must be 16, 32 or 64");
  STK_CHECK(q_ld % 4 == 0 && kv1_ld % 4 == 0 && (S2 == 0 || kv2_ld % 4 == 0), -1, "attention_f32: strides must be multiples of 4");
  AttnParams p{q, q_ld, q_bs, k1, v1, kv1_ld, kv1_bs, S1, k2, v2, kv2_ld, kv2_bs, S2, out, Sq, H, ctx_rows, ctx_keys,
               1.0f / sqrtf((float)hd), n_ctx, kc};
  dim3 grid((Sq + 63) / 64, H, B);
  size_t smem = sizeof(float) * (size_t)(hd * 68 * 2 + 64 * hd + 64 * 68);
  if (hd == 64) {
    static bool attr[64];                                        // per device (one handle per GPU may share the process)
    int dev = 0;
    STK_CUDA(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && !attr[dev]) {
      STK_CUDA(cudaFuncSetAttribute(attention_f32_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      STK_CUDA(cudaFuncSetAttribute(attention_f32_kernel<64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      attr[dev] = true;
    }
    if (n_ctx) attention_f32_kernel<64, true><<<grid, 256, smem, s>>>(p);
    else attention_f32_kernel<64><<<grid, 256, smem, s>>>(p);
  } else if (hd == 32) {
    attention_f32_kernel<32><<<grid, 256, smem, s>>>(p);
  } else {
    attention_f32_kernel<16><<<grid, 256, smem, s>>>(p);
  }
  count_launch();
  STK_CUDA(cudaGetLastError());
  return 0;
}

// =================================================================================================== VQ
// One CTA = 64 rows.  Prologue: x = z W_in^T + b (Q -> 16), x_hat = x / max(||x||, 1e-12).  Main loop: the codebook
// (pre-transposed [16][N], 2 MiB, L2 resident) is streamed in 128-code chunks through a cp.async double buffer;
// thread (ty,tx) keeps its 4 rows' x_hat in registers (64 regs) and scores 8 codes per chunk, tracking a running
// (max, first index).  Nothing of the [R, N] similarity matrix is ever materialised.
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

constexpr int VQ_TM = 64, VQ_CH = 128, VQ_DIM = 16;

__global__ void __launch_bounds__(256) vq_kernel(const float* __restrict__ z, int64_t R, int Q,
                                                 const float* __restrict__ w_in, const float* __restrict__ b_in,
                                                 const float* __restrict__ codebook, const float* __restrict__ cbt,
                                                 int n_codes, const float* __restrict__ ln_w,
                                                 const float* __restrict__ ln_b, int64_t* __restrict__ ids,
                                                 float* __restrict__ outs_q) {
  // phase 1 (projection) and phase 2 (codebook sweep) reuse the same 25 KiB of shared memory
  __shared__ __align__(16) float pool[2 * VQ_DIM * (VQ_CH + 4) + 2 * VQ_TM * 16];
  __shared__ __align__(16) float xt[VQ_DIM][VQ_TM + 4];         // x_hat transposed
  float (*zs)[68] = reinterpret_cast<float (*)[68]>(pool);                        // [64 rows][64 k] (+pad)
  float (*wsm)[68] = reinterpret_cast<float (*)[68]>(pool + VQ_TM * 68);          // [16][64 k] (+pad)
  float (*cs)[VQ_DIM][VQ_CH + 4] = reinterpret_cast<float (*)[VQ_DIM][VQ_CH + 4]>(pool);   // [2][16][128+4]
  float (*red_v)[16] = reinterpret_cast<float (*)[16]>(pool + 2 * VQ_DIM * (VQ_CH + 4));
  int (*red_i)[16] = reinterpret_cast<int (*)[16]>(pool + 2 * VQ_DIM * (VQ_CH + 4) + VQ_TM * 16);
  static_assert(VQ_TM * 68 + VQ_DIM * 68 <= 2 * VQ_DIM * (VQ_CH + 4) + 2 * VQ_TM * 16, "phase-1 tiles must fit the pool");
  const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
  const int64_t r0 = (int64_t)blockIdx.x * VQ_TM;
  // ---- projection: thread (row = tid/4, outputs (tid%4)*4 .. +3)
  {
    const int prow = tid / 4, po = (tid % 4) * 4;
    float pacc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int k0 = 0; k0 < Q; k0 += 64) {
      __syncthreads();
      for (int f = tid; f < VQ_TM * 16; f += 256) {
        int r = f / 16, c4 = (f % 16) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r0 + r < R && k0 + c4 < Q) v = *reinterpret_cast<const float4*>(z + (r0 + r) * (int64_t)Q + k0 + c4);
        *reinterpret_cast<float4*>(&zs[r][c4]) = v;
      }
      {
        int o = tid / 16, c4 = (tid % 16) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k0 + c4 < Q) v = *reinterpret_cast<const float4*>(w_in + (int64_t)o * Q + k0 + c4);
        *reinterpret_cast<float4*>(&wsm[o][c4]) = v;
      }
      __syncthreads();
#pragma unroll 16
      for (int k = 0; k < 64; ++k) {
        const float zv = zs[prow][k];
#pragma unroll
        for (int j = 0; j < 4; ++j) pacc[j] = fmaf(zv, wsm[po + j][k], pacc[j]);
      }
    }
    float ss = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) { pacc[j] += b_in[po + j]; ss += pacc[j] * pacc[j]; }
    ss += __shfl_xor_sync(0xffffffffu, ss, 1);
    ss += __shfl_xor_sync(0xffffffffu, ss, 2);
    const float nrm = fmaxf(sqrtf(ss), 1e-12f);                   // F.normalize(p=2, eps=1e-12)
#pragma unroll
    for (int j = 0; j < 4; ++j) xt[po + j][prow] = pacc[j] / nrm;
  }
  __syncthreads();
  float xr[4][VQ_DIM];
#pragma unroll
  for (int d = 0; d < VQ_DIM; ++d) {
    float4 v = *reinterpret_cast<const float4*>(&xt[d][ty * 4]);
    xr[0][d] = v.x; xr[1][d] = v.y; xr[2][d] = v.z; xr[3][d] = v.w;
  }
  float best[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
  int besti[4] = {0, 0, 0, 0};
  const int nch = (n_codes + VQ_CH - 1) / VQ_CH;
  auto issue = [&](int ch, int buf) {
    // 16 dims x 128 codes = 512 x 16 B; 2 per thread
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      int f = tid + i * 256;
      int d = f / 32, c4 = (f % 32) * 4;
      int code = ch * VQ_CH + c4;
      if (code + 3 < n_codes) cp_async16(&cs[buf][d][c4], cbt + (int64_t)d * n_codes + code);
      else {
        for (int j = 0; j < 4; ++j) cs[buf][d][c4 + j] = (code + j < n_codes) ? cbt[(int64_t)d * n_codes + code + j] : 0.f;
      }
    }
    cp_async_commit();
  };
  issue(0, 0);
  for (int ch = 0; ch < nch; ++ch) {
    const int buf = ch & 1;
    if (ch + 1 < nch) { issue(ch + 1, buf ^ 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
    __syncthreads();
    // scores of this thread's 4 rows x 8 codes as packed pairs (acc[i][2 j2], acc[i][2 j2 + 1]) on FFMA2 (fma.rn.f32x2: two
    // independent round-to-nearest FMAs per issue slot, the same d order -> bit-identical to the scalar fmaf chain): the scalar
    // version was issue-bound (ncu: issue 73 %, FMA pipe 51 %), the packed one leaves the slots to the LDS.128 and the argmax
    unsigned long long acc2[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc2[i][j] = 0ull;
#pragma unroll
    for (int d = 0; d < VQ_DIM; ++d) {
      const ulonglong2 c0 = *reinterpret_cast<const ulonglong2*>(&cs[buf][d][tx * 4]);
      const ulonglong2 c1 = *reinterpret_cast<const ulonglong2*>(&cs[buf][d][64 + tx * 4]);
      const unsigned long long cv2[4] = {c0.x, c0.y, c1.x, c1.y};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        unsigned long long xd;
        asm("mov.b64 %0, {%1, %1};" : "=l"(xd) : "f"(xr[i][d]));
#pragma unroll
        for (int j = 0; j < 4; ++j) asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc2[i][j]) : "l"(xd), "l"(cv2[j]));
      }
    }
    float acc[4][8];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        acc[i][2 * j] = __uint_as_float((uint32_t)acc2[i][j]);
        acc[i][2 * j + 1] = __uint_as_float((uint32_t)(acc2[i][j] >> 32));
      }
    const int base = ch * VQ_CH;
    if (base + VQ_CH <= n_codes) {
      // whole chunk valid: one max tree per row; the (rare: ~ln(#chunks) times per row) improvement then looks up the FIRST code
      // that attains it -- j ascending is code ascending, so this is the same winner as a strict-> scan in code order
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float m = fmaxf(fmaxf(fmaxf(acc[i][0], acc[i][1]), fmaxf(acc[i][2], acc[i][3])),
                              fmaxf(fmaxf(acc[i][4], acc[i][5]), fmaxf(acc[i][6], acc[i][7])));
        if (m > best[i]) {
          best[i] = m;
          int jj = 7;
#pragma unroll
          for (int j = 6; j >= 0; --j)
            if (acc[i][j] == m) jj = j;
          besti[i] = base + (jj / 4) * 64 + tx * 4 + (jj % 4);
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int code = base + (j / 4) * 64 + tx * 4 + (j % 4);
        if (code < n_codes) {
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (acc[i][j] > best[i]) { best[i] = acc[i][j]; besti[i] = code; }   // strict >: first maximum wins
        }
      }
    }
    __syncthreads();
  }
  // ---- reduce across the 16 tx threads of each row (lowest index wins ties, as torch.argmax)
#pragma unroll
  for (int i = 0; i < 4; ++i) { red_v[ty * 4 + i][tx] = best[i]; red_i[ty * 4 + i][tx] = besti[i]; }
  __syncthreads();
  if (tid < VQ_TM) {
    const int64_t row = r0 + tid;
    if (row < R) {
      float bv = red_v[tid][0]; int bi = red_i[tid][0];
      for (int t = 1; t < 16; ++t) {
        float v = red_v[tid][t]; int ii = red_i[tid][t];
        if (v > bv || (v == bv && ii < bi)) { bv = v; bi = ii; }
      }
      ids[row] = (int64_t)bi;
      if (outs_q) {
        // gather + final_layer_norm3 (affine LayerNorm over code_dim = 16, eps 1e-6)
        float c[VQ_DIM];
        float mean = 0.f;
#pragma unroll
        for (int d = 0; d < VQ_DIM; ++d) { c[d] = codebook[(int64_t)bi * VQ_DIM + d]; mean += c[d]; }
        mean *= (1.0f / VQ_DIM);
        float var = 0.f;
#pragma unroll
        for (int d = 0; d < VQ_DIM; ++d) { float t = c[d] - mean; var += t * t; }
        const float rstd = rsqrtf(var * (1.0f / VQ_DIM) + 1e-6f);
#pragma unroll
        for (int d = 0; d < VQ_DIM; ++d) outs_q[row * VQ_DIM + d] = (c[d] - mean) * rstd * ln_w[d] + ln_b[d];
      }
    }
  }
}

int launch_vq(const float* z, int64_t R, int Q, const float* w_in, const float* b_in, const float* codebook,
              const float* codebook_t, int n_codes, int code_dim, const float* ln_w, const float* ln_b,
              int64_t* ids, float* outs_q, cudaStream_t s) {
  STK_CHECK(z && w_in && b_in && codebook && codebook_t && ids && R > 0, -1, "vq: bad arguments");
  STK_CHECK(code_dim == VQ_DIM, -2, "vq: code_dim must be 16");
  STK_CHECK(Q % 4 == 0 && n_codes % 4 == 0, -2, "vq: Q and codebook size must be multiples of 4");
  STK_CHECK(outs_q == nullptr || (ln_w && ln_b), -1, "vq: LayerNorm parameters missing");
  dim3 grid((unsigned)((R + VQ_TM - 1) / VQ_TM));
  vq_kernel<<<grid, 256, 0, s>>>(z, R, Q, w_in, b_in, codebook, codebook_t, n_codes, ln_w, ln_b, ids, outs_q);
  count_launch();
  STK_CUDA(cudaGetLastError());
  return 0;
}

// An id outside [0, n_codes) is an ERROR, as `codebook[idx]` is in the reference (vector_quantize_pytorch.py:310-314 raises /
// device-asserts): the row is poisoned with NaN and counted in *bad_ids, which the engine reports (selftok_id_errors; the
// host-buffer entry points return SELFTOK_ERR_BAD_ARG).  Nothing is clamped silently.
__device__ __forceinline__ void lookup_ln3_row(int64_t row, const int64_t* __restrict__ ids, const float* __restrict__ codebook,
                                               int n_codes, int dim, const float* __restrict__ ln_w, const float* __restrict__ ln_b,
                                               float* __restrict__ outs_q, int* __restrict__ bad_ids) {
  const int64_t id = ids[row];
  if (id < 0 || id >= n_codes) {
    if (bad_ids) atomicAdd(bad_ids, 1);
    for (int d = 0; d < dim; ++d) outs_q[row * dim + d] = __int_as_float(0x7fc00000);
    return;
  }
  float mean = 0.f;
  for (int d = 0; d < dim; ++d) mean += codebook[id * dim + d];
  mean /= (float)dim;
  float var = 0.f;
  for (int d = 0; d < dim; ++d) { float t = codebook[id * dim + d] - mean; var += t * t; }
  const float rstd = rsqrtf(var / (float)dim + 1e-6f);
  for (int d = 0; d < dim; ++d) outs_q[row * dim + d] = (codebook[id * dim + d] - mean) * rstd * ln_w[d] + ln_b[d];
}
__global__ void lookup_ln3_kernel(const int64_t* __restrict__ ids, int64_t R, const float* __restrict__ codebook,
                                  int n_codes, int dim, const float* __restrict__ ln_w, const float* __restrict__ ln_b,
                                  float* __restrict__ outs_q, int* __restrict__ bad_ids) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= R) return;
  lookup_ln3_row(row, ids, codebook, n_codes, dim, ln_w, ln_b, outs_q, bad_ids);
}
// Positions >= n_tok[b] get zero rows (the padding of the reference's cut_of_k branch, rectified_flow.py:217-225): they are
// masked as keys downstream, and their K / V rows must stay finite because a masked key still enters P V with P = 0.
__global__ void lookup_ln3_prefix_kernel(const int64_t* __restrict__ ids, int B, int K, const int32_t* __restrict__ n_tok,
                                         const float* __restrict__ codebook, int n_codes, int dim, const float* __restrict__ ln_w,
                                         const float* __restrict__ ln_b, float* __restrict__ outs_q, int* __restrict__ bad_ids) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= (int64_t)B * K) return;
  if ((int)(row % K) >= n_tok[row / K]) {
    for (int d = 0; d < dim; ++d) outs_q[row * dim + d] = 0.f;
    return;
  }
  lookup_ln3_row(row, ids, codebook, n_codes, dim, ln_w, ln_b, outs_q, bad_ids);
}

int launch_lookup_ln3(const int64_t* ids, int64_t R, const float* codebook, int n_codes, int code_dim,
                      const float* ln_w, const float* ln_b, float* outs_q, int* bad_ids, cudaStream_t s) {
  STK_CHECK(ids && codebook && ln_w && ln_b && outs_q && R > 0, -1, "lookup: bad arguments");
  lookup_ln3_kernel<<<(unsigned)((R + 127) / 128), 128, 0, s>>>(ids, R, codebook, n_codes, code_dim, ln_w, ln_b, outs_q, bad_ids);
  count_launch();
  STK_CUDA(cudaGetLastError());
  return 0;
}

int launch_lookup_ln3_prefix(const int64_t* ids, int B, int K, const int32_t* n_tok, const float* codebook, int n_codes,
                             int code_dim, const float* ln_w, const float* ln_b, float* outs_q, int* bad_ids, cudaStream_t s) {
  STK_CHECK(ids && n_tok && codebook && ln_w && ln_b && outs_q && B > 0 && K > 0, -1, "lookup_prefix: bad arguments");
  const int64_t R = (int64_t)B * K;
  lookup_ln3_prefix_kernel<<<(unsigned)((R + 127) / 128), 128, 0, s>>>(ids, B, K, n_tok, codebook, n_codes, code_dim, ln_w, ln_b,
                                                                       outs_q, bad_ids);
  count_launch();
  STK_CUDA(cudaGetLastError());
  return 0;
}

// =================================================================================================== layout kernels
__global__ void patchify_kernel(const float* __restrict__ x, float* __restrict__ out, int B, int C, int Hh, int Ww, int p) {
  const int gh = Hh / p, gw = Ww / p, pk = C * p * p;
  const int64_t total = (int64_t)B * gh * gw * pk;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int kk = (int)(i % pk); int64_t t = i / pk;
    int w = (int)(t % gw); t /= gw; int h = (int)(t % gh); int b = (int)(t / gh);
    int pw = kk % p, ph = (kk / p) % p, c = kk / (p * p);
    out[i] = x[(((int64_t)b * C + c) * Hh + h * p + ph) * Ww + w * p + pw];
  }
}
int launch_patchify(const float* x, float* out, int B, int C, int Hh, int Ww, int p, cudaStream_t s) {
  STK_CHECK(x && out && Hh % p == 0 && Ww % p == 0, -1, "patchify: bad arguments");
  int64_t total = (int64_t)B * C * Hh * Ww;
  patchify_kernel<<<(unsigned)((total + 255) / 256 > 4096 ? 4096 : (total + 255) / 256), 256, 0, s>>>(x, out, B, C, Hh, Ww, p);
  count_launch();
  STK_CUDA(cudaGetLastError());
  return 0;
}

// unpatchify (sd3/mmdit.py:898-916: x.reshape(N,h,w,p,p,c) -> 'nhwpqc->nchpwq') fused with the Euler update
// x_prev = x - (a_t - a_prev) * v (sd3/rectified_flow.py:303).
// Guided sampler (rectified_flow.py:280-289): with o_u the velocity is  v = v_u + cfg_scale * (v_c - v_u)  before the update.
__global__ void unpatchify_axpy_kernel(const float* __restrict__ o, const float* __restrict__ x_in, float* __restrict__ x_out,
                                       float dt, int B, int C, int g, int p, const float* __restrict__ o_u, float cfg_scale) {
  const int Hh = g * p;
  const int64_t total = (int64_t)B * C * Hh * Hh;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int xw = (int)(i % Hh); int64_t t = i / Hh;
    int yh = (int)(t % Hh); t /= Hh; int c = (int)(t % C); int b = (int)(t / C);
    int h = yh / p, ph = yh % p, w = xw / p, pw = xw % p;
    const int64_t oi = ((int64_t)b * g * g + h * g + w) * (p * p * C) + (ph * p + pw) * C + c;
    float v = o[oi];
    if (o_u) { const float vu = o_u[oi]; v = vu + cfg_scale * (v - vu); }
    x_out[i] = x_in ? (x_in[i] - dt * v) : v;
  }
}
int launch_unpatchify_axpy(const float* o, const float* x_in, float* x_out, float dt, int B, int C, int g, int p,
                           cudaStream_t s, const float* o_u, float cfg_scale) {
  STK_CHECK(o && x_out, -1, "unpatchify: bad arguments");
  int64_t total = (int64_t)B * C * g * p * g * p;
  unpatchify_axpy_kernel<<<(unsigned)((total + 255) / 256 > 4096 ? 4096 : (total + 255) / 256), 256, 0, s>>>(o, x_in, x_out, dt, B, C, g, p, o_u, cfg_scale);
  count_launch();
  STK_CUDA(cudaGetLastError());
  return 0;
}

__global__ void transpose_kernel(const float* __restrict__ in, float* __restrict__ out, int rows, int cols) {
  __shared__ float t[32][33];
  int c = blockIdx.x * 32 + threadIdx.x, r0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += 8)
    if (r0 + j < rows && c < cols) t[j][threadIdx.x] = in[(int64_t)(r0 + j) * cols + c];
  __syncthreads();
  int r = r0 + threadIdx.x, c0 = blockIdx.x * 32;
  for (int j = threadIdx.y; j < 32; j += 8)
    if (c0 + j < cols && r < rows) out[(int64_t)(c0 + j) * rows + r] = t[threadIdx.x][j];
}
int launch_transpose(const float* in, float* out, int rows, int cols, cudaStream_t s) {
  dim3 grid((cols + 31) / 32, (rows + 31) / 32), block(32, 8);
  transpose_kernel<<<grid, block, 0, s>>>(in, out, rows, cols);
  count_launch();
  STK_CUDA(cudaGetLastError());
  return 0;
}

__global__ void split_bf16_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, int64_t n, int fp16) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    uint16_t h, l;
    split16(in[i], fp16, h, l);
    reinterpret_cast<uint16_t*>(hi)[i] = h;
    if (lo) reinterpret_cast<uint16_t*>(lo)[i] = l;
  }
}
int launch_split_bf16(const float* in, __nv_bfloat16* hi, __nv_bfloat16* lo, int64_t n, cudaStream_t s, int fp16) {
  STK_CHECK(in && hi && n > 0, -1, "split_bf16: bad arguments");
  int64_t blocks = (n + 255) / 256;
  split_bf16_kernel<<<(unsigned)(blocks > 16384 ? 16384 : blocks), 256, 0, s>>>(in, hi, lo, n, fp16);
  count_launch();
  STK_CUDA(cudaGetLastError());
  return 0;
}

__global__ void bcast_rows_kernel(const float* __restrict__ src, const float* __restrict__ add, float* __restrict__ out,
                                  int B, int64_t n) {
  const int64_t total = (int64_t)B * n;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i % n;
    out[i] = src[r] + (add ? add[r] : 0.f);
  }
}
int launch_bcast_rows(const float* src, const float* add, float* out, int B, int64_t rows, int64_t cols, cudaStream_t s) {
  int64_t n = rows * cols, blocks = ((int64_t)B * n + 255) / 256;
  bcast_rows_kernel<<<(unsigned)(blocks > 16384 ? 16384 : blocks), 256, 0, s>>>(src, add, out, B, n);
  count_launch();
  STK_CUDA(cudaGetLastError());
  return 0;
}

__global__ void crop_pos_kernel(const float* __restrict__ pos, float* __restrict__ out, int max_size, int g, int D) {
  const int top = (max_size - g) / 2, left = (max_size - g) / 2;
  const int64_t total = (int64_t)g * g * D;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int d = (int)(i % D); int64_t t = i / D; int w = (int)(t % g), h = (int)(t / g);
    out[i] = pos[((int64_t)(top + h) * max_size + left + w) * D + d];
  }
}
int launch_crop_pos(const float* pos, float* out, int max_size, int g, int D, cudaStream_t s) {
  int64_t total = (int64_t)g * g * D;
  crop_pos_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(pos, out, max_size, g, D);
  count_launch();
  STK_CUDA(cudaGetLastError());
  return 0;
}

__global__ void copy_rows_kernel(const float4* __restrict__ src, int64_t src_bs4, float4* __restrict__ dst, int64_t dst_bs4,
                                 int B, int64_t n4) {
  const int64_t total = (int64_t)B * n4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t b = i / n4, r = i % n4;
    dst[b * dst_bs4 + r] = src[b * src_bs4 + r];
  }
}
int launch_copy_rows(const float* src, int64_t src_bs, float* dst, int64_t dst_bs, int B, int64_t n_per_batch, cudaStream_t s) {
  STK_CHECK(src_bs % 4 == 0 && dst_bs % 4 == 0 && n_per_batch % 4 == 0, -1, "copy_rows: sizes must be multiples of 4");
  int64_t blocks = ((int64_t)B * n_per_batch / 4 + 255) / 256;
  copy_rows_kernel<<<(unsigned)(blocks > 16384 ? 16384 : blocks), 256, 0, s>>>(
      reinterpret_cast<const float4*>(src), src_bs / 4, reinterpret_cast<float4*>(dst), dst_bs / 4, B, n_per_batch / 4);
  count_launch();
  STK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace stk
