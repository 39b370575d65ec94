// Launch wrappers shared by engine.cu and the kernel-level C-ABI entry points.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace stk {

// Epilogue description common to the fp32-FFMA and the tcgen05 GEMMs:  y = act(A W^T + bias)
//   mode EPI_STORE : out[orow, n] = y (+ addtab[(m % add_period) * add_ld + n])
//   mode EPI_RESID : out[orow, n] = resid[orow, n] + gate[(m % gate_period) * gate_ld + n] * y   (gate NULL -> 1)
//   mode EPI_SPLIT : out_hi/out_lo[orow, n] = bf16 split of y            (tensor-core A-operand planes)
// Row remap (joint attention buffer):  orow = (m / rpb_in) * rpb_out + row_off + m % rpb_in   (rpb_in == 0: orow = m)
enum EpiMode { EPI_STORE = 0, EPI_RESID = 1, EPI_SPLIT = 2 };
struct Epilogue {
  int mode = EPI_STORE;
  int act = 0;
  const float* bias = nullptr;
  float* out = nullptr;
  int64_t ldo = 0;
  const float* resid = nullptr;          // EPI_RESID (may alias out)
  const float* gate = nullptr;
  int64_t gate_ld = 0;
  int gate_period = 1;
  const float* addtab = nullptr;         // EPI_STORE
  int64_t add_ld = 0;
  int add_period = 1;
  __nv_bfloat16* out_hi = nullptr;       // EPI_SPLIT
  __nv_bfloat16* out_lo = nullptr;       // may be NULL (single-pass bf16)
  int rpb_in = 0, rpb_out = 0, row_off = 0;
  int fp16 = 0;                          // EPI_SPLIT: planes hold IEEE half (single-pass fp16 mode) instead of bf16
};

// ---- fp32 FFMA kernels (kernels_simt.cu) ---------------------------------------------------------------------
int launch_linear_f32(const float* A, int64_t lda, const float* W, int64_t ldw, int64_t M, int N, int K,
                      const Epilogue& ep, cudaStream_t s);
// LN (no affine, eps) + modulate; writes fp32 and/or bf16 planes.  shift/scale NULL -> plain LN.
int launch_ln_mod(const float* x, int64_t ldx, const float* shift, const float* scale, int64_t ld_mod, int period,
                  float* out_f32, __nv_bfloat16* out_hi, __nv_bfloat16* out_lo, int64_t ldo, int64_t M, int D,
                  float eps, cudaStream_t s, int fp16 = 0);
// Two LN + modulate problems (the context- and the image-row pass of one MMDiT layer stage) in ONE launch, 16-bit plane
// output (IEEE half when fp16, else bf16 hi [+ lo]).  period > 1: rows are [image][position] with a per-position table row
// (M must be a multiple of period); period <= 1: one table row for all rows.
struct LnProblem {
  const float* x = nullptr;          // [M, D] fp32, contiguous rows
  const float* shift = nullptr;
  const float* scale = nullptr;
  int64_t ld_mod = 0;
  int period = 1;
  __nv_bfloat16* out_hi = nullptr;
  __nv_bfloat16* out_lo = nullptr;
  int64_t M = 0;
  int imgs = 0;                      // filled by the launcher
};
int launch_ln_mod_pair(const LnProblem* probs, int n, int D, float eps, cudaStream_t s, int fp16);
// Attention output routing: query rows [0,split) of every image go to the compact buffer A ([B*split, ld]),
// rows [split,Sq) to buffer B ([B*(Sq-split), ld]).  split == Sq -> everything in A.  Each buffer is fp32 and/or
// bf16 hi(/lo) planes (NULL pointers are skipped).
struct AttnOut {
  float* f32_a = nullptr; __nv_bfloat16* hi_a = nullptr; __nv_bfloat16* lo_a = nullptr;
  float* f32_b = nullptr; __nv_bfloat16* hi_b = nullptr; __nv_bfloat16* lo_b = nullptr;
  int split = 0;
  int64_t ld = 0;
  int fp16 = 0;                          // planes hold IEEE half instead of bf16
};
// softmax(q k^T / sqrt(hd)) v in fp32.  q rows: q + b*q_bs + s*q_ld + h*hd; keys = segment 1 (S1 rows) followed by
// segment 2 (S2 rows).  Rows < ctx_rows only see keys < ctx_keys (renderer rule); ctx_rows = 0 -> dense.
// n_ctx != NULL: the context-prefix window of launch_attention_tc5 over the key index (kc = context keys).
int launch_attention_f32(const float* q, int64_t q_ld, int64_t q_bs, const float* k1, const float* v1, int64_t kv1_ld,
                         int64_t kv1_bs, int S1, const float* k2, const float* v2, int64_t kv2_ld, int64_t kv2_bs,
                         int S2, const AttnOut& out, int B, int Sq, int H, int hd, int ctx_rows, int ctx_keys,
                         cudaStream_t s, const int32_t* n_ctx = nullptr, int kc = 0);
// Fused VQ: project_in + l2norm + argmax over the codebook + gather + final_layer_norm3.
int launch_vq(const float* z, int64_t R, int Q, const float* w_in, const float* b_in, const float* codebook,
              const float* codebook_t, int n_codes, int code_dim, const float* ln_w, const float* ln_b,
              int64_t* ids, float* outs_q, cudaStream_t s);
// ids outside [0, n_codes): row poisoned with NaN and counted in *bad_ids (may be NULL)
int launch_lookup_ln3(const int64_t* ids, int64_t R, const float* codebook, int n_codes, int code_dim,
                      const float* ln_w, const float* ln_b, float* outs_q, int* bad_ids, cudaStream_t s);
// the same over B images of K ids, image b from its first n_tok[b] ids only (device array [B]): later positions get zero
// rows and their ids are never read
int launch_lookup_ln3_prefix(const int64_t* ids, int B, int K, const int32_t* n_tok, const float* codebook, int n_codes,
                             int code_dim, const float* ln_w, const float* ln_b, float* outs_q, int* bad_ids, cudaStream_t s);
// [B,C,Hh,Ww] latents -> [B*(Hh/p)*(Ww/p), C*p*p] patch rows ((c,ph,pw) fastest-last, Conv2d weight order)
int launch_patchify(const float* x, float* out, int B, int C, int Hh, int Ww, int p, cudaStream_t s);
// x_lat[b,c,h*p+ph,w*p+pw] = x_in[...] - dt * o[b, h*g+w, (ph*p+pw)*C + c]   (unpatchify + Euler; dt = -1 & x_in NULL: plain unpatchify)
// o_u != NULL (guided sampler): v = o_u + cfg_scale * (o - o_u) first
int launch_unpatchify_axpy(const float* o, const float* x_in, float* x_out, float dt, int B, int C, int g, int p,
                           cudaStream_t s, const float* o_u = nullptr, float cfg_scale = 1.f);
int launch_transpose(const float* in, float* out, int rows, int cols, cudaStream_t s);
int launch_split_bf16(const float* in, __nv_bfloat16* hi, __nv_bfloat16* lo, int64_t n, cudaStream_t s, int fp16 = 0);
// out[b, r, :] = src[r, :] for b in 0..B-1 (broadcast rows), optionally + add[r,:]
int launch_bcast_rows(const float* src, const float* add, float* out, int B, int64_t rows, int64_t cols, cudaStream_t s);
// centre crop of a [max,max,D] positional grid to [g,g,D]
int launch_crop_pos(const float* pos, float* out, int max_size, int g, int D, cudaStream_t s);
int launch_copy_rows(const float* src, int64_t src_bs, float* dst, int64_t dst_bs, int B, int64_t n_per_batch, cudaStream_t s);

// ---- tcgen05 GEMM (gemm_tc.cu) --------------------------------------------------------------------------------
// A planes [M,K] bf16 row-major (lo NULL iff nsplit == 1), W planes [N,K] bf16 row-major.
// fp16 != 0: operands are IEEE half planes (nsplit must be 1).
int launch_gemm_tc(const __nv_bfloat16* A_hi, const __nv_bfloat16* A_lo, const __nv_bfloat16* W_hi,
                   const __nv_bfloat16* W_lo, int64_t M, int N, int K, int nsplit, const Epilogue& ep,
                   cudaStream_t s, int fp16 = 0);
struct TcProblem {
  const __nv_bfloat16* A_hi; const __nv_bfloat16* A_lo; const __nv_bfloat16* W_hi; const __nv_bfloat16* W_lo;
  int64_t M; int N; int K;
  Epilogue ep;
  // conv_C > 0: implicit-GEMM 3x3 convolution (stride 1, pad 1): A planes are NHWC activations [M / (H W), H, W, C], W planes
  // [N, 9 C] with K index = (ky * 3 + kx) * C + c, M = output pixels, K = 9 C.  conv_stride == 2: A planes are the four
  // polyphase components of the input [images * 4, H_out, W_out, C] (pad right / bottom), conv_H / conv_W = output dims
  int conv_C = 0, conv_H = 0, conv_W = 0, conv_stride = 1;
};
// one launch for one or two independent problems of the same operand type (cta_group::2 kernel)
int launch_gemm_tc_grouped(const TcProblem* probs, int n, int nsplit, cudaStream_t s, int fp16 = 0);
int gemm_tc_init();   // resolves cuTensorMapEncodeTiled, sets smem attributes; idempotent
void gemm_tc_set_ctas(int n);   // 2 (default): cta_group::2 pair kernel; 1: single-CTA kernel

// ---- tensor-core attention -----------------------------------------------------------------------------------
// qkv planes: packed 16-bit [B,S,3,H,64] (hi, and lo for the split mode), written by the QKV GEMM epilogue
// tcgen05 / TMEM attention (attn_tc5.cu): single-pass 16-bit operands (fp16 != 0: IEEE half, else bf16), or -- with the lo
// planes given -- the fp32-faithful split-bf16 mode (three MMAs per product, P split in registers)
// n_ctx != NULL (decode from a token prefix): image b additionally ignores the context keys [min(kc, n_ctx[b]), kc), kc = the
// context rows of the joint sequence (ctx_keys must be 0 or kc); n_ctx is a device array [B], every entry >= 1
int launch_attention_tc5(const __nv_bfloat16* qkv16, int B, int S, int H, int ctx_rows, int ctx_keys, const AttnOut& out,
                         cudaStream_t s, int fp16, const __nv_bfloat16* qkv_lo = nullptr, const int32_t* n_ctx = nullptr,
                         int kc = 0);

}  // namespace stk
