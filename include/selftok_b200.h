/*
 * selftok_b200.h — C ABI of the B200-native SelftokTokenizer encode / decode hot path.
 *
 * The reference (selftok-team/SelftokTokenizer) is pure Python; the boundary it exposes for this path is the
 * class API of mimogpt/infer/SelftokPipeline.py (SelftokPipeline.encoding :210-225, .decoding :227-294,
 * .decoding_with_renderer :296-322) and it has no FFI of its own.  This header is what a maintainer binds
 * (ctypes; see INTEGRATION.md) to replace the torch modules behind those three methods:
 *
 *   reference call site (file:line)                                     replaced by
 *   ------------------------------------------------------------------  ---------------------------------------
 *   SelftokPipeline.__init__  ImageTokenizer(**cfg.tokenizer.params)     selftok_create
 *       mimogpt/infer/SelftokPipeline.py:168
 *   self.model.load_state_dict(state_dict, strict=False)   :190-195      selftok_load_tensor (one call per key)
 *   RectifiedFlow(50, ...).make_schedule / DiTi_cont      :201-204       selftok_set_schedule + selftok_finalize
 *       sd3/rectified_flow.py:66-80, diti_utils.py:84-110
 *   self.model.encoder(x_0, d=None)                        :220-221      selftok_encode
 *       models_ours.py:204-251 (16 x DualBlock modules.py:310-327, VectorQuantize vector_quantize_pytorch.py:811-876)
 *   CosineSimCodebook.forward eval (einsum+argmax+gather)                selftok_vq_argmax
 *       vector_quantize_pytorch.py:525-563,580
 *   quantizer.get_output_from_indices + final_layer_norm3  :236-240      selftok_lookup
 *   flow.p_sample_loop(self.model.model, ...)              :277-282      selftok_decode
 *       sd3/rectified_flow.py:165-309 driving MMDiT.forward sd3/mmdit.py:992-1101
 *   self.model.model(y=None, encoder_hidden_states=outs_q) :310          selftok_render
 *       MMDiT_Renderer.forward sd3/mmdit.py:1511-1620
 *
 * Conventions: every function returns 0 on success and a negative selftok_status otherwise (never throws,
 * never aborts); selftok_last_error() returns a thread-local description of the last failure.  Pointers named
 * *_dev are CUDA device pointers on the handle's device, *_host are host pointers.  All launches are ordered on
 * the `stream` argument (a cudaStream_t passed as void*; NULL = legacy default stream).  One handle per
 * device; a handle may be used by one host thread at a time and has ONE set of workspaces: at most one hot-path call per
 * handle may be in flight (issue the next one on the same stream, or synchronise first).  The library allocates its weights, static
 * tables and activation workspace with cudaMalloc at finalize / first use of a batch size and frees them in
 * selftok_destroy; it never touches caller buffers other than the documented outputs.
 */
#ifndef SELFTOK_B200_H_
#define SELFTOK_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct selftok_engine* selftok_handle_t;

typedef enum selftok_status {
  SELFTOK_OK = 0,
  SELFTOK_ERR_BAD_ARG = -1,       /* null pointer, bad shape, batch <= 0 ...                       */
  SELFTOK_ERR_UNSUPPORTED = -2,   /* configuration outside what the kernels implement              */
  SELFTOK_ERR_STATE = -3,         /* call order violated (e.g. decode before finalize)             */
  SELFTOK_ERR_MISSING_TENSOR = -4,/* finalize: a checkpoint key the path needs was never loaded    */
  SELFTOK_ERR_CUDA = -5,          /* a CUDA runtime / driver call failed; see selftok_last_error() */
  SELFTOK_ERR_NO_DEVICE = -6      /* no sm_100 device visible — there is no CPU fallback            */
} selftok_status;

/* GEMM arithmetic of the decoder (MMDiT / renderer).  The encoder and VQ always run fp32 FFMA (token ids must
 * be bit-stable; SURVEY 7 hard part 2). */
typedef enum selftok_precision {
  SELFTOK_PREC_FP32_SIMT = 0,     /* fp32 FFMA GEMMs + fp32 attention (bring-up / bisecting reference)       */
  SELFTOK_PREC_BF16X3 = 1,        /* tcgen05 kind::f16: a_hi*b_hi + a_hi*b_lo + a_lo*b_hi, fp32 accumulate   */
  SELFTOK_PREC_BF16 = 2,          /* tcgen05 kind::f16 single pass (bf16 operands, fp32 accumulate)          */
  SELFTOK_PREC_FP16 = 3           /* tcgen05 kind::f16 single pass (IEEE half operands, fp32 accumulate)     */
} selftok_precision;

/* Flat view of cfg.tokenizer.params (configs/res256/256-eval.yml:48-105) after the reference's registries
 * (model_zoo.py:22-60,177-180) are resolved.  Mirrors selftoktokenizer_b200/config.py:SelftokDims. */
typedef struct selftok_config_t {
  int32_t K;                /* tokens per image (k: 512)                                        */
  int32_t latent;           /* latent side = image_size / 8 (32)                                */
  int32_t in_channels;      /* 16                                                               */
  int32_t enc_patch, enc_hidden, enc_heads, enc_depth, enc_qdim, enc_qheads, enc_pos_max;
  int32_t codebook_size, code_dim;
  int32_t dit_depth;        /* hidden = 64*depth, heads = depth (sd3/mmdit.py:708-709)          */
  int32_t dit_patch, dit_pos_max;
  int32_t renderer;         /* 0: MMDiT (50-step decode)   1: MMDiT_Renderer (one pass)        */
  int32_t context_see_xt;   /* 256-eval.yml:88                                                   */
  int32_t precision;        /* selftok_precision                                                 */
  int32_t device;           /* CUDA device ordinal                                               */
} selftok_config_t;

enum { SELFTOK_F32 = 0, SELFTOK_I64 = 1 };

/* ---- lifetime ---------------------------------------------------------------------------------------- */
int selftok_create(const selftok_config_t* cfg, selftok_handle_t* out);
int selftok_destroy(selftok_handle_t h);
const char* selftok_last_error(void);
/* ABI / build identification: "selftok_b200 <abi> sm_100a <build flags>" */
const char* selftok_version(void);

/* ---- weights: one call per checkpoint key, names exactly as in the reference state dict ------------------
 * (SURVEY 8 a14: "encoder.blocks.3.attn.qkv.weight", "model.joint_blocks.7.x_block.mlp.fc1.bias", ...).
 * `data` may be a host or a device pointer (is_device); fp32 only.  Unknown names are accepted and ignored at
 * finalize (the reference loads with strict=False). */
int selftok_load_tensor(selftok_handle_t h, const char* name, const void* data, int dtype,
                        int ndim, const int64_t* shape, int is_device);

/* ---- static sampler tables (host pointers), evaluated by the caller with the reference's own torch
 * expressions (selftoktokenizer_b200/schedule.py):  t/dt [steps] fp32, k [steps] int32 (last visible context
 * index), t_freq [steps,256] sinusoidal features of 1000*t_i, pos_freq [K,256] features of 1000+8k. */
int selftok_set_schedule(selftok_handle_t h, int steps, const float* t_host, const float* dt_host,
                         const int32_t* k_host, const float* t_freq_host, const float* pos_freq_host);

/* Packs weights (bf16 hi/lo planes for the tensor-core GEMMs), builds every input-independent table
 * (encoder adaLN [depth,K,6Q]; decoder context adaLN [L-1,K,6D]; per-step x adaLN [L,steps,6D]; cropped
 * positional embeddings) on the device, and frees staging copies. */
int selftok_finalize(selftok_handle_t h, void* stream);

/* ---- prepack cache: the finalized device state (fp32 tensors that stay fp32, 16-bit operand planes, static tables,
 * schedule) as one file.  selftok_export_packed needs a finalized handle; selftok_import_packed needs a FRESH handle
 * (selftok_create only) of the same configuration / precision and leaves it finalized -- no selftok_load_tensor,
 * selftok_set_schedule or selftok_finalize.  Replaces the per-process torch.load + load_state_dict of the fp32 checkpoint
 * (SelftokPipeline.py:188-199). */
int selftok_export_packed(selftok_handle_t h, const char* path);
int selftok_import_packed(selftok_handle_t h, const char* path);

/* ---- hot path, device buffers ---------------------------------------------------------------------------- */
/* x0_dev [B,C,latent,latent] fp32 (VAE latent after SD3LatentFormat.process_in) -> tokens_dev [B,K] int64,
 * outs_q_dev [B,K,code_dim] fp32 (may be NULL), feats_dev [B,K,enc_qdim] fp32 pre-VQ features (may be NULL). */
int selftok_encode(selftok_handle_t h, const float* x0_dev, int B, int64_t* tokens_dev, float* outs_q_dev,
                   float* feats_dev, void* stream);
/* Standalone fused VQ: z_dev [R,enc_qdim] fp32 -> ids_dev [R] int64, outs_q_dev [R,code_dim] (may be NULL). */
int selftok_vq_argmax(selftok_handle_t h, const float* z_dev, int64_t R, int64_t* ids_dev, float* outs_q_dev,
                      void* stream);
/* tokens_dev [B,K] int64 -> outs_q_dev [B,K,code_dim] fp32 (codebook gather + final_layer_norm3). */
int selftok_lookup(selftok_handle_t h, const int64_t* tokens_dev, int B, float* outs_q_dev, void* stream);
/* tokens_dev [B,K], noise_dev [B,C,latent,latent] fp32 -> x0_out_dev (same shape): `steps` Euler steps of the
 * rectified flow (steps <= the schedule's; the loop is captured in one CUDA graph per batch size).
 * x0_out_dev may alias noise_dev. */
int selftok_decode(selftok_handle_t h, const int64_t* tokens_dev, const float* noise_dev, int B, int steps,
                   float* x0_out_dev, void* stream);
/* Guided sampler (classifier-free guidance): the reference's p_sample_loop(..., uncond_scale = cfg_scale)
 * (sd3/rectified_flow.py:165-294, 280-289): per step one conditional evaluation (context rows blind to the image keys, as that
 * call site omits context_see_xt) and MMDiT.cfg_inference (sd3/mmdit.py:1117-1163: no context, integer timestep), combined as
 * v_u + cfg_scale (v_c - v_u).  selftok_set_cfg_schedule (host pointer, [steps,256] sinusoidal features of
 * floor(1000 t_i).clamp(0, 999)) must be called between selftok_set_schedule and selftok_finalize. */
int selftok_set_cfg_schedule(selftok_handle_t h, const float* t_freq_uncond_host);
int selftok_decode_cfg(selftok_handle_t h, const int64_t* tokens_dev, const float* noise_dev, int B, int steps,
                       float cfg_scale, float* x0_out_dev, void* stream);
/* One MMDiT velocity evaluation at schedule index `step` on latents x_dev (testing / bisecting entry). */
int selftok_dit_velocity(selftok_handle_t h, const int64_t* tokens_dev, const float* x_dev, int B, int step,
                         float* v_out_dev, void* stream);
/* renderer handles only: tokens_dev [B,K] -> pred_x0 [B,C,latent,latent]. */
int selftok_render(selftok_handle_t h, const int64_t* tokens_dev, int B, float* x0_out_dev, void* stream);

/* ---- decode from a token prefix: image b from its first n_b tokens (the reference's super_mask[b] = arange(K) < n_b,
 * sd3/rectified_flow.py:182,227-228; renderer: mask[b], sd3/mmdit.py:1511,1529).  At step i image b sees the context tokens
 * < min(k_i + 1, n_b); ids at positions >= n_b are never read (not range-checked, may be -1); n_b = K for every image gives
 * the result of the entry point without a prefix.  Per-image results depend only on that image and max_b n_b.
 * n_tokens_host: int32 [B] host array, 1 <= n_b <= K (read before the call returns; the host needs max n to shape launches);
 * any other value returns SELFTOK_ERR_BAD_ARG and launches nothing.
 * cfg_scale == 1: plain sampler (captured graphs keyed by batch, steps and the per-step context rows, which every
 * max n >= k_0 + 1 shares); otherwise the guided sampler with the prefix applied to its conditional branch. */
int selftok_decode_prefix(selftok_handle_t h, const int64_t* tokens_dev, const int32_t* n_tokens_host, const float* noise_dev,
                          int B, int steps, float cfg_scale, float* x0_out_dev, void* stream);
int selftok_render_prefix(selftok_handle_t h, const int64_t* tokens_dev, const int32_t* n_tokens_host, int B,
                          float* x0_out_dev, void* stream);
/* testing / bisecting entry, like selftok_dit_velocity */
int selftok_dit_velocity_prefix(selftok_handle_t h, const int64_t* tokens_dev, const int32_t* n_tokens_host, const float* x_dev,
                                int B, int step, float* v_out_dev, void* stream);

/* ---- hot path, host buffers (what SelftokPipeline's numpy-in / tensor-out API maps to; H2D and D2H copies are
 * inside the call, on `stream`, followed by a stream synchronize) --------------------------------------------- */
int selftok_encode_host(selftok_handle_t h, const float* x0_host, int B, int64_t* tokens_host, void* stream);
int selftok_decode_host(selftok_handle_t h, const int64_t* tokens_host, const float* noise_host, int B, int steps,
                        float* x0_out_host, void* stream);
int selftok_render_host(selftok_handle_t h, const int64_t* tokens_host, int B, float* x0_out_host, void* stream);

/* Token ids outside [0, codebook_size) are an error, as `codebook[idx]` is in the reference: the lookup poisons the row
 * with NaN (so everything derived from it is NaN) and counts it.  The *_host entry points return SELFTOK_ERR_BAD_ARG;
 * after a device-buffer call, selftok_id_errors synchronises `stream`, returns the count since the last query and
 * resets it (< 0: CUDA error). */
int64_t selftok_id_errors(selftok_handle_t h, void* stream);

/* ---- SD3 VAE on the device (SURVEY 8f rank 1): replaces `self.vae.decode(pred_x0_out)` of SelftokPipeline.decoding /
 * decoding_with_renderer (SelftokPipeline.py:288,316) and `self.vae.encode(images)[0].mode()` of SelftokPipeline.encoding (:215);
 * architecture: sd3/sd3_impls.py:314-444.  Weights are loaded under the in-tree SDVAE key names ("decoder.conv_in.weight",
 * "decoder.up.3.block.0.norm1.bias", "encoder.down.0.downsample.conv.weight", ...), fp32, one call per tensor; either half may
 * be omitted (the matching entry point then returns SELFTOK_ERR_MISSING_TENSOR).
 * selftok_vae_decode: z_dev [B,16,h,w] fp32 in VAE latent space (after SD3LatentFormat.process_out), h = w in {8,16,32,64}
 * -> out_dev [B,3,8h,8w] fp32; norm_ip != 0 applies the pipeline's clamp to [-1,1] + rescale to [0,1]. */
typedef struct selftok_vae* selftok_vae_t;
int selftok_vae_create(int ch /* 128 */, int device, selftok_vae_t* out);
int selftok_vae_destroy(selftok_vae_t v);
int selftok_vae_load_tensor(selftok_vae_t v, const char* name, const void* data, int ndim, const int64_t* shape, int is_device);
int selftok_vae_finalize(selftok_vae_t v, void* stream);
int selftok_vae_decode(selftok_vae_t v, const float* z_dev, int B, int h, int w, float* out_dev, int norm_ip, void* stream);
/* images_dev [B,3,H,W] fp32 in [-1,1], H = W in {128,256,512} -> mean_out_dev [B,16,H/8,W/8] fp32 (the distribution's mode, VAE
 * latent space: apply SD3LatentFormat.process_in afterwards); logvar_out_dev (same shape) may be NULL. */
int selftok_vae_encode(selftok_vae_t v, const float* images_dev, int B, int H, int W, float* mean_out_dev, float* logvar_out_dev,
                       void* stream);
int64_t selftok_vae_device_bytes(selftok_vae_t v);

/* ---- activation workspace.  By default the library allocates ONE device block per operation class (0 = encode,
 * 1 = decode / render / velocity) with cudaMalloc at the first call of a batch size.  A caller that owns device memory
 * (PyTorch's caching allocator) can size it with selftok_workspace_bytes and hand it over with selftok_set_workspace; the
 * library then allocates nothing at call time. */
int64_t selftok_workspace_bytes(selftok_handle_t h, int B, int op);
int selftok_set_workspace(selftok_handle_t h, int op, void* ws_dev, size_t bytes);

/* ---- introspection ----------------------------------------------------------------------------------------- */
/* Number of kernel launches issued (or replayed from a graph) by the last hot-path call on this handle. */
int64_t selftok_last_launch_count(selftok_handle_t h);
/* Device bytes currently held by the handle (weights + tables + workspaces). */
int64_t selftok_device_bytes(selftok_handle_t h);
/* Enable (1) / disable (0) CUDA-graph capture of the decode loop (default 1). */
int selftok_set_use_graph(selftok_handle_t h, int enable);

/* Per-kernel-class device timing: with profiling on (and graphs off) every launch of a hot-path call is bracketed
 * by CUDA events on its stream.  selftok_get_profile synchronises, writes the summed milliseconds and launch counts
 * of the 8 classes (0 tcgen05 GEMM, 1 attention, 2 LayerNorm+modulate, 3 fp32 FFMA linear, 4 VQ, 5 other) and resets. */
int selftok_set_profile(selftok_handle_t h, int enable);
int selftok_get_profile(selftok_handle_t h, double* ms_out /*[8]*/, int64_t* count_out /*[8]*/);

/* ---- kernel-level entry points (parity tests and micro-benchmarks call these through the same ABI) ---------- */
/* y[M,N] = act(A[M,K] W[N,K]^T + bias) (+ epilogue), fp32 FFMA.  act: 0 none, 1 gelu-tanh, 2 silu. */
int selftok_k_linear_f32(const float* A_dev, const float* W_dev, const float* bias_dev, float* out_dev,
                         int64_t M, int N, int K, int act, void* stream);
/* Same product on the tcgen05 path: A/W given as fp32, converted to 16-bit planes internally
 * (nsplit 3: bf16 hi+lo split, 1: bf16, 0: IEEE half single pass). */
int selftok_k_linear_tc(const float* A_dev, const float* W_dev, const float* bias_dev, float* out_dev,
                        int64_t M, int N, int K, int nsplit, void* stream);
/* Process-wide choice of the tcgen05 GEMM variant: 2 = cta_group::2 SM-pair kernel (default), 1 = single-CTA kernel. */
int selftok_k_set_gemm_ctas(int n);
/* out = LN(x) * (1 + scale[m % period]) + shift[m % period], rows of D; eps 1e-6, no affine. */
int selftok_k_ln_mod_f32(const float* x_dev, const float* shift_dev, const float* scale_dev, int64_t ld_mod,
                         int period, float* out_dev, int64_t M, int D, void* stream);
/* softmax(Q K^T / sqrt(hd)) V, fp32; q [B,Sq,H*hd], k/v two concatenated segments [B,S1,H*hd] + [B,S2,H*hd]
 * (S2 may be 0), each with its own row stride in floats. */
int selftok_k_attention_f32(const float* q_dev, int64_t q_ld, const float* k1_dev, const float* v1_dev, int64_t kv1_ld,
                            int S1, const float* k2_dev, const float* v2_dev, int64_t kv2_ld, int S2,
                            float* out_dev, int64_t out_ld, int B, int Sq, int H, int hd, void* stream);
/* Tensor-core (bf16x3 / bf16) attention over a packed qkv buffer [B,S,3,H,64]; ctx_rows = number of leading rows
 * whose queries may only see the first `ctx_keys` keys (renderer rule; pass 0 for plain dense attention).
 * nsplit 3: bf16 hi+lo split, 1: bf16, 0: IEEE half single pass (mma.sync kernel); 10 / 11: the tcgen05 + TMEM kernel
 * with IEEE half / bf16 operands. */
int selftok_k_attention_tc(const float* qkv_dev, float* out_dev, int B, int S, int H, int nsplit,
                           int ctx_rows, int ctx_keys, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SELFTOK_B200_H_ */
