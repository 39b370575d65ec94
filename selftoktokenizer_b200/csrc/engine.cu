// selftok_b200 engine: the C ABI of include/selftok_b200.h.
//
// Host-side orchestration of the encode / decode hot path of mimogpt/infer/SelftokPipeline.py — weights under the
// reference's checkpoint key names, every input-independent table built once at finalize, one workspace per batch
// size, and the 50-step sampler captured in one CUDA graph.  All arithmetic is in the kernels of kernels_simt.cu
// (fp32 FFMA: encoder, VQ, tables), gemm_tc.cu (tcgen05 GEMMs of the MMDiT) and attn_tc5.cu (tcgen05 joint attention).
#include "../../include/selftok_b200.h"
#include "common.cuh"
#include "kernels.h"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <map>
#include <string>
#include <unordered_map>
#include <vector>

namespace stk {
static thread_local std::string g_error;
thread_local int64_t g_launch_count = 0;
void set_error(const std::string& msg) { g_error = msg; }
}  // namespace stk

using namespace stk;
typedef __nv_bfloat16 bf16;

struct Tensor {
  float* d = nullptr;
  std::vector<int64_t> shape;
  int64_t numel = 0;
};
struct WPack {
  bf16* hi = nullptr;
  bf16* lo = nullptr;
};

// Bump allocator over ONE block of device memory: the activation workspaces are carved from it.  The block is either the
// caller's (selftok_set_workspace: PyTorch keeps ownership, nothing is allocated behind its caching allocator) or one
// cudaMalloc of exactly selftok_workspace_bytes.  dry = sizing pass only.
struct Arena {
  char* base = nullptr;
  size_t cap = 0, off = 0;
  bool dry = false;
  template <typename T> int take(T** p, int64_t n) {
    const size_t bytes = (sizeof(T) * (size_t)(n > 0 ? n : 1) + 255) & ~(size_t)255;
    if (!dry) {
      if (off + bytes > cap) { set_error("workspace too small"); return SELFTOK_ERR_BAD_ARG; }
      *p = reinterpret_cast<T*>(base + off);
    }
    off += bytes;
    return 0;
  }
};

struct DecodeWs {       // activation workspace of the MMDiT for one batch size
  int B = 0;
  int64_t* tokens = nullptr;
  float *outs_q = nullptr, *x_lat = nullptr, *patch = nullptr, *ctx0 = nullptr, *ctx = nullptr, *x = nullptr;
  float *qkv = nullptr, *o_final = nullptr;      // qkv: fp32 joint buffer (fp32 mode only)
  float* o_final_u = nullptr;                    // final-layer output of the unconditional branch (guided sampler)
  // split-bf16 operand planes of the two skinny fp32-faithful GEMMs of every evaluation (patch embedding K = 64, final layer N = 64)
  bf16 *patch_hi = nullptr, *patch_lo = nullptr, *fin_hi = nullptr, *fin_lo = nullptr;
  bf16 *qkv_hi = nullptr, *qkv_lo = nullptr;     // joint q/k/v as 16-bit planes [B,S,3,H,64] (tensor-core modes)
  // fp32 mode activations
  float *a_c = nullptr, *a_x = nullptr, *attn_c = nullptr, *attn_x = nullptr, *h_c = nullptr, *h_x = nullptr;
  // tensor-core mode activations (bf16 planes)
  bf16 *a_c_hi = nullptr, *a_c_lo = nullptr, *a_x_hi = nullptr, *a_x_lo = nullptr;
  bf16 *attn_c_hi = nullptr, *attn_c_lo = nullptr, *attn_x_hi = nullptr, *attn_x_lo = nullptr;
  bf16 *h_c_hi = nullptr, *h_c_lo = nullptr, *h_x_hi = nullptr, *h_x_lo = nullptr;
  void* own = nullptr;                           // the library's own block (NULL when the caller's workspace is in use)
  size_t own_bytes = 0;
};
struct EncodeWs {
  int B = 0;
  float *x0 = nullptr, *patch = nullptr, *x = nullptr, *q = nullptr, *xn = nullptr, *qn = nullptr, *xqkv = nullptr,
        *xkv = nullptr, *qqkv = nullptr, *xattn = nullptr, *qattn = nullptr, *xh = nullptr, *qh = nullptr, *outs_q = nullptr;
  int64_t* tokens = nullptr;
  void* own = nullptr;
  size_t own_bytes = 0;
};

struct selftok_engine {
  selftok_config_t cfg;
  int D = 0, H = 0, Nimg = 0, Nenc = 0;
  bool finalized = false;
  bool use_graph = true;
  std::unordered_map<std::string, Tensor> w;
  std::unordered_map<std::string, WPack> wp;
  std::vector<void*> allocs;            // tables + packed weights
  int64_t bytes = 0;
  // schedule
  int steps = 0;
  std::vector<float> t, dt;
  std::vector<int> k;
  float *t_freq = nullptr, *pos_freq = nullptr;
  float* t_freq_u = nullptr;            // classifier-free guidance: features of floor(1000 t).clamp(0, 999) (MMDiT.cfg_inference)
  // tables
  float *enc_mod = nullptr, *enc_pos = nullptr, *cbt = nullptr;
  float *ctx_mod = nullptr, *x_mod = nullptr, *ctx_last_mod = nullptr, *final_mod = nullptr, *dit_pos = nullptr;
  float *x_mod_u = nullptr, *final_mod_u = nullptr;     // unconditional branch of the guided sampler (optional)
  float* rend_x0 = nullptr;
  bool has_cfg = false;                 // unconditional-branch tables built (selftok_set_cfg_schedule before finalize)
  int* bad_ids = nullptr;               // device counter of out-of-range token ids seen by the lookup kernel
  DecodeWs dws;
  EncodeWs ews;
  void* user_ws[2] = {nullptr, nullptr};          // caller-provided workspaces (selftok_set_workspace): [0] encode, [1] decode / render
  size_t user_ws_bytes[2] = {0, 0};
  std::map<std::pair<int, int>, std::pair<cudaGraphExec_t, int64_t>> graphs;   // (B, steps) -> (exec, launches)
  std::map<int, std::pair<cudaGraphExec_t, int64_t>> enc_graphs;               // encode, B -> (exec, launches)
  // decode from a token prefix: per-image visible-token counts at a fixed device address (captured graphs read it), and the
  // graphs keyed by (B, steps, per-step context rows), least recently used dropped beyond kPrefixGraphs
  int32_t* n_dev = nullptr;
  int n_cap = 0;
  struct PrefixGraph { cudaGraphExec_t exec; int64_t launches; uint64_t used; };
  std::map<std::vector<int>, PrefixGraph> prefix_graphs;
  uint64_t prefix_tick = 0;
  int64_t last_launches = 0;
  // optional per-kernel-class timing (CUDA events around every launch; only meaningful with graphs disabled)
  bool prof_on = false;
  std::vector<cudaEvent_t> prof_ev;     // pairs (start, stop)
  std::vector<int> prof_cat;
};

enum ProfCat { PC_GEMM_TC = 0, PC_ATTN = 1, PC_LN = 2, PC_LINEAR_F32 = 3, PC_VQ = 4, PC_OTHER = 5, PC_COUNT = 8 };
struct ProfScope {
  selftok_engine* e; cudaStream_t s; bool on;
  ProfScope(selftok_engine* e_, int cat, cudaStream_t s_) : e(e_), s(s_), on(e_->prof_on) {
    if (!on) return;
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    e->prof_ev.push_back(a); e->prof_ev.push_back(b); e->prof_cat.push_back(cat);
    cudaEventRecord(a, s);
  }
  void end() { if (on) cudaEventRecord(e->prof_ev.back(), s); }
};
#define PROF(cat, expr)                         \
  do {                                          \
    ProfScope _ps(e, (cat), s);                 \
    int _st = (expr);                           \
    _ps.end();                                  \
    if (_st != 0) return _st;                   \
  } while (0)

static int dmalloc(selftok_engine* e, std::vector<void*>& pool, void** p, size_t bytes) {
  STK_CUDA(cudaMalloc(p, bytes ? bytes : 16));
  pool.push_back(*p);
  e->bytes += (int64_t)bytes;
  return 0;
}
template <typename T>
static int dalloc(selftok_engine* e, std::vector<void*>& pool, T** p, int64_t n) {
  return dmalloc(e, pool, reinterpret_cast<void**>(p), sizeof(T) * (size_t)n);
}
static void free_pool(selftok_engine* e, std::vector<void*>& pool) {
  for (void* p : pool) cudaFree(p);
  pool.clear();
}

static const Tensor* find(selftok_engine* e, const std::string& name) {
  auto it = e->w.find(name);
  return it == e->w.end() ? nullptr : &it->second;
}
#define GETW(var, name)                                                             \
  const Tensor* var = find(e, (name));                                              \
  if (!var) {                                                                       \
    set_error(std::string("checkpoint key not loaded: ") + (name));                 \
    return SELFTOK_ERR_MISSING_TENSOR;                                              \
  }

static bool tc_mode(const selftok_engine* e) { return e->cfg.precision != SELFTOK_PREC_FP32_SIMT; }
static int nsplit(const selftok_engine* e) { return e->cfg.precision == SELFTOK_PREC_BF16X3 ? 3 : 1; }
static int is_fp16(const selftok_engine* e) { return e->cfg.precision == SELFTOK_PREC_FP16 ? 1 : 0; }

// y = act(A W^T + b) with weights looked up by checkpoint prefix (fp32 FFMA path)
static int lin32(selftok_engine* e, const std::string& prefix, const float* A, int64_t lda, int64_t M, Epilogue ep,
                 cudaStream_t s) {
  GETW(W, prefix + ".weight");
  GETW(Bv, prefix + ".bias");
  int N = (int)W->shape[0];
  int K = (int)(W->numel / W->shape[0]);
  ep.bias = Bv->d;
  if (ep.ldo == 0) ep.ldo = N;
  PROF(PC_LINEAR_F32, launch_linear_f32(A, lda, W->d, K, M, N, K, ep, s));
  return 0;
}
// tcgen05 path: A given as bf16 planes
static int lintc(selftok_engine* e, const std::string& prefix, const bf16* A_hi, const bf16* A_lo, int64_t M,
                 Epilogue ep, cudaStream_t s) {
  GETW(W, prefix + ".weight");
  GETW(Bv, prefix + ".bias");
  auto it = e->wp.find(prefix + ".weight");
  STK_CHECK(it != e->wp.end(), SELFTOK_ERR_STATE, "packed weight missing");
  int N = (int)W->shape[0];
  int K = (int)(W->numel / W->shape[0]);
  ep.bias = Bv->d;
  if (ep.ldo == 0) ep.ldo = N;
  ep.fp16 = is_fp16(e);
  PROF(PC_GEMM_TC, launch_gemm_tc(A_hi, A_lo, it->second.hi, it->second.lo, M, N, K, nsplit(e), ep, s, is_fp16(e)));
  return 0;
}

// tcgen05 problem descriptor for a checkpoint linear (weights already packed at finalize)
static int tc_problem(selftok_engine* e, const std::string& prefix, const bf16* A_hi, const bf16* A_lo, int64_t M, Epilogue ep,
                      TcProblem* out) {
  GETW(W, prefix + ".weight");
  GETW(Bv, prefix + ".bias");
  auto it = e->wp.find(prefix + ".weight");
  STK_CHECK(it != e->wp.end(), SELFTOK_ERR_STATE, "packed weight missing");
  const int N = (int)W->shape[0];
  const int K = (int)(W->numel / W->shape[0]);
  ep.bias = Bv->d;
  if (ep.ldo == 0) ep.ldo = N;
  ep.fp16 = is_fp16(e);
  *out = TcProblem{A_hi, A_lo, it->second.hi, it->second.lo, M, N, K, ep};
  return 0;
}
// the context- and image-stream GEMM of a layer in ONE launch (n == 1: image stream only)
static int lintc2(selftok_engine* e, const TcProblem* probs, int n, cudaStream_t s) {
  PROF(PC_GEMM_TC, launch_gemm_tc_grouped(probs, n, nsplit(e), s, is_fp16(e)));
  return 0;
}

// ------------------------------------------------------------------------------------------------ C ABI: lifetime
extern "C" __attribute__((visibility("default"))) const char* selftok_last_error(void) { return g_error.c_str(); }
extern "C" __attribute__((visibility("default"))) const char* selftok_version(void) { return "selftok_b200 abi1 sm_100a (fp32-ffma + tcgen05 kind::f16)"; }

extern "C" __attribute__((visibility("default"))) int selftok_create(const selftok_config_t* cfg, selftok_handle_t* out) {
  STK_CHECK(cfg && out, SELFTOK_ERR_BAD_ARG, "selftok_create: null argument");
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev <= 0) {
    set_error("no CUDA device visible: selftok_b200 has no CPU fallback");
    return SELFTOK_ERR_NO_DEVICE;
  }
  STK_CHECK(cfg->device >= 0 && cfg->device < ndev, SELFTOK_ERR_BAD_ARG, "bad device ordinal");
  cudaDeviceProp prop;
  STK_CUDA(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10) {
    set_error("device is not sm_100 (Blackwell B200): kernels are built for sm_100a only");
    return SELFTOK_ERR_NO_DEVICE;
  }
  STK_CHECK(cfg->K > 0 && cfg->latent > 0 && cfg->dit_depth > 0 && cfg->enc_depth > 0, SELFTOK_ERR_BAD_ARG, "bad dims");
  STK_CHECK(cfg->code_dim == 16, SELFTOK_ERR_UNSUPPORTED, "code_dim must be 16");
  STK_CHECK(cfg->enc_hidden % cfg->enc_heads == 0 && cfg->enc_qdim % cfg->enc_qheads == 0, SELFTOK_ERR_BAD_ARG, "bad heads");
  int hd1 = cfg->enc_hidden / cfg->enc_heads, hd2 = cfg->enc_qdim / cfg->enc_qheads;
  STK_CHECK((hd1 == 16 || hd1 == 32 || hd1 == 64) && (hd2 == 16 || hd2 == 32 || hd2 == 64), SELFTOK_ERR_UNSUPPORTED,
            "encoder head_dim must be 16/32/64");
  STK_CHECK(cfg->precision >= 0 && cfg->precision <= 3, SELFTOK_ERR_BAD_ARG, "bad precision");
  STK_CUDA(cudaSetDevice(cfg->device));
  selftok_engine* e = new selftok_engine();
  e->cfg = *cfg;
  e->D = 64 * cfg->dit_depth;
  e->H = cfg->dit_depth;
  e->Nimg = (cfg->latent / cfg->dit_patch) * (cfg->latent / cfg->dit_patch);
  e->Nenc = (cfg->latent / cfg->enc_patch) * (cfg->latent / cfg->enc_patch);
  if (tc_mode(e)) {
    int st = gemm_tc_init();
    if (st != 0) { delete e; return st; }
  }
  if (cudaMalloc(&e->bad_ids, sizeof(int)) != cudaSuccess || cudaMemset(e->bad_ids, 0, sizeof(int)) != cudaSuccess) {
    set_error("cudaMalloc failed in selftok_create");
    delete e;
    return SELFTOK_ERR_CUDA;
  }
  *out = e;
  return SELFTOK_OK;
}

static const size_t kPrefixGraphs = 4;
// captured decode graphs hold pointers into the decode workspace and the prefix-count buffer
static void drop_decode_graphs(selftok_engine* e) {
  for (auto& g : e->graphs) cudaGraphExecDestroy(g.second.first);
  e->graphs.clear();
  for (auto& g : e->prefix_graphs) cudaGraphExecDestroy(g.second.exec);
  e->prefix_graphs.clear();
}
static void free_dws(selftok_engine* e) {
  if (e->dws.own) { cudaFree(e->dws.own); e->bytes -= (int64_t)e->dws.own_bytes; }
  e->dws = DecodeWs();
}
static void free_ews(selftok_engine* e) {
  for (auto& g : e->enc_graphs) cudaGraphExecDestroy(g.second.first);         // graphs hold pointers into the workspace
  e->enc_graphs.clear();
  if (e->ews.own) { cudaFree(e->ews.own); e->bytes -= (int64_t)e->ews.own_bytes; }
  e->ews = EncodeWs();
}

extern "C" __attribute__((visibility("default"))) int selftok_destroy(selftok_handle_t e) {
  if (!e) return SELFTOK_OK;
  cudaSetDevice(e->cfg.device);
  cudaDeviceSynchronize();
  drop_decode_graphs(e);
  if (e->n_dev) cudaFree(e->n_dev);
  for (auto& kv : e->w) cudaFree(kv.second.d);
  free_pool(e, e->allocs);
  if (e->bad_ids) cudaFree(e->bad_ids);
  free_dws(e);
  free_ews(e);
  delete e;
  return SELFTOK_OK;
}

extern "C" __attribute__((visibility("default"))) int selftok_load_tensor(selftok_handle_t e, const char* name, const void* data, int dtype, int ndim,
                                   const int64_t* shape, int is_device) {
  STK_CHECK(e && name && data && shape && ndim >= 0 && ndim <= 8, SELFTOK_ERR_BAD_ARG, "selftok_load_tensor: bad argument");
  STK_CHECK(dtype == SELFTOK_F32, SELFTOK_ERR_UNSUPPORTED, "only fp32 checkpoint tensors are supported");
  STK_CHECK(!e->finalized, SELFTOK_ERR_STATE, "load_tensor after finalize");
  STK_CUDA(cudaSetDevice(e->cfg.device));
  Tensor t;
  t.numel = 1;
  for (int i = 0; i < ndim; ++i) { t.shape.push_back(shape[i]); t.numel *= shape[i]; }
  STK_CHECK(t.numel > 0, SELFTOK_ERR_BAD_ARG, "empty tensor");
  auto it = e->w.find(name);
  if (it != e->w.end()) { cudaFree(it->second.d); e->bytes -= it->second.numel * 4; e->w.erase(it); }
  STK_CUDA(cudaMalloc(&t.d, sizeof(float) * (size_t)t.numel));
  e->bytes += t.numel * 4;
  STK_CUDA(cudaMemcpy(t.d, data, sizeof(float) * (size_t)t.numel, is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
  e->w[name] = t;
  return SELFTOK_OK;
}

extern "C" __attribute__((visibility("default"))) int selftok_set_schedule(selftok_handle_t e, int steps, const float* t_host, const float* dt_host,
                                    const int32_t* k_host, const float* t_freq_host, const float* pos_freq_host) {
  STK_CHECK(e && steps > 0 && t_host && dt_host && k_host && t_freq_host && pos_freq_host, SELFTOK_ERR_BAD_ARG,
            "selftok_set_schedule: bad argument");
  STK_CHECK(!e->finalized, SELFTOK_ERR_STATE, "set_schedule after finalize");
  STK_CUDA(cudaSetDevice(e->cfg.device));
  e->steps = steps;
  e->t.assign(t_host, t_host + steps);
  e->dt.assign(dt_host, dt_host + steps);
  e->k.assign(k_host, k_host + steps);
  for (int i = 0; i < steps; ++i)
    STK_CHECK(e->k[i] >= 0 && e->k[i] < e->cfg.K, SELFTOK_ERR_BAD_ARG, "schedule k out of range");
  STK_TRY(dalloc(e, e->allocs, &e->t_freq, (int64_t)steps * 256));
  STK_TRY(dalloc(e, e->allocs, &e->pos_freq, (int64_t)e->cfg.K * 256));
  STK_CUDA(cudaMemcpy(e->t_freq, t_freq_host, sizeof(float) * steps * 256, cudaMemcpyHostToDevice));
  STK_CUDA(cudaMemcpy(e->pos_freq, pos_freq_host, sizeof(float) * e->cfg.K * 256, cudaMemcpyHostToDevice));
  return SELFTOK_OK;
}

// Optional, before finalize: sinusoidal features [steps,256] of floor(1000 t_i).clamp(0, 999), the timestep the unconditional
// branch of the guided sampler is embedded with (MMDiT.cfg_inference, sd3/mmdit.py:1127).  Enables selftok_decode_cfg.
extern "C" __attribute__((visibility("default"))) int selftok_set_cfg_schedule(selftok_handle_t e, const float* t_freq_uncond_host) {
  STK_CHECK(e && t_freq_uncond_host, SELFTOK_ERR_BAD_ARG, "selftok_set_cfg_schedule: bad argument");
  STK_CHECK(!e->finalized && e->steps > 0, SELFTOK_ERR_STATE, "selftok_set_cfg_schedule: after selftok_set_schedule, before selftok_finalize");
  STK_CHECK(!e->cfg.renderer, SELFTOK_ERR_STATE, "the renderer has no guided path");
  STK_CUDA(cudaSetDevice(e->cfg.device));
  if (!e->t_freq_u) STK_TRY(dalloc(e, e->allocs, &e->t_freq_u, (int64_t)e->steps * 256));
  STK_CUDA(cudaMemcpy(e->t_freq_u, t_freq_uncond_host, sizeof(float) * e->steps * 256, cudaMemcpyHostToDevice));
  return SELFTOK_OK;
}

// ------------------------------------------------------------------------------------------------ finalize
// adaLN table of a position-indexed block:  Linear(SiLU(t_embedder(pos_freq)))  (modules.py:311-318; mmdit.py:446-458)
static int build_pos_table(selftok_engine* e, const std::string& blk, const float* freq, int rows, float* tmp1, float* tmp2,
                           float* out, cudaStream_t s) {
  Epilogue ep;
  ep.act = ACT_SILU; ep.out = tmp1;
  STK_TRY(lin32(e, blk + "t_embedder.mlp.0", freq, 256, rows, ep, s));
  GETW(W2, blk + "t_embedder.mlp.2.weight");
  int dim = (int)W2->shape[0];
  ep.out = tmp2;                                            // SiLU applied here: t_emb is only consumed through SiLU
  STK_TRY(lin32(e, blk + "t_embedder.mlp.2", tmp1, dim, rows, ep, s));
  Epilogue ep2;
  ep2.out = out;
  STK_TRY(lin32(e, blk + "adaLN_modulation.1", tmp2, dim, rows, ep2, s));
  return 0;
}

extern "C" __attribute__((visibility("default"))) int selftok_finalize(selftok_handle_t e, void* stream) {
  STK_CHECK(e, SELFTOK_ERR_BAD_ARG, "null handle");
  STK_CHECK(!e->finalized, SELFTOK_ERR_STATE, "already finalized");
  STK_CHECK(e->steps > 0, SELFTOK_ERR_STATE, "selftok_set_schedule must precede finalize");
  STK_CUDA(cudaSetDevice(e->cfg.device));
  cudaStream_t s = (cudaStream_t)stream;
  const selftok_config_t& c = e->cfg;
  const int K = c.K, Q = c.enc_qdim, D = e->D, L = c.dit_depth, T = e->steps;
  // scratch for the table MLPs
  float *tmp1, *tmp2;
  int64_t rows_max = K > T ? K : T, dim_max = D > Q ? D : Q;
  std::vector<void*> scratch;
  STK_TRY(dalloc(e, scratch, &tmp1, rows_max * dim_max));
  STK_TRY(dalloc(e, scratch, &tmp2, rows_max * dim_max));
  // ---- encoder: adaLN tables [depth][K][6Q], cropped positional grid, transposed codebook
  STK_TRY(dalloc(e, e->allocs, &e->enc_mod, (int64_t)c.enc_depth * K * 6 * Q));
  for (int i = 0; i < c.enc_depth; ++i)
    STK_TRY(build_pos_table(e, "encoder.blocks." + std::to_string(i) + ".", e->pos_freq, K, tmp1, tmp2,
                            e->enc_mod + (int64_t)i * K * 6 * Q, s));
  {
    GETW(pe, "encoder.pos_embed");
    STK_CHECK(pe->numel == (int64_t)c.enc_pos_max * c.enc_pos_max * c.enc_hidden, SELFTOK_ERR_BAD_ARG, "encoder.pos_embed shape");
    int g = c.latent / c.enc_patch;
    STK_TRY(dalloc(e, e->allocs, &e->enc_pos, (int64_t)g * g * c.enc_hidden));
    PROF(PC_OTHER, launch_crop_pos(pe->d, e->enc_pos, c.enc_pos_max, g, c.enc_hidden, s));
    GETW(cb, "encoder.quantizer._codebook.embed");
    STK_CHECK(cb->numel == (int64_t)c.codebook_size * c.code_dim, SELFTOK_ERR_BAD_ARG, "codebook shape");
    STK_TRY(dalloc(e, e->allocs, &e->cbt, cb->numel));
    PROF(PC_OTHER, launch_transpose(cb->d, e->cbt, c.codebook_size, c.code_dim, s));
  }
  // ---- decoder tables
  STK_TRY(dalloc(e, e->allocs, &e->ctx_mod, (int64_t)(L - 1 > 0 ? L - 1 : 1) * K * 6 * D));
  for (int j = 0; j < L - 1; ++j)
    STK_TRY(build_pos_table(e, "model.joint_blocks." + std::to_string(j) + ".context_block.", e->pos_freq, K, tmp1, tmp2,
                            e->ctx_mod + (int64_t)j * K * 6 * D, s));
  {
    // csil = SiLU(t_embedder(t_freq)) [T, D]  (mmdit.py:1022; every consumer is Sequential(SiLU, Linear))
    float* csil;
    STK_TRY(dalloc(e, scratch, &csil, (int64_t)T * D));
    Epilogue ep;
    ep.act = ACT_SILU; ep.out = tmp1;
    STK_TRY(lin32(e, "model.t_embedder.mlp.0", e->t_freq, 256, T, ep, s));
    ep.out = csil;
    STK_TRY(lin32(e, "model.t_embedder.mlp.2", tmp1, D, T, ep, s));
    STK_TRY(dalloc(e, e->allocs, &e->x_mod, (int64_t)L * T * 6 * D));
    for (int j = 0; j < L; ++j) {
      Epilogue e2;
      e2.out = e->x_mod + (int64_t)j * T * 6 * D;
      STK_TRY(lin32(e, "model.joint_blocks." + std::to_string(j) + ".x_block.adaLN_modulation.1", csil, D, T, e2, s));
    }
    STK_TRY(dalloc(e, e->allocs, &e->ctx_last_mod, (int64_t)T * 2 * D));
    Epilogue e3;
    e3.out = e->ctx_last_mod;
    STK_TRY(lin32(e, "model.joint_blocks." + std::to_string(L - 1) + ".context_block.adaLN_modulation.1", csil, D, T, e3, s));
    STK_TRY(dalloc(e, e->allocs, &e->final_mod, (int64_t)T * 2 * D));
    Epilogue e4;
    e4.out = e->final_mod;
    STK_TRY(lin32(e, "model.final_layer.adaLN_modulation.1", csil, D, T, e4, s));
    if (e->t_freq_u) {
      // unconditional branch of the guided sampler: same MLPs on the integer-floored timestep (mmdit.py:1127-1130), image
      // stream only (every row of that pass is blind to the context keys, so the context stream never reaches the output)
      ep.act = ACT_SILU; ep.out = tmp1;
      STK_TRY(lin32(e, "model.t_embedder.mlp.0", e->t_freq_u, 256, T, ep, s));
      ep.out = csil;
      STK_TRY(lin32(e, "model.t_embedder.mlp.2", tmp1, D, T, ep, s));
      STK_TRY(dalloc(e, e->allocs, &e->x_mod_u, (int64_t)L * T * 6 * D));
      for (int j = 0; j < L; ++j) {
        Epilogue e2;
        e2.out = e->x_mod_u + (int64_t)j * T * 6 * D;
        STK_TRY(lin32(e, "model.joint_blocks." + std::to_string(j) + ".x_block.adaLN_modulation.1", csil, D, T, e2, s));
      }
      STK_TRY(dalloc(e, e->allocs, &e->final_mod_u, (int64_t)T * 2 * D));
      Epilogue e5;
      e5.out = e->final_mod_u;
      STK_TRY(lin32(e, "model.final_layer.adaLN_modulation.1", csil, D, T, e5, s));
    }
  }
  if (c.renderer) {
    GETW(pe, "model.positional_embedding");
    GETW(mt, "model.mask_token");
    STK_CHECK(pe->numel == (int64_t)e->Nimg * D && mt->numel == D, SELFTOK_ERR_UNSUPPORTED,
              "renderer expects positional_embedding [N,D] and mask_token [1,1,D] (repeat=True)");
    float* tmp;
    STK_TRY(dalloc(e, scratch, &tmp, (int64_t)e->Nimg * D));
    STK_TRY(dalloc(e, e->allocs, &e->rend_x0, (int64_t)e->Nimg * D));
    PROF(PC_OTHER, launch_bcast_rows(mt->d, nullptr, tmp, e->Nimg, 1, D, s));
    PROF(PC_OTHER, launch_bcast_rows(tmp, pe->d, e->rend_x0, 1, e->Nimg, D, s));
  } else {
    GETW(pe, "model.pos_embed");
    STK_CHECK(pe->numel == (int64_t)c.dit_pos_max * c.dit_pos_max * D, SELFTOK_ERR_BAD_ARG, "model.pos_embed shape");
    int g = c.latent / c.dit_patch;
    STK_TRY(dalloc(e, e->allocs, &e->dit_pos, (int64_t)g * g * D));
    PROF(PC_OTHER, launch_crop_pos(pe->d, e->dit_pos, c.dit_pos_max, g, D, s));
  }
  // ---- tensor-core operand planes of the MMDiT linears
  std::vector<std::string> packed_names;
  if (tc_mode(e)) {
    const char* blocks[2] = {"context_block", "x_block"};
    const char* lins[4] = {"attn.qkv", "attn.proj", "mlp.fc1", "mlp.fc2"};
    for (int j = 0; j < L; ++j)
      for (int b = 0; b < 2; ++b)
        for (int l = 0; l < 4; ++l) {
          if (j == L - 1 && b == 0 && l > 0) continue;          // pre_only context block: qkv only
          std::string name = "model.joint_blocks." + std::to_string(j) + "." + blocks[b] + "." + lins[l] + ".weight";
          GETW(W, name);
          WPack p;
          STK_TRY(dalloc(e, e->allocs, &p.hi, W->numel));
          if (nsplit(e) == 3) STK_TRY(dalloc(e, e->allocs, &p.lo, W->numel));
          PROF(PC_OTHER, launch_split_bf16(W->d, p.hi, p.lo, W->numel, s, is_fp16(e)));
          e->wp[name] = p;
          packed_names.push_back(name);
        }
  }
  if (tc_mode(e)) {
    // the patch embedding (K = 64) and the final layer (N = 64) stay fp32-faithful in every tensor-core mode: split-bf16 planes
    // (hi + lo, three MMAs per product); their fp32 copies are kept (the fp32 FFMA mode and the table MLPs read them)
    for (const char* nm : {"model.x_embedder.proj.weight", "model.final_layer.linear.weight"}) {
      if (c.renderer && std::string(nm) == "model.x_embedder.proj.weight") continue;      // the renderer has no x_embedder
      GETW(W, nm);
      WPack p;
      STK_TRY(dalloc(e, e->allocs, &p.hi, W->numel));
      STK_TRY(dalloc(e, e->allocs, &p.lo, W->numel));
      PROF(PC_OTHER, launch_split_bf16(W->d, p.hi, p.lo, W->numel, s, 0));
      e->wp[nm] = p;
    }
  }
  STK_CUDA(cudaStreamSynchronize(s));
  for (void* p : scratch) cudaFree(p);
  // the fp32 staging copies of the packed MMDiT weights are not read again (their shapes are): release 8.3 GB
  for (const std::string& name : packed_names) {
    Tensor& t = e->w[name];
    cudaFree(t.d);
    t.d = nullptr;
    e->bytes -= t.numel * 4;
  }
  e->has_cfg = e->x_mod_u != nullptr;
  e->finalized = true;
  return SELFTOK_OK;
}

// ------------------------------------------------------------------------------------------------ prepack cache
// The finalized device state (fp32 tensors that stay fp32, 16-bit operand planes, every static table, the schedule) as ONE
// file, so that a later process skips torch.load of the fp32 checkpoint, the per-tensor uploads, the table MLPs and the
// packing (SURVEY 8f rank 2: checkpoint loader + prepack cache; SelftokPipeline.py:188-199 reloads 8.3 GB of fp32 per process).
struct TableRef { const char* tag; float** ptr; int64_t numel; };
static std::vector<TableRef> table_refs(selftok_engine* e) {
  const selftok_config_t& c = e->cfg;
  const int64_t K = c.K, Q = c.enc_qdim, D = e->D, L = c.dit_depth, T = e->steps;
  const int64_t ge = c.latent / c.enc_patch, gd = c.latent / c.dit_patch;
  std::vector<TableRef> t = {
      {"t_freq", &e->t_freq, T * 256}, {"pos_freq", &e->pos_freq, K * 256},
      {"enc_mod", &e->enc_mod, (int64_t)c.enc_depth * K * 6 * Q}, {"enc_pos", &e->enc_pos, ge * ge * c.enc_hidden},
      {"cbt", &e->cbt, (int64_t)c.codebook_size * c.code_dim},
      {"ctx_mod", &e->ctx_mod, (L - 1 > 0 ? L - 1 : 1) * K * 6 * D}, {"x_mod", &e->x_mod, L * T * 6 * D},
      {"ctx_last_mod", &e->ctx_last_mod, T * 2 * D}, {"final_mod", &e->final_mod, T * 2 * D}};
  if (c.renderer) t.push_back({"rend_x0", &e->rend_x0, (int64_t)e->Nimg * D});
  else t.push_back({"dit_pos", &e->dit_pos, gd * gd * D});
  if (e->has_cfg) {
    t.push_back({"x_mod_u", &e->x_mod_u, L * T * 6 * D});
    t.push_back({"final_mod_u", &e->final_mod_u, T * 2 * D});
  }
  return t;
}
static const char kPackMagic[8] = {'S', 'T', 'K', 'P', 'A', 'C', 'K', '3'};
static bool same_model(const selftok_config_t& a, const selftok_config_t& b) {
  selftok_config_t x = a, y = b;
  x.device = y.device = 0;
  return memcmp(&x, &y, sizeof(x)) == 0;
}
namespace {
struct PackIO {
  FILE* f = nullptr;
  void* bounce = nullptr;                                     // pinned staging buffer
  static constexpr size_t CH = 64u << 20;
  ~PackIO() { if (f) fclose(f); if (bounce) cudaFreeHost(bounce); }
  bool w(const void* p, size_t n) { return fwrite(p, 1, n, f) == n; }
  bool r(void* p, size_t n) { return fread(p, 1, n, f) == n; }
  bool wdev(const void* d, size_t n) {
    for (size_t o = 0; o < n; o += CH) {
      const size_t m = n - o < CH ? n - o : CH;
      if (cudaMemcpy(bounce, (const char*)d + o, m, cudaMemcpyDeviceToHost) != cudaSuccess || !w(bounce, m)) return false;
    }
    return true;
  }
  bool rdev(void* d, size_t n) {
    for (size_t o = 0; o < n; o += CH) {
      const size_t m = n - o < CH ? n - o : CH;
      if (!r(bounce, m) || cudaMemcpy((char*)d + o, bounce, m, cudaMemcpyHostToDevice) != cudaSuccess) return false;
    }
    return true;
  }
  bool wstr(const std::string& s) { uint32_t n = (uint32_t)s.size(); return w(&n, 4) && w(s.data(), n); }
  bool rstr(std::string& s) { uint32_t n = 0; if (!r(&n, 4) || n > 4096) return false; s.resize(n); return r(&s[0], n); }
};
}  // namespace

extern "C" __attribute__((visibility("default"))) int selftok_export_packed(selftok_handle_t e, const char* path) {
  STK_CHECK(e && path, SELFTOK_ERR_BAD_ARG, "selftok_export_packed: bad argument");
  STK_CHECK(e->finalized, SELFTOK_ERR_STATE, "selftok_export_packed: finalize first");
  STK_CUDA(cudaSetDevice(e->cfg.device));
  STK_CUDA(cudaDeviceSynchronize());
  PackIO io;
  const std::string tmp = std::string(path) + ".tmp";
  io.f = fopen(tmp.c_str(), "wb");
  STK_CHECK(io.f, SELFTOK_ERR_BAD_ARG, "selftok_export_packed: cannot open the file for writing");
  STK_CUDA(cudaMallocHost(&io.bounce, PackIO::CH));
  bool ok = io.w(kPackMagic, 8);
  const uint32_t cfg_bytes = sizeof(selftok_config_t), steps = (uint32_t)e->steps, has_cfg = e->has_cfg ? 1u : 0u;
  ok = ok && io.w(&cfg_bytes, 4) && io.w(&e->cfg, cfg_bytes) && io.w(&has_cfg, 4) && io.w(&steps, 4) && io.w(e->t.data(), 4 * steps) &&
       io.w(e->dt.data(), 4 * steps) && io.w(e->k.data(), 4 * steps);
  const uint32_t n_w = (uint32_t)e->w.size(), n_p = (uint32_t)e->wp.size();
  ok = ok && io.w(&n_w, 4);
  for (auto& kv : e->w) {
    if (!ok) break;
    const Tensor& t = kv.second;
    const uint32_t nd = (uint32_t)t.shape.size(), has = t.d != nullptr;
    ok = io.wstr(kv.first) && io.w(&nd, 4) && io.w(t.shape.data(), 8 * nd) && io.w(&has, 4);
    if (ok && has) ok = io.wdev(t.d, sizeof(float) * (size_t)t.numel);
  }
  ok = ok && io.w(&n_p, 4);
  for (auto& kv : e->wp) {
    if (!ok) break;
    const int64_t numel = e->w[kv.first].numel;
    const uint32_t has_lo = kv.second.lo != nullptr;
    ok = io.wstr(kv.first) && io.w(&numel, 8) && io.w(&has_lo, 4) && io.wdev(kv.second.hi, 2 * (size_t)numel);
    if (ok && has_lo) ok = io.wdev(kv.second.lo, 2 * (size_t)numel);
  }
  for (const TableRef& t : table_refs(e)) {
    if (!ok) break;
    ok = io.wstr(t.tag) && io.w(&t.numel, 8) && io.wdev(*t.ptr, sizeof(float) * (size_t)t.numel);
  }
  fclose(io.f);
  io.f = nullptr;
  if (!ok) { remove(tmp.c_str()); set_error("selftok_export_packed: write failed"); return SELFTOK_ERR_CUDA; }
  STK_CHECK(rename(tmp.c_str(), path) == 0, SELFTOK_ERR_BAD_ARG, "selftok_export_packed: rename failed");
  return SELFTOK_OK;
}

// Fresh handle (selftok_create only) -> the finalized state of the file.  The file must have been exported for the same
// model configuration, precision and schedule length; anything else is SELFTOK_ERR_BAD_ARG and the handle stays fresh.
extern "C" __attribute__((visibility("default"))) int selftok_import_packed(selftok_handle_t e, const char* path) {
  STK_CHECK(e && path, SELFTOK_ERR_BAD_ARG, "selftok_import_packed: bad argument");
  STK_CHECK(!e->finalized && e->w.empty() && e->steps == 0, SELFTOK_ERR_STATE, "selftok_import_packed: the handle is not fresh");
  STK_CUDA(cudaSetDevice(e->cfg.device));
  PackIO io;
  io.f = fopen(path, "rb");
  STK_CHECK(io.f, SELFTOK_ERR_BAD_ARG, "selftok_import_packed: cannot open the file");
  char magic[8];
  uint32_t cfg_bytes = 0, steps = 0;
  selftok_config_t fc;
  STK_CHECK(io.r(magic, 8) && memcmp(magic, kPackMagic, 8) == 0 && io.r(&cfg_bytes, 4) && cfg_bytes == sizeof(fc) && io.r(&fc, cfg_bytes),
            SELFTOK_ERR_BAD_ARG, "selftok_import_packed: not a selftok_b200 pack file of this ABI");
  STK_CHECK(same_model(fc, e->cfg), SELFTOK_ERR_BAD_ARG, "selftok_import_packed: the file was exported for another configuration / precision");
  uint32_t has_cfg = 0;
  STK_CHECK(io.r(&has_cfg, 4) && io.r(&steps, 4) && steps > 0 && steps < 100000, SELFTOK_ERR_BAD_ARG, "selftok_import_packed: bad header");
  e->has_cfg = has_cfg != 0;
  STK_CUDA(cudaMallocHost(&io.bounce, PackIO::CH));
  e->steps = (int)steps;
  e->t.resize(steps); e->dt.resize(steps); e->k.resize(steps);
  bool ok = io.r(e->t.data(), 4 * steps) && io.r(e->dt.data(), 4 * steps) && io.r(e->k.data(), 4 * steps);
  uint32_t n_w = 0, n_p = 0;
  ok = ok && io.r(&n_w, 4) && n_w < 100000;
  for (uint32_t i = 0; ok && i < n_w; ++i) {
    std::string name;
    uint32_t nd = 0, has = 0;
    Tensor t;
    ok = io.rstr(name) && io.r(&nd, 4) && nd <= 8;
    if (!ok) break;
    t.shape.resize(nd);
    ok = io.r(t.shape.data(), 8 * nd) && io.r(&has, 4);
    t.numel = 1;
    for (int64_t d : t.shape) t.numel *= d;
    if (ok && has) {
      ok = cudaMalloc(&t.d, sizeof(float) * (size_t)t.numel) == cudaSuccess && io.rdev(t.d, sizeof(float) * (size_t)t.numel);
      e->bytes += t.numel * 4;
    }
    e->w[name] = t;
  }
  ok = ok && io.r(&n_p, 4) && n_p < 100000;
  for (uint32_t i = 0; ok && i < n_p; ++i) {
    std::string name;
    int64_t numel = 0;
    uint32_t has_lo = 0;
    WPack pk;
    ok = io.rstr(name) && io.r(&numel, 8) && io.r(&has_lo, 4) && numel > 0;
    if (!ok) break;
    ok = dalloc(e, e->allocs, &pk.hi, numel) == 0 && io.rdev(pk.hi, 2 * (size_t)numel);
    if (ok && has_lo) ok = dalloc(e, e->allocs, &pk.lo, numel) == 0 && io.rdev(pk.lo, 2 * (size_t)numel);
    e->wp[name] = pk;
  }
  for (const TableRef& t : table_refs(e)) {
    if (!ok) break;
    std::string tag;
    int64_t numel = 0;
    ok = io.rstr(tag) && tag == t.tag && io.r(&numel, 8) && numel == t.numel && dalloc(e, e->allocs, t.ptr, numel) == 0 &&
         io.rdev(*t.ptr, sizeof(float) * (size_t)numel);
  }
  if (!ok) {
    set_error("selftok_import_packed: truncated or mismatching pack file (destroy the handle)");
    return SELFTOK_ERR_BAD_ARG;
  }
  e->finalized = true;
  return SELFTOK_OK;
}

// ------------------------------------------------------------------------------------------------ encode
static int layout_ews(selftok_engine* e, EncodeWs& w, int64_t B, Arena& A) {
  const selftok_config_t& c = e->cfg;
  const int64_t Ni = e->Nenc, K = c.K, Hh = c.enc_hidden, Q = c.enc_qdim;
  STK_TRY(A.take(&w.x0, B * c.in_channels * c.latent * c.latent));
  STK_TRY(A.take(&w.patch, B * Ni * c.in_channels * c.enc_patch * c.enc_patch));
  STK_TRY(A.take(&w.x, B * Ni * Hh));
  STK_TRY(A.take(&w.q, B * K * Q));
  STK_TRY(A.take(&w.xn, B * Ni * Hh));
  STK_TRY(A.take(&w.qn, B * K * Q));
  STK_TRY(A.take(&w.xqkv, B * Ni * 3 * Hh));
  STK_TRY(A.take(&w.xkv, B * Ni * 2 * Q));
  STK_TRY(A.take(&w.qqkv, B * K * 3 * Q));
  STK_TRY(A.take(&w.xattn, B * Ni * Hh));
  STK_TRY(A.take(&w.qattn, B * K * Q));
  STK_TRY(A.take(&w.xh, B * Ni * 4 * Hh));
  STK_TRY(A.take(&w.qh, B * K * 4 * Q));
  STK_TRY(A.take(&w.outs_q, B * K * c.code_dim));
  STK_TRY(A.take(&w.tokens, B * K));
  return 0;
}
// carve the workspace of `op` (0 encode, 1 decode / render) for batch B from the caller's block if it is large enough, else from
// one cudaMalloc of exactly the needed size
template <typename WS, typename LAYOUT>
static int place_ws(selftok_engine* e, int op, WS& w, int B, LAYOUT layout) {
  Arena dry;
  dry.dry = true;
  WS scratch;
  STK_TRY(layout(scratch, (int64_t)B, dry));
  Arena A;
  if (e->user_ws[op] && e->user_ws_bytes[op] >= dry.off) {
    A.base = reinterpret_cast<char*>(e->user_ws[op]);
    A.cap = e->user_ws_bytes[op];
  } else {
    STK_CUDA(cudaMalloc(&w.own, dry.off));
    w.own_bytes = dry.off;
    e->bytes += (int64_t)dry.off;
    A.base = reinterpret_cast<char*>(w.own);
    A.cap = dry.off;
  }
  STK_TRY(layout(w, (int64_t)B, A));
  w.B = B;
  return 0;
}
static int ensure_ews(selftok_engine* e, int B) {
  if (e->ews.B >= B) return 0;
  free_ews(e);
  return place_ws(e, 0, e->ews, B, [&](EncodeWs& w, int64_t b, Arena& A) { return layout_ews(e, w, b, A); });
}

// Encoder.forward up to the quantizer input (models_ours.py:204-219,315-343; modules.py:310-327)
static int encoder_features(selftok_engine* e, const float* x0, int B, cudaStream_t s) {
  EncodeWs& w = e->ews;
  const selftok_config_t& c = e->cfg;
  const int Ni = e->Nenc, K = c.K, Hh = c.enc_hidden, Q = c.enc_qdim;
  const int64_t Mx = (int64_t)B * Ni, Mq = (int64_t)B * K;
  const float eps = 1e-6f;
  PROF(PC_OTHER, launch_patchify(x0, w.patch, B, c.in_channels, c.latent, c.latent, c.enc_patch, s));
  {
    Epilogue ep;
    ep.out = w.x; ep.addtab = e->enc_pos; ep.add_ld = Hh; ep.add_period = Ni;
    STK_TRY(lin32(e, "encoder.x_embedder.proj", w.patch, c.in_channels * c.enc_patch * c.enc_patch, Mx, ep, s));
    GETW(qt, "encoder.query_tokens");
    STK_CHECK(qt->numel == (int64_t)K * Q, SELFTOK_ERR_BAD_ARG, "query_tokens shape");
    PROF(PC_OTHER, launch_bcast_rows(qt->d, nullptr, w.q, B, K, Q, s));
  }
  for (int i = 0; i < c.enc_depth; ++i) {
    const std::string p = "encoder.blocks." + std::to_string(i) + ".";
    const float* mod = e->enc_mod + (int64_t)i * K * 6 * Q;     // [K][shift_msa|scale_msa|gate_msa|shift_mlp|scale_mlp|gate_mlp]
    PROF(PC_LN, launch_ln_mod(w.x, Hh, nullptr, nullptr, 0, 1, w.xn, nullptr, nullptr, Hh, Mx, Hh, eps, s));
    PROF(PC_LN, launch_ln_mod(w.q, Q, mod, mod + Q, 6 * Q, K, w.qn, nullptr, nullptr, Q, Mq, Q, eps, s));
    Epilogue ep;
    ep.out = w.xqkv; STK_TRY(lin32(e, p + "attn.qkv", w.xn, Hh, Mx, ep, s));
    ep.out = w.xkv; STK_TRY(lin32(e, p + "attn.to_query_kv", w.xn, Hh, Mx, ep, s));
    ep.out = w.qqkv; STK_TRY(lin32(e, p + "attn.query_linear", w.qn, Q, Mq, ep, s));
    AttnOut ox;
    ox.f32_a = w.xattn; ox.split = Ni; ox.ld = Hh;
    PROF(PC_ATTN, launch_attention_f32(w.xqkv, 3 * Hh, (int64_t)Ni * 3 * Hh, w.xqkv + Hh, w.xqkv + 2 * Hh, 3 * Hh, (int64_t)Ni * 3 * Hh, Ni,
                                 nullptr, nullptr, 0, 0, 0, ox, B, Ni, c.enc_heads, Hh / c.enc_heads, 0, 0, s));
    AttnOut oq;
    oq.f32_a = w.qattn; oq.split = K; oq.ld = Q;
    PROF(PC_ATTN, launch_attention_f32(w.qqkv, 3 * Q, (int64_t)K * 3 * Q, w.xkv, w.xkv + Q, 2 * Q, (int64_t)Ni * 2 * Q, Ni,
                                 w.qqkv + Q, w.qqkv + 2 * Q, 3 * Q, (int64_t)K * 3 * Q, K, oq, B, K, c.enc_qheads,
                                 Q / c.enc_qheads, 0, 0, s));
    // image stream: x += proj(x_attn); x += mlp(norm2(x))
    Epilogue er;
    er.mode = EPI_RESID; er.out = w.x; er.resid = w.x; er.ldo = Hh;
    STK_TRY(lin32(e, p + "attn.proj", w.xattn, Hh, Mx, er, s));
    PROF(PC_LN, launch_ln_mod(w.x, Hh, nullptr, nullptr, 0, 1, w.xn, nullptr, nullptr, Hh, Mx, Hh, eps, s));
    Epilogue eg;
    eg.act = ACT_GELU; eg.out = w.xh;
    STK_TRY(lin32(e, p + "mlp.fc1", w.xn, Hh, Mx, eg, s));
    STK_TRY(lin32(e, p + "mlp.fc2", w.xh, 4 * Hh, Mx, er, s));
    // query stream: q += gate_msa * query_proj(q_attn); q += gate_mlp * q_mlp(modulate(norm2(q)))
    Epilogue eq;
    eq.mode = EPI_RESID; eq.out = w.q; eq.resid = w.q; eq.ldo = Q; eq.gate = mod + 2 * Q; eq.gate_ld = 6 * Q; eq.gate_period = K;
    STK_TRY(lin32(e, p + "attn.query_proj", w.qattn, Q, Mq, eq, s));
    PROF(PC_LN, launch_ln_mod(w.q, Q, mod + 3 * Q, mod + 4 * Q, 6 * Q, K, w.qn, nullptr, nullptr, Q, Mq, Q, eps, s));
    eg.out = w.qh;
    STK_TRY(lin32(e, p + "q_mlp.fc1", w.qn, Q, Mq, eg, s));
    eq.gate = mod + 5 * Q;
    STK_TRY(lin32(e, p + "q_mlp.fc2", w.qh, 4 * Q, Mq, eq, s));
  }
  return 0;
}

static int run_vq(selftok_engine* e, const float* z, int64_t R, int64_t* ids, float* outs_q, cudaStream_t s) {
  const selftok_config_t& c = e->cfg;
  GETW(wi, "encoder.quantizer.project_in.weight");
  GETW(bi, "encoder.quantizer.project_in.bias");
  GETW(cb, "encoder.quantizer._codebook.embed");
  GETW(lw, "encoder.final_layer_norm3.weight");
  GETW(lb, "encoder.final_layer_norm3.bias");
  PROF(PC_VQ, launch_vq(z, R, c.enc_qdim, wi->d, bi->d, cb->d, e->cbt, c.codebook_size, c.code_dim, lw->d, lb->d, ids, outs_q, s));
  return 0;
}

#define HOT_PROLOGUE(e)                                                                  \
  STK_CHECK(e, SELFTOK_ERR_BAD_ARG, "null handle");                                      \
  STK_CHECK(e->finalized, SELFTOK_ERR_STATE, "selftok_finalize has not been called");    \
  STK_CUDA(cudaSetDevice(e->cfg.device));                                                \
  cudaStream_t s = (cudaStream_t)stream;                                                 \
  const int64_t launches0 = g_launch_count;

extern "C" __attribute__((visibility("default"))) int selftok_encode(selftok_handle_t e, const float* x0_dev, int B, int64_t* tokens_dev, float* outs_q_dev,
                              float* feats_dev, void* stream) {
  HOT_PROLOGUE(e);
  STK_CHECK(x0_dev && tokens_dev && B > 0, SELFTOK_ERR_BAD_ARG, "selftok_encode: bad argument");
  STK_TRY(ensure_ews(e, B));
  const int64_t R = (int64_t)B * e->cfg.K;
  EncodeWs& w = e->ews;
  if (!e->use_graph || e->prof_on) {                       // eager (per-launch profiling needs real launches)
    STK_TRY(encoder_features(e, x0_dev, B, s));
    STK_TRY(run_vq(e, w.q, R, tokens_dev, outs_q_dev ? outs_q_dev : w.outs_q, s));
    e->last_launches = g_launch_count - launches0;
  } else {
    // one CUDA graph per batch size over the workspace's own input / output buffers (the ~250 launches of the 16 dual blocks
    // dominate a small-batch encode when issued one by one); the caller's buffers are copied in and out around the replay
    const int64_t nlat = (int64_t)B * e->cfg.in_channels * e->cfg.latent * e->cfg.latent;
    if (x0_dev != w.x0) STK_CUDA(cudaMemcpyAsync(w.x0, x0_dev, sizeof(float) * nlat, cudaMemcpyDeviceToDevice, s));
    auto it = e->enc_graphs.find(B);
    if (it == e->enc_graphs.end()) {
      cudaStream_t cs;
      STK_CUDA(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
      {
        const cudaError_t be = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
        if (be != cudaSuccess) {
          cudaStreamDestroy(cs);
          STK_CUDA(be);
        }
      }
      const int64_t l0 = g_launch_count;
      int st = encoder_features(e, w.x0, B, cs);
      if (!st) st = run_vq(e, w.q, R, w.tokens, w.outs_q, cs);
      cudaGraph_t graph = nullptr;
      cudaError_t ce = cudaStreamEndCapture(cs, &graph);
      cudaStreamDestroy(cs);
      if (st != 0) { if (graph) cudaGraphDestroy(graph); return st; }
      STK_CUDA(ce);
      cudaGraphExec_t exec;
      STK_CUDA(cudaGraphInstantiate(&exec, graph, 0));
      cudaGraphDestroy(graph);
      it = e->enc_graphs.emplace(B, std::make_pair(exec, g_launch_count - l0)).first;
    }
    STK_CUDA(cudaGraphLaunch(it->second.first, s));
    e->last_launches = it->second.second;
    if (tokens_dev != w.tokens) STK_CUDA(cudaMemcpyAsync(tokens_dev, w.tokens, sizeof(int64_t) * R, cudaMemcpyDeviceToDevice, s));
    if (outs_q_dev && outs_q_dev != w.outs_q)
      STK_CUDA(cudaMemcpyAsync(outs_q_dev, w.outs_q, sizeof(float) * R * e->cfg.code_dim, cudaMemcpyDeviceToDevice, s));
  }
  if (feats_dev) STK_CUDA(cudaMemcpyAsync(feats_dev, w.q, sizeof(float) * R * e->cfg.enc_qdim, cudaMemcpyDeviceToDevice, s));
  return SELFTOK_OK;
}

extern "C" __attribute__((visibility("default"))) int selftok_vq_argmax(selftok_handle_t e, const float* z_dev, int64_t R, int64_t* ids_dev, float* outs_q_dev,
                                 void* stream) {
  HOT_PROLOGUE(e);
  STK_CHECK(z_dev && ids_dev && R > 0, SELFTOK_ERR_BAD_ARG, "selftok_vq_argmax: bad argument");
  STK_TRY(run_vq(e, z_dev, R, ids_dev, outs_q_dev, s));
  e->last_launches = g_launch_count - launches0;
  return SELFTOK_OK;
}

// n_tok (device [B], optional): image b from its first n_tok[b] tokens
static int run_lookup(selftok_engine* e, const int64_t* tokens, int B, float* outs_q, cudaStream_t s, const int32_t* n_tok = nullptr) {
  GETW(cb, "encoder.quantizer._codebook.embed");
  GETW(lw, "encoder.final_layer_norm3.weight");
  GETW(lb, "encoder.final_layer_norm3.bias");
  if (n_tok) {
    PROF(PC_OTHER, launch_lookup_ln3_prefix(tokens, B, e->cfg.K, n_tok, cb->d, e->cfg.codebook_size, e->cfg.code_dim, lw->d, lb->d,
                                            outs_q, e->bad_ids, s));
    return 0;
  }
  PROF(PC_OTHER, launch_lookup_ln3(tokens, (int64_t)B * e->cfg.K, cb->d, e->cfg.codebook_size, e->cfg.code_dim, lw->d, lb->d, outs_q,
                                   e->bad_ids, s));
  return 0;
}

// Synchronises `stream`, returns how many token ids outside [0, codebook_size) the lookups on this handle have seen since
// the last call (their rows were poisoned with NaN) and resets the counter; < 0 on a CUDA error.
extern "C" __attribute__((visibility("default"))) int64_t selftok_id_errors(selftok_handle_t e, void* stream) {
  if (!e || !e->bad_ids) return -1;
  int n = 0;
  if (cudaSetDevice(e->cfg.device) != cudaSuccess) return -1;
  cudaStream_t s = (cudaStream_t)stream;
  if (cudaMemcpyAsync(&n, e->bad_ids, sizeof(int), cudaMemcpyDeviceToHost, s) != cudaSuccess) return -1;
  if (cudaMemsetAsync(e->bad_ids, 0, sizeof(int), s) != cudaSuccess) return -1;
  if (cudaStreamSynchronize(s) != cudaSuccess) return -1;
  return n;
}
static int check_ids_after_sync(selftok_engine* e, void* stream, const char* who) {
  const int64_t n = selftok_id_errors(e, stream);
  STK_CHECK(n >= 0, SELFTOK_ERR_CUDA, "selftok_id_errors failed");
  if (n > 0) {
    set_error(std::string(who) + ": " + std::to_string(n) + " token id(s) outside [0, codebook_size)");
    return SELFTOK_ERR_BAD_ARG;
  }
  return 0;
}

extern "C" __attribute__((visibility("default"))) int selftok_lookup(selftok_handle_t e, const int64_t* tokens_dev, int B, float* outs_q_dev, void* stream) {
  HOT_PROLOGUE(e);
  STK_CHECK(tokens_dev && outs_q_dev && B > 0, SELFTOK_ERR_BAD_ARG, "selftok_lookup: bad argument");
  STK_TRY(run_lookup(e, tokens_dev, B, outs_q_dev, s));
  e->last_launches = g_launch_count - launches0;
  return SELFTOK_OK;
}

// ------------------------------------------------------------------------------------------------ decode
static int layout_dws(selftok_engine* e, DecodeWs& w, int64_t B, Arena& A) {
  const selftok_config_t& c = e->cfg;
  const int64_t K = c.K, N = e->Nimg, D = e->D, S = K + N;
  STK_TRY(A.take(&w.tokens, B * K));
  STK_TRY(A.take(&w.outs_q, B * K * c.code_dim));
  STK_TRY(A.take(&w.x_lat, B * c.in_channels * c.latent * c.latent));
  STK_TRY(A.take(&w.patch, B * N * c.in_channels * c.dit_patch * c.dit_patch));
  STK_TRY(A.take(&w.ctx0, B * K * D));
  STK_TRY(A.take(&w.ctx, B * K * D));
  STK_TRY(A.take(&w.x, B * N * D));
  STK_TRY(A.take(&w.o_final, B * N * c.dit_patch * c.dit_patch * c.in_channels));
  STK_TRY(A.take(&w.o_final_u, B * N * c.dit_patch * c.dit_patch * c.in_channels));
  STK_TRY(A.take(&w.a_x, B * N * D));                       // fp32 LN output of the final layer (both modes)
  if (!tc_mode(e)) {
    STK_TRY(A.take(&w.qkv, B * S * 3 * D));
    STK_TRY(A.take(&w.a_c, B * K * D));
    STK_TRY(A.take(&w.attn_c, B * K * D));
    STK_TRY(A.take(&w.attn_x, B * N * D));
    STK_TRY(A.take(&w.h_c, B * K * 4 * D));
    STK_TRY(A.take(&w.h_x, B * N * 4 * D));
  } else {
    const bool lo = nsplit(e) == 3;
    STK_TRY(A.take(&w.patch_hi, B * N * c.in_channels * c.dit_patch * c.dit_patch));
    STK_TRY(A.take(&w.patch_lo, B * N * c.in_channels * c.dit_patch * c.dit_patch));
    STK_TRY(A.take(&w.fin_hi, B * N * D));
    STK_TRY(A.take(&w.fin_lo, B * N * D));
    STK_TRY(A.take(&w.qkv_hi, B * S * 3 * D));
    if (lo) STK_TRY(A.take(&w.qkv_lo, B * S * 3 * D));
    STK_TRY(A.take(&w.a_c_hi, B * K * D));
    STK_TRY(A.take(&w.a_x_hi, B * N * D));
    STK_TRY(A.take(&w.attn_c_hi, B * K * D));
    STK_TRY(A.take(&w.attn_x_hi, B * N * D));
    STK_TRY(A.take(&w.h_c_hi, B * K * 4 * D));
    STK_TRY(A.take(&w.h_x_hi, B * N * 4 * D));
    if (lo) {
      STK_TRY(A.take(&w.a_c_lo, B * K * D));
      STK_TRY(A.take(&w.a_x_lo, B * N * D));
      STK_TRY(A.take(&w.attn_c_lo, B * K * D));
      STK_TRY(A.take(&w.attn_x_lo, B * N * D));
      STK_TRY(A.take(&w.h_c_lo, B * K * 4 * D));
      STK_TRY(A.take(&w.h_x_lo, B * N * 4 * D));
    }
  }
  return 0;
}
static int ensure_dws(selftok_engine* e, int B) {
  if (e->dws.B >= B) return 0;
  drop_decode_graphs(e);
  free_dws(e);
  return place_ws(e, 1, e->dws, B, [&](DecodeWs& w, int64_t b, Arena& A) { return layout_dws(e, w, b, A); });
}

// One stream of one JointBlock: LN+modulate -> qkv GEMM into the joint buffer   (mmdit.py:441-483, 521-529)
static int pre_attention(selftok_engine* e, const std::string& blk, const float* resid, int64_t M, const float* shift,
                         const float* scale, int64_t ld_mod, int period, float* a32, bf16* a_hi, bf16* a_lo, int rpb_in,
                         int S, int row_off, cudaStream_t s) {
  const int D = e->D;
  DecodeWs& w = e->dws;
  Epilogue ep;
  ep.out = w.qkv; ep.ldo = 3 * D; ep.rpb_in = rpb_in; ep.rpb_out = S; ep.row_off = row_off;
  if (!tc_mode(e)) {
    PROF(PC_LN, launch_ln_mod(resid, D, shift, scale, ld_mod, period, a32, nullptr, nullptr, D, M, D, 1e-6f, s));
    return lin32(e, blk + "attn.qkv", a32, D, M, ep, s);
  }
  PROF(PC_LN, launch_ln_mod(resid, D, shift, scale, ld_mod, period, nullptr, a_hi, a_lo, D, M, D, 1e-6f, s, is_fp16(e)));
  ep.mode = EPI_SPLIT; ep.out = nullptr; ep.out_hi = w.qkv_hi; ep.out_lo = w.qkv_lo;      // q/k/v leave the GEMM as 16-bit planes
  return lintc(e, blk + "attn.qkv", a_hi, a_lo, M, ep, s);
}

// post_attention (mmdit.py:485-496): x += gate_msa*proj(attn); x += gate_mlp*mlp(modulate(norm2(x)))
static int post_attention(selftok_engine* e, const std::string& blk, float* resid, int64_t M, const float* mod, int64_t ld_mod,
                          int period, const float* attn32, const bf16* attn_hi, const bf16* attn_lo, float* a32, bf16* a_hi,
                          bf16* a_lo, float* h32, bf16* h_hi, bf16* h_lo, cudaStream_t s) {
  const int D = e->D;
  Epilogue er;
  er.mode = EPI_RESID; er.out = resid; er.resid = resid; er.ldo = D;
  er.gate = mod + 2 * D; er.gate_ld = ld_mod; er.gate_period = period;
  Epilogue eh;
  eh.act = ACT_GELU;
  if (!tc_mode(e)) {
    STK_TRY(lin32(e, blk + "attn.proj", attn32, D, M, er, s));
    PROF(PC_LN, launch_ln_mod(resid, D, mod + 3 * D, mod + 4 * D, ld_mod, period, a32, nullptr, nullptr, D, M, D, 1e-6f, s));
    eh.out = h32; eh.ldo = 4 * D;
    STK_TRY(lin32(e, blk + "mlp.fc1", a32, D, M, eh, s));
    er.gate = mod + 5 * D;
    return lin32(e, blk + "mlp.fc2", h32, 4 * D, M, er, s);
  }
  STK_TRY(lintc(e, blk + "attn.proj", attn_hi, attn_lo, M, er, s));
  PROF(PC_LN, launch_ln_mod(resid, D, mod + 3 * D, mod + 4 * D, ld_mod, period, nullptr, a_hi, a_lo, D, M, D, 1e-6f, s, is_fp16(e)));
  eh.mode = EPI_SPLIT; eh.out_hi = h_hi; eh.out_lo = h_lo; eh.ldo = 4 * D;
  STK_TRY(lintc(e, blk + "mlp.fc1", a_hi, a_lo, M, eh, s));
  er.gate = mod + 5 * D;
  return lintc(e, blk + "mlp.fc2", h_hi, h_lo, M, er, s);
}

// x = x_embedder(patches) + cropped pos_embed (mmdit.py:1000-1001) from ws.patch into ws.x.  Tensor-core modes: the K = 64 GEMM on
// the tcgen05 kernel with split-bf16 operands (fp32-faithful) instead of the fp32 FFMA kernel (0.3 ms -> ~20 us per evaluation).
static int x_embed(selftok_engine* e, int B, cudaStream_t s) {
  const selftok_config_t& c = e->cfg;
  DecodeWs& w = e->dws;
  const int D = e->D, N = e->Nimg, Kp = c.in_channels * c.dit_patch * c.dit_patch;
  Epilogue ep;
  ep.out = w.x; ep.addtab = e->dit_pos; ep.add_ld = D; ep.add_period = N;
  if (!tc_mode(e) || Kp % 8 != 0) return lin32(e, "model.x_embedder.proj", w.patch, Kp, (int64_t)B * N, ep, s);
  PROF(PC_OTHER, launch_split_bf16(w.patch, w.patch_hi, w.patch_lo, (int64_t)B * N * Kp, s, 0));
  GETW(Bv, "model.x_embedder.proj.bias");
  auto it = e->wp.find("model.x_embedder.proj.weight");
  STK_CHECK(it != e->wp.end(), SELFTOK_ERR_STATE, "packed x_embedder missing");
  ep.bias = Bv->d; ep.ldo = D;
  PROF(PC_GEMM_TC, launch_gemm_tc(w.patch_hi, w.patch_lo, it->second.hi, it->second.lo, (int64_t)B * N, D, Kp, 3, ep, s, 0));
  return 0;
}
// FinalLayer (mmdit.py:641-645): LN + modulate, then the N = p*p*C = 64 column linear -> o_out [B*N, 64] fp32
static int final_layer(selftok_engine* e, int B, const float* fm, float* o_out, cudaStream_t s) {
  DecodeWs& w = e->dws;
  const int D = e->D;
  const int64_t Mx = (int64_t)B * e->Nimg;
  if (!tc_mode(e)) {
    PROF(PC_LN, launch_ln_mod(w.x, D, fm, fm + D, 2 * D, 1, w.a_x, nullptr, nullptr, D, Mx, D, 1e-6f, s));
    Epilogue ep;
    ep.out = o_out;
    return lin32(e, "model.final_layer.linear", w.a_x, D, Mx, ep, s);
  }
  LnProblem lp;
  lp.x = w.x; lp.shift = fm; lp.scale = fm + D; lp.ld_mod = 2 * D; lp.period = 1; lp.out_hi = w.fin_hi; lp.out_lo = w.fin_lo; lp.M = Mx;
  PROF(PC_LN, launch_ln_mod_pair(&lp, 1, D, 1e-6f, s, 0));
  GETW(W, "model.final_layer.linear.weight");
  GETW(Bv, "model.final_layer.linear.bias");
  auto it = e->wp.find("model.final_layer.linear.weight");
  STK_CHECK(it != e->wp.end(), SELFTOK_ERR_STATE, "packed final layer missing");
  Epilogue ep;
  ep.out = o_out; ep.bias = Bv->d; ep.ldo = (int)W->shape[0];
  PROF(PC_GEMM_TC, launch_gemm_tc(w.fin_hi, w.fin_lo, it->second.hi, it->second.lo, Mx, (int)W->shape[0], D, 3, ep, s, 0));
  return 0;
}

// forward_core_with_concat (mmdit.py:918-933) on the residual streams already initialised in ws.ctx / ws.x.
//   Kc         visible context rows (prefix; rows >= Kc are dropped — exact, SURVEY 8a note)
//   step       row of the per-step tables (x adaLN, final adaLN, last-layer context adaLN)
//   ctx_self   context rows attend to context keys only (renderer; mmdit.py:1581)
//   uncond     unconditional branch of the guided sampler (MMDiT.cfg_inference, mmdit.py:1117-1163): Kc must be 0 (no row of
//              that pass sees a context key, so the context stream is dropped -- exact), x-stream adaLN from the integer timestep
//   o_out      final-layer output [B*N, p*p*C]
//   n_ctx      optional device [B]: image b sees only the context keys < min(Kc, n_ctx[b]) (decode from a token prefix)
static int joint_blocks(selftok_engine* e, int B, int Kc, int step, bool ctx_self, cudaStream_t s, bool uncond = false,
                        float* o_out = nullptr, const int32_t* n_ctx = nullptr) {
  const selftok_config_t& c = e->cfg;
  DecodeWs& w = e->dws;
  const int D = e->D, N = e->Nimg, L = c.dit_depth, T = e->steps, S = Kc + N;
  const int64_t Mc = (int64_t)B * Kc, Mx = (int64_t)B * N;
  const bool ctx = Kc > 0;                                                      // is there a context stream in this pass at all
  STK_CHECK(!uncond || (!ctx && e->x_mod_u), SELFTOK_ERR_STATE, "unconditional pass needs the guided-sampler tables and no context");
  const float* x_mod_base = uncond ? e->x_mod_u : e->x_mod;
  for (int j = 0; j < L; ++j) {
    const bool last = j == L - 1;
    const bool ctx_post = ctx && !last;                                         // the last context block is pre_only
    const std::string pc = "model.joint_blocks." + std::to_string(j) + ".context_block.";
    const std::string px = "model.joint_blocks." + std::to_string(j) + ".x_block.";
    const float* cmod = e->ctx_mod + (int64_t)j * c.K * 6 * D;                  // [K][6D]
    const float* xmod = x_mod_base + ((int64_t)j * T + step) * 6 * D;           // [6D]
    if (tc_mode(e)) {
      // ---- tensor-core path: the two streams' GEMMs of every stage share one launch (lintc2)
      const int fp16 = is_fp16(e);
      const float* lm = e->ctx_last_mod + (int64_t)step * 2 * D;                // last layer: pre_only (shift, scale) from c
      // LN + modulate of both streams in one launch (context rows: per-position adaLN table; image rows: the step's row)
      LnProblem lp[2];
      lp[0].x = w.ctx; lp[0].out_hi = w.a_c_hi; lp[0].out_lo = w.a_c_lo; lp[0].M = Mc;
      if (!last) { lp[0].shift = cmod; lp[0].scale = cmod + D; lp[0].ld_mod = 6 * D; lp[0].period = Kc; }
      else { lp[0].shift = lm; lp[0].scale = lm + D; lp[0].ld_mod = 2 * D; lp[0].period = 1; }
      lp[1].x = w.x; lp[1].out_hi = w.a_x_hi; lp[1].out_lo = w.a_x_lo; lp[1].M = Mx;
      lp[1].shift = xmod; lp[1].scale = xmod + D; lp[1].ld_mod = 6 * D; lp[1].period = 1;
      if (ctx) PROF(PC_LN, launch_ln_mod_pair(lp, 2, D, 1e-6f, s, fp16));
      else PROF(PC_LN, launch_ln_mod_pair(lp + 1, 1, D, 1e-6f, s, fp16));
      TcProblem pr[2];
      Epilogue eq;                                                              // q/k/v leave the GEMM as 16-bit planes in the joint buffer
      eq.mode = EPI_SPLIT; eq.out_hi = w.qkv_hi; eq.out_lo = w.qkv_lo; eq.ldo = 3 * D; eq.rpb_out = S;
      int np = 0;
      eq.rpb_in = Kc; eq.row_off = 0;
      if (ctx) STK_TRY(tc_problem(e, pc + "attn.qkv", w.a_c_hi, w.a_c_lo, Mc, eq, &pr[np++]));
      eq.rpb_in = N; eq.row_off = Kc;
      STK_TRY(tc_problem(e, px + "attn.qkv", w.a_x_hi, w.a_x_lo, Mx, eq, &pr[np++]));
      STK_TRY(lintc2(e, pr, np, s));
      AttnOut ao;
      ao.split = Kc; ao.ld = D;
      ao.hi_a = w.attn_c_hi; ao.lo_a = w.attn_c_lo; ao.hi_b = w.attn_x_hi; ao.lo_b = w.attn_x_lo;
      ao.fp16 = fp16;
      const int ctx_rows = ctx_self ? Kc : 0, ctx_keys = ctx_self ? Kc : 0;
      PROF(PC_ATTN, launch_attention_tc5(w.qkv_hi, B, S, e->H, ctx_rows, ctx_keys, ao, s, fp16, nsplit(e) == 3 ? w.qkv_lo : nullptr,
                                         n_ctx, Kc));
      // post_attention (mmdit.py:485-496); the pre_only context block of the last layer stops here
      Epilogue erx, erc;
      erx.mode = EPI_RESID; erx.out = w.x; erx.resid = w.x; erx.ldo = D; erx.gate = xmod + 2 * D; erx.gate_ld = 6 * D; erx.gate_period = 1;
      erc.mode = EPI_RESID; erc.out = w.ctx; erc.resid = w.ctx; erc.ldo = D; erc.gate = cmod + 2 * D; erc.gate_ld = 6 * D; erc.gate_period = Kc;
      np = 0;
      if (ctx_post) STK_TRY(tc_problem(e, pc + "attn.proj", w.attn_c_hi, w.attn_c_lo, Mc, erc, &pr[np++]));
      STK_TRY(tc_problem(e, px + "attn.proj", w.attn_x_hi, w.attn_x_lo, Mx, erx, &pr[np++]));
      STK_TRY(lintc2(e, pr, np, s));
      lp[0].shift = cmod + 3 * D; lp[0].scale = cmod + 4 * D; lp[0].ld_mod = 6 * D; lp[0].period = Kc;
      lp[1].shift = xmod + 3 * D; lp[1].scale = xmod + 4 * D;
      if (ctx_post) PROF(PC_LN, launch_ln_mod_pair(lp, 2, D, 1e-6f, s, fp16));
      else PROF(PC_LN, launch_ln_mod_pair(lp + 1, 1, D, 1e-6f, s, fp16));
      Epilogue ehc, ehx;
      ehc.mode = EPI_SPLIT; ehc.act = ACT_GELU; ehc.out_hi = w.h_c_hi; ehc.out_lo = w.h_c_lo; ehc.ldo = 4 * D;
      ehx = ehc; ehx.out_hi = w.h_x_hi; ehx.out_lo = w.h_x_lo;
      np = 0;
      if (ctx_post) STK_TRY(tc_problem(e, pc + "mlp.fc1", w.a_c_hi, w.a_c_lo, Mc, ehc, &pr[np++]));
      STK_TRY(tc_problem(e, px + "mlp.fc1", w.a_x_hi, w.a_x_lo, Mx, ehx, &pr[np++]));
      STK_TRY(lintc2(e, pr, np, s));
      erc.gate = cmod + 5 * D; erx.gate = xmod + 5 * D;
      np = 0;
      if (ctx_post) STK_TRY(tc_problem(e, pc + "mlp.fc2", w.h_c_hi, w.h_c_lo, Mc, erc, &pr[np++]));
      STK_TRY(tc_problem(e, px + "mlp.fc2", w.h_x_hi, w.h_x_lo, Mx, erx, &pr[np++]));
      STK_TRY(lintc2(e, pr, np, s));
      continue;
    }
    if (ctx && !last) {
      STK_TRY(pre_attention(e, pc, w.ctx, Mc, cmod, cmod + D, 6 * D, Kc, w.a_c, w.a_c_hi, w.a_c_lo, Kc, S, 0, s));
    } else if (ctx) {
      const float* lm = e->ctx_last_mod + (int64_t)step * 2 * D;                // pre_only: (shift, scale) from c
      STK_TRY(pre_attention(e, pc, w.ctx, Mc, lm, lm + D, 2 * D, 1, w.a_c, w.a_c_hi, w.a_c_lo, Kc, S, 0, s));
    }
    STK_TRY(pre_attention(e, px, w.x, Mx, xmod, xmod + D, 6 * D, 1, w.a_x, w.a_x_hi, w.a_x_lo, N, S, Kc, s));
    AttnOut ao;
    ao.split = Kc; ao.ld = D;
    const int ctx_rows = ctx_self ? Kc : 0, ctx_keys = ctx_self ? Kc : 0;
    if (!tc_mode(e)) {
      ao.f32_a = w.attn_c; ao.f32_b = w.attn_x;
      PROF(PC_ATTN, launch_attention_f32(w.qkv, 3 * D, (int64_t)S * 3 * D, w.qkv + D, w.qkv + 2 * D, 3 * D, (int64_t)S * 3 * D, S,
                                   nullptr, nullptr, 0, 0, 0, ao, B, S, e->H, 64, ctx_rows, ctx_keys, s, n_ctx, Kc));
    } else {
      ao.hi_a = w.attn_c_hi; ao.lo_a = w.attn_c_lo; ao.hi_b = w.attn_x_hi; ao.lo_b = w.attn_x_lo;
      ao.fp16 = is_fp16(e);
      PROF(PC_ATTN, launch_attention_tc5(w.qkv_hi, B, S, e->H, ctx_rows, ctx_keys, ao, s, is_fp16(e), nsplit(e) == 3 ? w.qkv_lo : nullptr,
                                         n_ctx, Kc));
    }
    if (ctx_post)
      STK_TRY(post_attention(e, pc, w.ctx, Mc, cmod, 6 * D, Kc, w.attn_c, w.attn_c_hi, w.attn_c_lo, w.a_c, w.a_c_hi, w.a_c_lo,
                             w.h_c, w.h_c_hi, w.h_c_lo, s));
    STK_TRY(post_attention(e, px, w.x, Mx, xmod, 6 * D, 1, w.attn_x, w.attn_x_hi, w.attn_x_lo, w.a_x, w.a_x_hi, w.a_x_lo,
                           w.h_x, w.h_x_hi, w.h_x_lo, s));
  }
  const float* fm = (uncond ? e->final_mod_u : e->final_mod) + (int64_t)step * 2 * D;
  return final_layer(e, B, fm, o_out ? o_out : w.o_final, s);
}

// context_embedder(outs_q) + context_pos_embed (mmdit.py:1026) — step invariant, computed once per call
static int context_embed(selftok_engine* e, int B, cudaStream_t s) {
  DecodeWs& w = e->dws;
  GETW(cp, "model.context_pos_embed");
  STK_CHECK(cp->numel == (int64_t)e->cfg.K * e->D, SELFTOK_ERR_BAD_ARG, "context_pos_embed shape");
  Epilogue ep;
  ep.out = w.ctx0; ep.addtab = cp->d; ep.add_ld = e->D; ep.add_period = e->cfg.K;
  return lin32(e, "model.context_embedder", w.outs_q, e->cfg.code_dim, (int64_t)B * e->cfg.K, ep, s);
}

// Context rows of schedule row `step`: the visible prefix k + 1 (rows beyond it are masked everywhere and dropped -- exact),
// capped at n_max, the longest token prefix of the batch (decode from a token prefix, the same truncation with min(k + 1, n))
static int ctx_rows_at(const selftok_engine* e, int step, int n_max) {
  return (e->k[step] < n_max - 1 ? e->k[step] : n_max - 1) + 1;
}

// Per-image token prefixes of one call: device counts [B] (engine-owned buffer) and their maximum; n == NULL: every K token
struct Prefix {
  const int32_t* n = nullptr;
  int n_max = 0;
};

// One MMDiT.forward (mmdit.py:992-1101) at schedule row `step` on ws.x_lat; leaves the patch outputs in ws.o_final.
static int dit_forward(selftok_engine* e, int B, int step, cudaStream_t s, Prefix pre = Prefix()) {
  const selftok_config_t& c = e->cfg;
  DecodeWs& w = e->dws;
  const int D = e->D, Kc = pre.n ? ctx_rows_at(e, step, pre.n_max) : e->k[step] + 1;
  PROF(PC_OTHER, launch_patchify(w.x_lat, w.patch, B, c.in_channels, c.latent, c.latent, c.dit_patch, s));
  STK_TRY(x_embed(e, B, s));
  PROF(PC_OTHER, launch_copy_rows(w.ctx0, (int64_t)c.K * D, w.ctx, (int64_t)Kc * D, B, (int64_t)Kc * D, s));
  // context rows see the image keys unless the handle was created with context_see_xt = 0 (sd3/mmdit.py:1012,1060; the
  // reference pipeline's sampler passes context_see_xt=True, SelftokPipeline.py:259)
  return joint_blocks(e, B, Kc, step, /*ctx_self=*/e->cfg.context_see_xt == 0, s, false, nullptr, pre.n);
}

// The two evaluations of one guided step (sample_one_step with cfg_scale != 1, rectified_flow.py:280-289): the conditional
// one -- called there WITHOUT context_see_xt, i.e. context rows only see the visible context keys -- into ws.o_final, and
// MMDiT.cfg_inference (context = zeros, every context key masked for every row: the image stream alone, integer timestep)
// into ws.o_final_u.
static int dit_forward_cfg(selftok_engine* e, int B, int step, cudaStream_t s, Prefix pre = Prefix()) {
  const selftok_config_t& c = e->cfg;
  DecodeWs& w = e->dws;
  const int D = e->D, Kc = pre.n ? ctx_rows_at(e, step, pre.n_max) : e->k[step] + 1;
  STK_CHECK(e->has_cfg, SELFTOK_ERR_STATE, "guided sampling needs selftok_set_cfg_schedule before selftok_finalize");
  PROF(PC_OTHER, launch_patchify(w.x_lat, w.patch, B, c.in_channels, c.latent, c.latent, c.dit_patch, s));
  STK_TRY(x_embed(e, B, s));
  PROF(PC_OTHER, launch_copy_rows(w.ctx0, (int64_t)c.K * D, w.ctx, (int64_t)Kc * D, B, (int64_t)Kc * D, s));
  STK_TRY(joint_blocks(e, B, Kc, step, /*ctx_self=*/true, s, /*uncond=*/false, w.o_final, pre.n));
  STK_TRY(x_embed(e, B, s));
  return joint_blocks(e, B, 0, step, /*ctx_self=*/false, s, /*uncond=*/true, w.o_final_u);
}

static int decode_body(selftok_engine* e, int B, int steps, cudaStream_t s, bool guided = false, float cfg_scale = 1.f,
                       Prefix pre = Prefix()) {
  const selftok_config_t& c = e->cfg;
  DecodeWs& w = e->dws;
  STK_TRY(run_lookup(e, w.tokens, B, w.outs_q, s, pre.n));
  STK_TRY(context_embed(e, B, s));
  for (int i = 0; i < steps; ++i) {
    // euler_step (rectified_flow.py:301-303): x <- x - (t_i - t_{i+1}) * v, fused with unpatchify
    if (!guided) {
      STK_TRY(dit_forward(e, B, i, s, pre));
      PROF(PC_OTHER, launch_unpatchify_axpy(w.o_final, w.x_lat, w.x_lat, e->dt[i], B, c.in_channels, c.latent / c.dit_patch, c.dit_patch, s));
    } else {
      STK_TRY(dit_forward_cfg(e, B, i, s, pre));
      PROF(PC_OTHER, launch_unpatchify_axpy(w.o_final, w.x_lat, w.x_lat, e->dt[i], B, c.in_channels, c.latent / c.dit_patch, c.dit_patch, s,
                                            w.o_final_u, cfg_scale));
    }
  }
  return 0;
}

// Bytes of activation workspace op (0: selftok_encode*, 1: selftok_decode* / selftok_render* / selftok_dit_velocity) needs for batch B.
extern "C" __attribute__((visibility("default"))) int64_t selftok_workspace_bytes(selftok_handle_t e, int B, int op) {
  if (!e || B <= 0 || (op != 0 && op != 1)) return -1;
  Arena dry;
  dry.dry = true;
  if (op == 0) { EncodeWs w; if (layout_ews(e, w, B, dry) != 0) return -1; }
  else { DecodeWs w; if (layout_dws(e, w, B, dry) != 0) return -1; }
  return (int64_t)dry.off;
}
// Hand the library a caller-owned device block for workspace `op` (NULL / 0 returns to library-owned memory).  While it is at
// least selftok_workspace_bytes(h, B, op) large, calls with batch <= B allocate nothing; the block must stay alive and must not
// be used by anything else while a call on this handle is in flight.  Captured CUDA graphs of the decode loop are dropped.
extern "C" __attribute__((visibility("default"))) int selftok_set_workspace(selftok_handle_t e, int op, void* ws_dev, size_t bytes) {
  STK_CHECK(e && (op == 0 || op == 1), SELFTOK_ERR_BAD_ARG, "selftok_set_workspace: bad argument");
  STK_CHECK((reinterpret_cast<uintptr_t>(ws_dev) & 255) == 0, SELFTOK_ERR_BAD_ARG, "selftok_set_workspace: the block must be 256-byte aligned");
  STK_CUDA(cudaSetDevice(e->cfg.device));
  STK_CUDA(cudaDeviceSynchronize());
  e->user_ws[op] = bytes ? ws_dev : nullptr;
  e->user_ws_bytes[op] = ws_dev ? bytes : 0;
  if (op == 0) free_ews(e);
  else {
    drop_decode_graphs(e);
    free_dws(e);
  }
  return SELFTOK_OK;
}

extern "C" __attribute__((visibility("default"))) int selftok_set_use_graph(selftok_handle_t e, int enable) {
  STK_CHECK(e, SELFTOK_ERR_BAD_ARG, "null handle");
  e->use_graph = enable != 0;
  return SELFTOK_OK;
}

static int decode_impl(selftok_handle_t e, const int64_t* tokens_dev, const float* noise_dev, int B, int steps, float* x0_out_dev,
                       void* stream, bool guided, float cfg_scale, const int32_t* n_host = nullptr);

// Per-image token prefixes from the host: every n_b in [1, K] (checked before anything is launched), copied into the
// engine-owned device buffer on `s` -- after the copy the caller's array is not read again
static int check_prefix(selftok_engine* e, const int32_t* n_host, int B, int* n_max) {
  STK_CHECK(n_host, SELFTOK_ERR_BAD_ARG, "token prefix: null n_tokens");
  *n_max = 0;
  for (int b = 0; b < B; ++b) {
    STK_CHECK(n_host[b] >= 1 && n_host[b] <= e->cfg.K, SELFTOK_ERR_BAD_ARG,
              "token prefix: n_tokens[" + std::to_string(b) + "] = " + std::to_string(n_host[b]) + " is outside [1, K]");
    if (n_host[b] > *n_max) *n_max = n_host[b];
  }
  return 0;
}
static int load_prefix(selftok_engine* e, const int32_t* n_host, int B, int n_max, cudaStream_t s, Prefix* pre) {
  if (e->n_cap < B) {
    drop_decode_graphs(e);
    if (e->n_dev) { cudaFree(e->n_dev); e->n_dev = nullptr; e->n_cap = 0; }
    STK_CUDA(cudaMalloc(&e->n_dev, sizeof(int32_t) * B));
    e->n_cap = B;
  }
  STK_CUDA(cudaMemcpyAsync(e->n_dev, n_host, sizeof(int32_t) * B, cudaMemcpyHostToDevice, s));
  pre->n = e->n_dev;
  pre->n_max = n_max;
  return 0;
}

extern "C" __attribute__((visibility("default"))) int selftok_decode(selftok_handle_t e, const int64_t* tokens_dev, const float* noise_dev, int B, int steps,
                              float* x0_out_dev, void* stream) {
  return decode_impl(e, tokens_dev, noise_dev, B, steps, x0_out_dev, stream, false, 1.f);
}

// Guided sampler: p_sample_loop(..., uncond_scale = cfg_scale) of the reference (rectified_flow.py:165-294): two MMDiT
// evaluations per step, v = v_u + cfg_scale (v_c - v_u).  Needs selftok_set_cfg_schedule before finalize.
extern "C" __attribute__((visibility("default"))) int selftok_decode_cfg(selftok_handle_t e, const int64_t* tokens_dev, const float* noise_dev, int B, int steps,
                                  float cfg_scale, float* x0_out_dev, void* stream) {
  return decode_impl(e, tokens_dev, noise_dev, B, steps, x0_out_dev, stream, true, cfg_scale);
}

// Decode from a token prefix: image b from its first n_tokens_host[b] tokens (super_mask of p_sample_loop, rectified_flow.py:
// 182,227-228).  cfg_scale == 1: the plain sampler (captured graph); otherwise the guided sampler (eager), the prefix applied
// to its conditional evaluation.
extern "C" __attribute__((visibility("default"))) int selftok_decode_prefix(selftok_handle_t e, const int64_t* tokens_dev, const int32_t* n_tokens_host,
                                                                       const float* noise_dev, int B, int steps, float cfg_scale,
                                                                       float* x0_out_dev, void* stream) {
  STK_CHECK(n_tokens_host, SELFTOK_ERR_BAD_ARG, "selftok_decode_prefix: null n_tokens");
  return decode_impl(e, tokens_dev, noise_dev, B, steps, x0_out_dev, stream, cfg_scale != 1.f, cfg_scale, n_tokens_host);
}

static int decode_impl(selftok_handle_t e, const int64_t* tokens_dev, const float* noise_dev, int B, int steps, float* x0_out_dev,
                       void* stream, bool guided, float cfg_scale, const int32_t* n_host) {
  HOT_PROLOGUE(e);
  STK_CHECK(!guided || e->has_cfg, SELFTOK_ERR_STATE, "selftok_decode_cfg: selftok_set_cfg_schedule was not called before finalize");
  STK_CHECK(tokens_dev && noise_dev && x0_out_dev && B > 0, SELFTOK_ERR_BAD_ARG, "selftok_decode: bad argument");
  STK_CHECK(!e->cfg.renderer, SELFTOK_ERR_STATE, "handle was created for the renderer; use selftok_render");
  STK_CHECK(steps > 0 && steps <= e->steps, SELFTOK_ERR_BAD_ARG, "steps exceeds the schedule");
  int n_max = 0;
  if (n_host) STK_TRY(check_prefix(e, n_host, B, &n_max));
  STK_TRY(ensure_dws(e, B));
  Prefix pre;
  if (n_host) STK_TRY(load_prefix(e, n_host, B, n_max, s, &pre));
  DecodeWs& w = e->dws;
  const int64_t nlat = (int64_t)B * e->cfg.in_channels * e->cfg.latent * e->cfg.latent;
  if (tokens_dev != w.tokens) STK_CUDA(cudaMemcpyAsync(w.tokens, tokens_dev, sizeof(int64_t) * B * e->cfg.K, cudaMemcpyDeviceToDevice, s));
  if (noise_dev != w.x_lat) STK_CUDA(cudaMemcpyAsync(w.x_lat, noise_dev, sizeof(float) * nlat, cudaMemcpyDeviceToDevice, s));
  // eager when asked to, for the guided loop (cfg_scale is a kernel argument) and whenever per-launch profiling is on (events
  // recorded inside a capture never execute on a real stream: their elapsed times would be garbage)
  if (!e->use_graph || guided || e->prof_on) {
    STK_TRY(decode_body(e, B, steps, s, guided, cfg_scale, pre));
    e->last_launches = g_launch_count - launches0;
  } else if (pre.n) {
    // one graph per (B, steps, context rows of every step); the counts it reads were refreshed above, on the same stream
    std::vector<int> key = {B, steps};
    for (int i = 0; i < steps; ++i) key.push_back(ctx_rows_at(e, i, pre.n_max));
    auto it = e->prefix_graphs.find(key);
    if (it == e->prefix_graphs.end()) {
      if (e->prefix_graphs.size() >= kPrefixGraphs) {
        auto lru = e->prefix_graphs.begin();
        for (auto j = e->prefix_graphs.begin(); j != e->prefix_graphs.end(); ++j)
          if (j->second.used < lru->second.used) lru = j;
        STK_CUDA(cudaStreamSynchronize(s));                          // a replay of it may still be queued on this stream
        cudaGraphExecDestroy(lru->second.exec);
        e->prefix_graphs.erase(lru);
      }
      cudaStream_t cs;
      STK_CUDA(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
      {
        const cudaError_t be = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
        if (be != cudaSuccess) {
          cudaStreamDestroy(cs);
          STK_CUDA(be);
        }
      }
      const int64_t l0 = g_launch_count;
      int st = decode_body(e, B, steps, cs, false, 1.f, pre);
      cudaGraph_t graph = nullptr;
      cudaError_t ce = cudaStreamEndCapture(cs, &graph);
      cudaStreamDestroy(cs);
      if (st != 0) { if (graph) cudaGraphDestroy(graph); return st; }
      STK_CUDA(ce);
      cudaGraphExec_t exec;
      STK_CUDA(cudaGraphInstantiate(&exec, graph, 0));
      cudaGraphDestroy(graph);
      it = e->prefix_graphs.emplace(key, selftok_engine::PrefixGraph{exec, g_launch_count - l0, 0}).first;
    }
    it->second.used = ++e->prefix_tick;
    STK_CUDA(cudaGraphLaunch(it->second.exec, s));
    e->last_launches = it->second.launches;
  } else {
    auto key = std::make_pair(B, steps);
    auto it = e->graphs.find(key);
    if (it == e->graphs.end()) {
      cudaStream_t cs;
      STK_CUDA(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
      {
        const cudaError_t be = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
        if (be != cudaSuccess) {
          cudaStreamDestroy(cs);                                       // no leak on the error path
          STK_CUDA(be);
        }
      }
      const int64_t l0 = g_launch_count;
      int st = decode_body(e, B, steps, cs);
      cudaGraph_t graph = nullptr;
      cudaError_t ce = cudaStreamEndCapture(cs, &graph);
      cudaStreamDestroy(cs);
      if (st != 0) { if (graph) cudaGraphDestroy(graph); return st; }
      STK_CUDA(ce);
      cudaGraphExec_t exec;
      STK_CUDA(cudaGraphInstantiate(&exec, graph, 0));
      cudaGraphDestroy(graph);
      it = e->graphs.emplace(key, std::make_pair(exec, g_launch_count - l0)).first;
    }
    STK_CUDA(cudaGraphLaunch(it->second.first, s));
    e->last_launches = it->second.second;
  }
  if (x0_out_dev != w.x_lat) STK_CUDA(cudaMemcpyAsync(x0_out_dev, w.x_lat, sizeof(float) * nlat, cudaMemcpyDeviceToDevice, s));
  return SELFTOK_OK;
}

static int velocity_impl(selftok_handle_t e, const int64_t* tokens_dev, const int32_t* n_host, const float* x_dev, int B, int step,
                         float* v_out_dev, void* stream) {
  HOT_PROLOGUE(e);
  STK_CHECK(tokens_dev && x_dev && v_out_dev && B > 0, SELFTOK_ERR_BAD_ARG, "selftok_dit_velocity: bad argument");
  STK_CHECK(!e->cfg.renderer, SELFTOK_ERR_STATE, "renderer handle");
  STK_CHECK(step >= 0 && step < e->steps, SELFTOK_ERR_BAD_ARG, "step out of range");
  int n_max = 0;
  if (n_host) STK_TRY(check_prefix(e, n_host, B, &n_max));
  STK_TRY(ensure_dws(e, B));
  Prefix pre;
  if (n_host) STK_TRY(load_prefix(e, n_host, B, n_max, s, &pre));
  DecodeWs& w = e->dws;
  const selftok_config_t& c = e->cfg;
  const int64_t nlat = (int64_t)B * c.in_channels * c.latent * c.latent;
  STK_CUDA(cudaMemcpyAsync(w.tokens, tokens_dev, sizeof(int64_t) * B * c.K, cudaMemcpyDeviceToDevice, s));
  STK_CUDA(cudaMemcpyAsync(w.x_lat, x_dev, sizeof(float) * nlat, cudaMemcpyDeviceToDevice, s));
  STK_TRY(run_lookup(e, w.tokens, B, w.outs_q, s, pre.n));
  STK_TRY(context_embed(e, B, s));
  STK_TRY(dit_forward(e, B, step, s, pre));
  PROF(PC_OTHER, launch_unpatchify_axpy(w.o_final, nullptr, v_out_dev, -1.f, B, c.in_channels, c.latent / c.dit_patch, c.dit_patch, s));
  e->last_launches = g_launch_count - launches0;
  return SELFTOK_OK;
}

extern "C" __attribute__((visibility("default"))) int selftok_dit_velocity(selftok_handle_t e, const int64_t* tokens_dev, const float* x_dev, int B, int step,
                                    float* v_out_dev, void* stream) {
  return velocity_impl(e, tokens_dev, nullptr, x_dev, B, step, v_out_dev, stream);
}

extern "C" __attribute__((visibility("default"))) int selftok_dit_velocity_prefix(selftok_handle_t e, const int64_t* tokens_dev, const int32_t* n_tokens_host,
                                                                             const float* x_dev, int B, int step, float* v_out_dev, void* stream) {
  STK_CHECK(n_tokens_host, SELFTOK_ERR_BAD_ARG, "selftok_dit_velocity_prefix: null n_tokens");
  return velocity_impl(e, tokens_dev, n_tokens_host, x_dev, B, step, v_out_dev, stream);
}

static int render_impl(selftok_handle_t e, const int64_t* tokens_dev, const int32_t* n_host, int B, float* x0_out_dev, void* stream) {
  HOT_PROLOGUE(e);
  STK_CHECK(tokens_dev && x0_out_dev && B > 0, SELFTOK_ERR_BAD_ARG, "selftok_render: bad argument");
  STK_CHECK(e->cfg.renderer, SELFTOK_ERR_STATE, "handle was not created for the renderer");
  int n_max = 0;
  if (n_host) STK_TRY(check_prefix(e, n_host, B, &n_max));
  STK_TRY(ensure_dws(e, B));
  Prefix pre;
  if (n_host) STK_TRY(load_prefix(e, n_host, B, n_max, s, &pre));
  DecodeWs& w = e->dws;
  const selftok_config_t& c = e->cfg;
  // context rows: all K, or the batch's longest prefix (image b then masks the context keys [n_b, n_max))
  const int Kc = pre.n ? pre.n_max : c.K;
  if (tokens_dev != w.tokens) STK_CUDA(cudaMemcpyAsync(w.tokens, tokens_dev, sizeof(int64_t) * B * c.K, cudaMemcpyDeviceToDevice, s));
  STK_TRY(run_lookup(e, w.tokens, B, w.outs_q, s, pre.n));
  STK_TRY(context_embed(e, B, s));
  // x = mask_token + positional_embedding (mmdit.py:1518-1522); context rows see context only
  PROF(PC_OTHER, launch_bcast_rows(e->rend_x0, nullptr, w.x, B, e->Nimg, e->D, s));
  PROF(PC_OTHER, launch_copy_rows(w.ctx0, (int64_t)c.K * e->D, w.ctx, (int64_t)Kc * e->D, B, (int64_t)Kc * e->D, s));
  STK_TRY(joint_blocks(e, B, Kc, 0, /*ctx_self=*/true, s, false, nullptr, pre.n));
  PROF(PC_OTHER, launch_unpatchify_axpy(w.o_final, nullptr, x0_out_dev, -1.f, B, c.in_channels, c.latent / c.dit_patch, c.dit_patch, s));
  e->last_launches = g_launch_count - launches0;
  return SELFTOK_OK;
}

extern "C" __attribute__((visibility("default"))) int selftok_render(selftok_handle_t e, const int64_t* tokens_dev, int B, float* x0_out_dev, void* stream) {
  return render_impl(e, tokens_dev, nullptr, B, x0_out_dev, stream);
}

extern "C" __attribute__((visibility("default"))) int selftok_render_prefix(selftok_handle_t e, const int64_t* tokens_dev, const int32_t* n_tokens_host,
                                                                       int B, float* x0_out_dev, void* stream) {
  STK_CHECK(n_tokens_host, SELFTOK_ERR_BAD_ARG, "selftok_render_prefix: null n_tokens");
  return render_impl(e, tokens_dev, n_tokens_host, B, x0_out_dev, stream);
}

// ------------------------------------------------------------------------------------------------ host-buffer variants
extern "C" __attribute__((visibility("default"))) int selftok_encode_host(selftok_handle_t e, const float* x0_host, int B, int64_t* tokens_host, void* stream) {
  STK_CHECK(e && x0_host && tokens_host && B > 0, SELFTOK_ERR_BAD_ARG, "selftok_encode_host: bad argument");
  STK_CHECK(e->finalized, SELFTOK_ERR_STATE, "selftok_finalize has not been called");
  STK_CUDA(cudaSetDevice(e->cfg.device));
  cudaStream_t s = (cudaStream_t)stream;
  STK_TRY(ensure_ews(e, B));
  const int64_t nlat = (int64_t)B * e->cfg.in_channels * e->cfg.latent * e->cfg.latent;
  STK_CUDA(cudaMemcpyAsync(e->ews.x0, x0_host, sizeof(float) * nlat, cudaMemcpyHostToDevice, s));
  STK_TRY(selftok_encode(e, e->ews.x0, B, e->ews.tokens, nullptr, nullptr, stream));
  STK_CUDA(cudaMemcpyAsync(tokens_host, e->ews.tokens, sizeof(int64_t) * B * e->cfg.K, cudaMemcpyDeviceToHost, s));
  STK_CUDA(cudaStreamSynchronize(s));
  return SELFTOK_OK;
}

extern "C" __attribute__((visibility("default"))) int selftok_decode_host(selftok_handle_t e, const int64_t* tokens_host, const float* noise_host, int B, int steps,
                                   float* x0_out_host, void* stream) {
  STK_CHECK(e && tokens_host && noise_host && x0_out_host && B > 0, SELFTOK_ERR_BAD_ARG, "selftok_decode_host: bad argument");
  STK_CHECK(e->finalized, SELFTOK_ERR_STATE, "selftok_finalize has not been called");
  STK_CUDA(cudaSetDevice(e->cfg.device));
  cudaStream_t s = (cudaStream_t)stream;
  STK_TRY(ensure_dws(e, B));
  DecodeWs& w = e->dws;
  const int64_t nlat = (int64_t)B * e->cfg.in_channels * e->cfg.latent * e->cfg.latent;
  STK_CUDA(cudaMemcpyAsync(w.tokens, tokens_host, sizeof(int64_t) * B * e->cfg.K, cudaMemcpyHostToDevice, s));
  STK_CUDA(cudaMemcpyAsync(w.x_lat, noise_host, sizeof(float) * nlat, cudaMemcpyHostToDevice, s));
  STK_TRY(selftok_decode(e, w.tokens, w.x_lat, B, steps, w.x_lat, stream));
  STK_CUDA(cudaMemcpyAsync(x0_out_host, w.x_lat, sizeof(float) * nlat, cudaMemcpyDeviceToHost, s));
  STK_CUDA(cudaStreamSynchronize(s));
  return check_ids_after_sync(e, stream, "selftok_decode_host");
}

extern "C" __attribute__((visibility("default"))) int selftok_render_host(selftok_handle_t e, const int64_t* tokens_host, int B, float* x0_out_host, void* stream) {
  STK_CHECK(e && tokens_host && x0_out_host && B > 0, SELFTOK_ERR_BAD_ARG, "selftok_render_host: bad argument");
  STK_CHECK(e->finalized, SELFTOK_ERR_STATE, "selftok_finalize has not been called");
  STK_CUDA(cudaSetDevice(e->cfg.device));
  cudaStream_t s = (cudaStream_t)stream;
  STK_TRY(ensure_dws(e, B));
  DecodeWs& w = e->dws;
  const int64_t nlat = (int64_t)B * e->cfg.in_channels * e->cfg.latent * e->cfg.latent;
  STK_CUDA(cudaMemcpyAsync(w.tokens, tokens_host, sizeof(int64_t) * B * e->cfg.K, cudaMemcpyHostToDevice, s));
  STK_TRY(selftok_render(e, w.tokens, B, w.x_lat, stream));
  STK_CUDA(cudaMemcpyAsync(x0_out_host, w.x_lat, sizeof(float) * nlat, cudaMemcpyDeviceToHost, s));
  STK_CUDA(cudaStreamSynchronize(s));
  return check_ids_after_sync(e, stream, "selftok_render_host");
}

extern "C" __attribute__((visibility("default"))) int selftok_set_profile(selftok_handle_t e, int enable) {
  STK_CHECK(e, SELFTOK_ERR_BAD_ARG, "null handle");
  e->prof_on = enable != 0;
  return SELFTOK_OK;
}

// Synchronises the device, sums the recorded event pairs per kernel class and clears them.
extern "C" __attribute__((visibility("default"))) int selftok_get_profile(selftok_handle_t e, double* ms_out, int64_t* count_out) {
  STK_CHECK(e && ms_out && count_out, SELFTOK_ERR_BAD_ARG, "selftok_get_profile: bad argument");
  STK_CUDA(cudaSetDevice(e->cfg.device));
  STK_CUDA(cudaDeviceSynchronize());
  for (int i = 0; i < PC_COUNT; ++i) { ms_out[i] = 0.0; count_out[i] = 0; }
  for (size_t i = 0; i < e->prof_cat.size(); ++i) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e->prof_ev[2 * i], e->prof_ev[2 * i + 1]);
    ms_out[e->prof_cat[i]] += ms;
    count_out[e->prof_cat[i]] += 1;
    cudaEventDestroy(e->prof_ev[2 * i]);
    cudaEventDestroy(e->prof_ev[2 * i + 1]);
  }
  e->prof_ev.clear();
  e->prof_cat.clear();
  return SELFTOK_OK;
}

extern "C" __attribute__((visibility("default"))) int64_t selftok_last_launch_count(selftok_handle_t e) { return e ? e->last_launches : -1; }
extern "C" __attribute__((visibility("default"))) int64_t selftok_device_bytes(selftok_handle_t e) { return e ? e->bytes : -1; }

// ------------------------------------------------------------------------------------------------ kernel-level ABI
extern "C" __attribute__((visibility("default"))) int selftok_k_linear_f32(const float* A, const float* W, const float* bias, float* out, int64_t M, int N, int K,
                                    int act, void* stream) {
  Epilogue ep;
  ep.act = act; ep.bias = bias; ep.out = out; ep.ldo = N;
  return launch_linear_f32(A, K, W, K, M, N, K, ep, (cudaStream_t)stream);
}

extern "C" __attribute__((visibility("default"))) int selftok_k_linear_tc(const float* A, const float* W, const float* bias, float* out, int64_t M, int N, int K,
                                   int ns, void* stream) {
  STK_CHECK(A && W && out && (ns == 0 || ns == 1 || ns == 3), SELFTOK_ERR_BAD_ARG, "selftok_k_linear_tc: bad argument");
  const int fp16 = ns == 0;
  if (fp16) ns = 1;
  STK_TRY(gemm_tc_init());
  cudaStream_t s = (cudaStream_t)stream;
  bf16 *ah, *al = nullptr, *wh, *wl = nullptr;
  STK_CUDA(cudaMalloc(&ah, sizeof(bf16) * M * K));
  STK_CUDA(cudaMalloc(&wh, sizeof(bf16) * (int64_t)N * K));
  if (ns == 3) {
    STK_CUDA(cudaMalloc(&al, sizeof(bf16) * M * K));
    STK_CUDA(cudaMalloc(&wl, sizeof(bf16) * (int64_t)N * K));
  }
  int st = launch_split_bf16(A, ah, al, M * K, s, fp16);
  if (!st) st = launch_split_bf16(W, wh, wl, (int64_t)N * K, s, fp16);
  Epilogue ep;
  ep.bias = bias; ep.out = out; ep.ldo = N;
  if (!st) st = launch_gemm_tc(ah, al, wh, wl, M, N, K, ns, ep, s, fp16);
  cudaStreamSynchronize(s);
  cudaFree(ah); cudaFree(wh);
  if (al) cudaFree(al);
  if (wl) cudaFree(wl);
  return st;
}

extern "C" __attribute__((visibility("default"))) int selftok_k_set_gemm_ctas(int n) {
  STK_CHECK(n == 1 || n == 2, SELFTOK_ERR_BAD_ARG, "selftok_k_set_gemm_ctas: n must be 1 or 2");
  gemm_tc_set_ctas(n);
  return SELFTOK_OK;
}

extern "C" __attribute__((visibility("default"))) int selftok_k_ln_mod_f32(const float* x, const float* shift, const float* scale, int64_t ld_mod, int period,
                                    float* out, int64_t M, int D, void* stream) {
  return launch_ln_mod(x, D, shift, scale, ld_mod, period, out, nullptr, nullptr, D, M, D, 1e-6f, (cudaStream_t)stream);
}

extern "C" __attribute__((visibility("default"))) int selftok_k_attention_f32(const float* q, int64_t q_ld, const float* k1, const float* v1, int64_t kv1_ld, int S1,
                                       const float* k2, const float* v2, int64_t kv2_ld, int S2, float* out, int64_t out_ld,
                                       int B, int Sq, int H, int hd, void* stream) {
  AttnOut ao;
  ao.f32_a = out; ao.split = Sq; ao.ld = out_ld;
  return launch_attention_f32(q, q_ld, (int64_t)Sq * q_ld, k1, v1, kv1_ld, (int64_t)S1 * kv1_ld, S1, k2, v2, kv2_ld,
                              (int64_t)S2 * kv2_ld, S2, ao, B, Sq, H, hd, 0, 0, (cudaStream_t)stream);
}

extern "C" __attribute__((visibility("default"))) int selftok_k_attention_tc(const float* qkv, float* out, int B, int S, int H, int ns, int ctx_rows, int ctx_keys,
                                      void* stream) {
  STK_CHECK(qkv && out && (ns == 0 || ns == 1 || ns == 3), SELFTOK_ERR_BAD_ARG, "selftok_k_attention_tc: bad argument");
  const int fp16 = ns == 0;                     // 0: IEEE half, 1: bf16, 3: split bf16 (hi + lo planes, three MMAs per product)
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t n = (int64_t)B * S * 3 * H * 64;
  bf16 *qh, *ql = nullptr;
  STK_CUDA(cudaMalloc(&qh, sizeof(bf16) * n));
  if (ns == 3) STK_CUDA(cudaMalloc(&ql, sizeof(bf16) * n));
  int st = launch_split_bf16(qkv, qh, ql, n, s, fp16);
  AttnOut ao;
  ao.f32_a = out; ao.split = S; ao.ld = (int64_t)H * 64;
  if (!st) st = launch_attention_tc5(qh, B, S, H, ctx_rows, ctx_keys, ao, s, fp16, ql);
  cudaStreamSynchronize(s);
  cudaFree(qh);
  if (ql) cudaFree(ql);
  return st;
}
